// stream_ceiling.cu -- what a 5-in/1-out and a 6-in/1-out Float64 stream reach on this GPU, with a trivial functor
// (y = a + b + c + d + e (+ f)), in the two forms the elementwise operators can take:
//   (a) ew_kernel<2, UNROLL, Op, NIN>: 16-byte ld.global.L1::no_allocate per thread, UNROLL 1/2, 3-4 CTAs per SM;
//   (b) ew_bulk_kernel<Op, TILE, STAGES, WARPS>: the producer-warp bulk-copy ring, swept over tile bytes, stages,
//       consumer warps and resident CTAs per SM.
// Both are the library's own kernels (spx_elementwise.cuh, spx_bulk.cuh), so the numbers bound what the Box operators can reach.
// n = 2^28 (2 GiB per operand, far above L2), 3 warm-ups, median of 20 runs timed with CUDA events.  Every variant's
// output is checked against the sum on the device, and the bulk form once more at an n that leaves a partial tile.
// One JSON line per variant on stdout.  Build and run: tools/stream_ceiling.sh
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../shiftedproximaloperators.jl_b200/csrc/spx_bulk.cuh"
#include "../shiftedproximaloperators.jl_b200/csrc/spx_elementwise.cuh"

using namespace spx;

// the spx_common.cuh error hooks, which the header declares
namespace spx {
void set_error(const char*, ...) {}
int32_t cuda_fail(cudaError_t e, const char*) { return (int32_t)e; }
}  // namespace spx

#define CK(x)                                                                              \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) {                                                               \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      exit(1);                                                                             \
    }                                                                                      \
  } while (0)

template <int NIN_, int MINB_, int UNROLL_> struct SumOp {
  using Real = double;
  static constexpr int NIN = NIN_, UNROLL = UNROLL_, MINB = MINB_;
  static constexpr bool OUT = true, ACC = false;
  const double* in[NIN];
  double fill[NIN];
  double* y;
  __device__ __forceinline__ double apply(const double (&x)[NIN], long long, Partial&) const {
    double s = x[0];
#pragma unroll
    for (int k = 1; k < NIN; ++k) s += x[k];
    return s;
  }
};

__global__ void fill_kernel(double* p, long long n, int k) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] = (double)((i * (k + 3)) % 1001) * 0.5;
}
template <int NIN>
__global__ void check_kernel(const double* const* in, const double* y, long long n, unsigned long long* bad) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double s = in[0][i];
    for (int k = 1; k < NIN; ++k) s += in[k][i];
    if (s != y[i]) atomicAdd(bad, 1ull);
  }
}

static std::string g_gpu;  // "name, power.limit, clocks.max.sm" of this device
static int g_sms = 148;
static double* g_in[6];
static double* g_y;
static const double** g_din;
static unsigned long long* g_bad;

template <int NIN> static unsigned long long check(long long n) {
  CK(cudaMemset(g_bad, 0, sizeof(unsigned long long)));
  check_kernel<NIN><<<g_sms * 8, 256>>>(g_din, g_y, n, g_bad);
  unsigned long long h = 0;
  CK(cudaMemcpy(&h, g_bad, sizeof h, cudaMemcpyDeviceToHost));
  return h;
}

template <class F> static double median_ms(F launch) {
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  for (int w = 0; w < 3; ++w) launch();
  CK(cudaGetLastError());
  std::vector<float> ms;
  for (int r = 0; r < 20; ++r) {
    CK(cudaEventRecord(a));
    launch();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, a, b));
    ms.push_back(t);
  }
  CK(cudaGetLastError());
  CK(cudaEventDestroy(a));
  CK(cudaEventDestroy(b));
  std::sort(ms.begin(), ms.end());
  return 0.5 * (ms[9] + ms[10]);
}

static void report(const char* form, int nin, const char* cfg, long long n, double ms, unsigned long long bad) {
  const double bytes = (double)(nin + 1) * 8.0 * (double)n;
  printf("{\"form\": \"%s\", \"stream\": \"%dR+1W f64\", \"config\": {%s}, \"n\": %lld, \"ms\": %.4f, \"TBps\": %.3f, "
         "\"mismatches\": %llu, \"gpu\": \"%s\"}\n",
         form, nin, cfg, n, ms, bytes / (ms * 1e-3) / 1e12, bad, g_gpu.c_str());
  fflush(stdout);
}

template <int NIN, int MINB, int U> static void run_direct(long long n) {
  using Op = SumOp<NIN, MINB, U>;
  Op op{};
  for (int k = 0; k < NIN; ++k) op.in[k] = g_in[k];
  op.y = g_y;
  auto kern = ew_kernel<2, U, Op, NIN>;
  int nb = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kEwThreads, 0));
  const long long want = (n / 2 + (long long)kEwThreads * U - 1) / ((long long)kEwThreads * U);
  const int grid = (int)std::min<long long>(want, (long long)g_sms * nb);
  const double ms = median_ms([&] { kern<<<grid, kEwThreads>>>(op, n, 0, nullptr); });
  char cfg[160];
  snprintf(cfg, sizeof cfg, "\"unroll\": %d, \"minb\": %d, \"ctas_per_sm\": %d", U, MINB, nb);
  report("ew_kernel", NIN, cfg, n, ms, check<NIN>(n));
}

template <int NIN, int TILE, int ST, int CW> static void run_bulk(long long n, long long n_tail) {
  using Op = SumOp<NIN, 1, 1>;
  Op op{};
  for (int k = 0; k < NIN; ++k) op.in[k] = g_in[k];
  op.y = g_y;
  constexpr size_t smem = (size_t)ST * NIN * TILE;
  if (smem > 227 * 1024) return;
  auto kern = ew_bulk_kernel<Op, TILE, ST, CW, 1>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, (CW + 1) * 32, smem));
  constexpr int TE = TILE / 8;
  for (int ctas = 1; ctas <= 3 && ctas <= occ; ++ctas) {
    const int grid = (int)std::min<long long>(n / TE, (long long)g_sms * ctas);
    const double ms = median_ms([&] { kern<<<grid, (CW + 1) * 32, smem>>>(op, n, 0, nullptr); });
    const unsigned long long bad = check<NIN>(n);
    // once more with a partial last tile (not timed)
    const int gt = (int)std::min<long long>(n_tail / TE, (long long)g_sms * ctas);
    CK(cudaMemset(g_y, 0xff, n * sizeof(double)));  // NaN: an element the kernel skips cannot pass the check
    kern<<<gt, (CW + 1) * 32, smem>>>(op, n_tail, 0, nullptr);
    CK(cudaDeviceSynchronize());
    const unsigned long long bad_tail = check<NIN>(n_tail);
    char cfg[200];
    snprintf(cfg, sizeof cfg,
             "\"tile_bytes\": %d, \"stages\": %d, \"consumer_warps\": %d, \"ctas_per_sm\": %d, \"smem_per_sm_kb\": %d",
             TILE, ST, CW, ctas, (int)(ctas * smem / 1024));
    report("ew_bulk_kernel", NIN, cfg, n, ms, bad + bad_tail);
  }
}

template <int NIN, int TILE, int ST> static void sweep_warps(long long n, long long nt) {
  run_bulk<NIN, TILE, ST, 4>(n, nt);
  run_bulk<NIN, TILE, ST, 8>(n, nt);
  run_bulk<NIN, TILE, ST, 12>(n, nt);
}
template <int NIN, int TILE> static void sweep_stages(long long n, long long nt) {
  sweep_warps<NIN, TILE, 3>(n, nt);
  sweep_warps<NIN, TILE, 4>(n, nt);
  sweep_warps<NIN, TILE, 6>(n, nt);
}
template <int NIN> static void sweep(long long n) {
  const long long nt = n - 777;
  run_direct<NIN, 3, 1>(n);
  run_direct<NIN, 3, 2>(n);
  run_direct<NIN, 4, 1>(n);
  run_direct<NIN, 4, 2>(n);
  sweep_stages<NIN, 2048>(n, nt);
  sweep_stages<NIN, 4096>(n, nt);
  sweep_stages<NIN, 8192>(n, nt);
}

int main(int argc, char** argv) {
  const int log2n = argc > 1 ? atoi(argv[1]) : 28;
  const long long n = 1ll << log2n;
  if (FILE* f = popen("nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader -i 0", "r")) {
    char buf[256] = {0};
    if (fgets(buf, sizeof buf, f)) {
      g_gpu = buf;
      while (!g_gpu.empty() && (g_gpu.back() == '\n' || g_gpu.back() == '\r')) g_gpu.pop_back();
    }
    pclose(f);
  }
  CK(cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, 0));
  for (int k = 0; k < 6; ++k) {
    CK(cudaMalloc(&g_in[k], n * sizeof(double)));
    fill_kernel<<<g_sms * 8, 256>>>(g_in[k], n, k);
  }
  CK(cudaMalloc(&g_y, n * sizeof(double)));
  CK(cudaMalloc(&g_din, 6 * sizeof(double*)));
  CK(cudaMemcpy(g_din, g_in, sizeof g_in, cudaMemcpyHostToDevice));
  CK(cudaMalloc(&g_bad, sizeof(unsigned long long)));
  CK(cudaDeviceSynchronize());
  sweep<5>(n);
  sweep<6>(n);
  for (int k = 0; k < 6; ++k) CK(cudaFree(g_in[k]));
  CK(cudaFree(g_y));
  return 0;
}
