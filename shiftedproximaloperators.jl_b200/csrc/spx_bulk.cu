// spx_bulk.cu -- ew_bulk_kernel for the operators that declare BULK, in a module of its own (spx_elementwise.cuh)
#include "spx_bulk.cuh"
#include "spx_ops.cuh"

namespace spx {

#define SPX_BULK_OP(...)                                                                                          \
  template int32_t ew_bulk_launch<__VA_ARGS__>(spx_ctx*, cudaStream_t, const __VA_ARGS__&, int64_t, int64_t, Partial*, \
                                               int*);
#define SPX_BULK_R(R)                                                                                             \
  SPX_BULK_OP(ProxL1Box<R, false>)                                                                                \
  SPX_BULK_OP(ProxL1Box<R, true>)                                                                                 \
  SPX_BULK_OP(ProxL0Box<R, false>)                                                                                \
  SPX_BULK_OP(ProxL0Box<R, true>)                                                                                 \
  SPX_BULK_OP(IproxL0Box<R, false>)                                                                               \
  SPX_BULK_OP(IproxL0Box<R, true>)
SPX_BULK_R(double)
SPX_BULK_R(float)

}  // namespace spx
