// The contraction engines and their companion kernels, compiled once for the whole library; the stages call them
// through the declarations in engines.cuh.
#include "gemm_gen.cuh"
#include "gemm_simt.cuh"
#include "gemm_tma.cuh"
#include "norm_ops.cuh"
#include "tc_ops.cuh"

template int gemm_simt_launch<XM_DIRECT>(const GemmP&, cudaStream_t);
template int gemm_simt_launch<XM_NORM_RELU>(const GemmP&, cudaStream_t);
template int gemm_simt_launch<XM_PAIR_MUL>(const GemmP&, cudaStream_t);
template int gemm_simt_launch<XM_PAIR_ABS>(const GemmP&, cudaStream_t);
template int gemm_simt_launch<XM_PAIR_SUB>(const GemmP&, cudaStream_t);
template int gemm_simt_launch<XM_CONV3>(const GemmP&, cudaStream_t);

#define GEN_LAUNCH(GEN)                                                                                               \
  template int gemm_gen_launch<GEN>(const GemmP&, const uint4*, float, const float*, int, const float*, const float*, \
                                    int, int, int, cudaStream_t)
GEN_LAUNCH(gen::GEN_PAIR_MUL);
GEN_LAUNCH(gen::GEN_PAIR_ABS);
GEN_LAUNCH(gen::GEN_PAIR_SUB);
GEN_LAUNCH(gen::GEN_NORM);
GEN_LAUNCH(gen::GEN_COPY);
