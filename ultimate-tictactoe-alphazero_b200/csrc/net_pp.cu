// net_pp.cu -- trunk_pp_large_kernel, the large-batch form of the two-groups-in-flight trunk (body: net_pp_kernel.cuh)
#include "net_pp_kernel.cuh"

namespace uttt {
namespace pp {

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
trunk_pp_large_kernel(const __nv_bfloat16* __restrict__ wq,
                      const __nv_bfloat16* __restrict__ wq_in,
                      const __nv_bfloat16* __restrict__ wq_bias,
                      const __nv_bfloat16* __restrict__ planes,
                      const float* __restrict__ headw,
                      float* headfeat,
                      uint4* skip,
                      const int32_t* __restrict__ count,
                      int cap1,                     // trunk_pp_cap1: smaller batches are trunk_auto_kernel's
                      long long* dbg) {
    const int n_pos = *count;
    if (n_pos <= cap1) return;
    count_batch(dbg, n_pos);
    trunk_pp_body<2>(wq, wq_in, wq_bias, planes, headw, headfeat, skip, dbg, n_pos);
}

}  // namespace pp


cudaError_t trunk_pp_init() {
    return cudaFuncSetAttribute(pp::trunk_pp_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pp::Cfg<2>::SMEM_BYTES);
}

// batches above trunk_pp_cap1 (what launch_trunk_auto leaves over): super-groups of up to 10 positions per CTA pair
cudaError_t launch_trunk_pp_large(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count,
                                  int max_rows, float* skip, int n_sm, cudaStream_t s, long long* dbg) {
    int pairs = n_sm / 2;
    if (max_rows < pairs) pairs = max_rows < 1 ? 1 : max_rows;
    pp::trunk_pp_large_kernel<<<2 * pairs, pp::THREADS, pp::Cfg<2>::SMEM_BYTES, s>>>(
        w.res_w_2sm, w.conv_in_w_2sm, w.bias_blk_2sm, planes, w.head_w, headfeat, reinterpret_cast<uint4*>(skip), count,
        trunk_pp_cap1(n_sm), dbg);
    return cudaGetLastError();
}

int trunk_pp_cap1(int n_sm) { return (n_sm / 2) * (pp::Cfg<1>::MAX_PA + pp::Cfg<1>::MAX_PB); }

}  // namespace uttt
