// net_pp.cu -- trunk_pp_large_kernel, the large-batch form of the two-groups-in-flight trunk (body: net_pp_kernel.cuh), and
// the weight splitting for the cta_group::2 B operand
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
    trunk_pp_body<2>(wq, wq_in, wq_bias, planes, headw, headfeat, skip, dbg, n_pos, nullptr);
}

}  // namespace pp


// [block][2 k-panels][128 co][8] -> [stage][cta rank][block of the stage][2 k-panels][64 co][8]: each CTA of a pair holds the
// output channels 64*rank .. 64*rank+63 of the B operand, and its share of a weight stage is one contiguous bulk copy
// (subs = 2: split-bf16 arrays, [block][hi, lo][2][128][8] -> [stage][rank][block][hi, lo][2][64][8])
__global__ void split_weights_2sm_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int n_blocks, int bps, int subs) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;               // one 16-byte (co, 8 ci) unit
    if (i >= n_blocks * subs * 256) return;
    int u = i >> 8, pnl = (i >> 7) & 1, co = i & 127;
    int b = u / subs, sub = u - b * subs;
    int stage = b / bps, j = b - stage * bps, r = co >> 6;
    dst[(((((size_t)stage * 2 + r) * bps + j) * subs + sub) * 2 + pnl) * 64 + (co & 63)] = src[i];
}
cudaError_t launch_split_weights_2sm(const __nv_bfloat16* src, __nv_bfloat16* dst, int n_blocks, int blocks_per_stage, cudaStream_t s,
                                     int subs) {
    split_weights_2sm_kernel<<<(n_blocks * subs * 256 + 255) / 256, 256, 0, s>>>(reinterpret_cast<const uint4*>(src),
                                                                                    reinterpret_cast<uint4*>(dst), n_blocks,
                                                                                    blocks_per_stage, subs);
    return cudaGetLastError();
}

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
