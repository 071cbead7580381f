// net_tc2.cu -- trunk_x3_kernel, the split-bf16 ("bf16x3") trunk behind UTTT_EVAL_NET_BF16X3, and its launcher (body:
// net_tc2_kernel.cuh; the bf16 trunk reaches the same body through trunk_auto_kernel, net_auto.cu).
#include "net_tc2_kernel.cuh"

namespace uttt {
namespace tc2 {

// The split-bf16 trunk.  A pair's share of the batch, ceil(n / pairs) positions, is evaluated as consecutive groups of up
// to 5 positions (2 + 2 accumulator tiles), each by one complete pass of the body (set-up and tear-down are ~1 % of a
// pass here: every layer issues 3 x 72 MMAs per tile).  7 positions per pair -- the 500-game cycle -- cost 2 + 1 tile
// times (groups of 5 and 2) instead of the 2 + 2 of two waves of 5-position groups over the whole grid.
// cta_group::2 MMAs, every CTA streams its output-channel half of the split weights (see Cfg: with cta_group::1 MMAs a
// one-tile pass was 13 % slower -- 347 -> 301 us at up to 148 positions, 1035 -> 982 us at 500 -- with bit-identical rows).
constexpr int X3_SMEM = Cfg<true>::SMEM_BYTES;
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<true>::THREADS, 1)
trunk_x3_kernel(const __nv_bfloat16* __restrict__ wq, const __nv_bfloat16* __restrict__ wq_in,
                const __nv_bfloat16* __restrict__ wq_bias, const __nv_bfloat16* __restrict__ planes,
                const float* __restrict__ headw, float* headfeat, uint4* skip, const int32_t* __restrict__ count,
                long long* dbg) {
    pdl_trigger();          // the heads kernel behind this one may be scheduled (it waits for this grid's head features)
    pdl_wait();             // this round's tree kernel has finished: queue length and planes are visible
    const int n_pos = *count;
    if (n_pos <= 0) return;
    count_batch(dbg, n_pos);
    const int n_pairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
    const int per_pair = (n_pos + n_pairs - 1) / n_pairs;
    const int first = pair * per_pair, last = min(n_pos, first + per_pair);
    for (int off = first; off < last; off += Cfg<true>::MAX_P)
        trunk_tc2_body<true>(wq, wq_in, wq_bias, planes, headw, headfeat, skip, off == first ? dbg : nullptr,
                             min(Cfg<true>::MAX_P, last - off), nullptr, off, true);     // (dbg: timeline of the first pass)
}

}  // namespace tc2


cudaError_t trunk_tc2_init() {
    return cudaFuncSetAttribute(tc2::trunk_x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::X3_SMEM);
}

// split-bf16 trunk: any batch size in one launch (see trunk_x3_kernel)
// (skip: 128 KiB per CTA, fp32)
cudaError_t launch_trunk_x3(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count,
                            int max_rows, float* skip, int n_sm, cudaStream_t s, long long* dbg) {
    int pairs = n_sm / 2;
    if (max_rows < pairs) pairs = max_rows < 1 ? 1 : max_rows;
    return launch_pdl(tc2::trunk_x3_kernel, dim3(2 * pairs), dim3(tc2::Cfg<true>::THREADS), tc2::X3_SMEM, s, w.res_w_x3p,
                      w.conv_in_w_x3p, w.bias_blk_x3p, planes, w.head_w, headfeat, reinterpret_cast<uint4*>(skip), count, dbg);
}

}  // namespace uttt
