// net_auto.cu -- trunk_auto_kernel: ONE launch per evaluator round.  The queue length is only known on the device, and a
// kernel that exits at once still costs a full kernel boundary (3.4 us under ncu, ~6 us between dependent launches), so
// the bodies sit behind one device-side branch on the batch size: batches of up to one wave of 5-position groups run
// tc2::trunk_tc2_body (next layer overlaps the epilogue), larger ones pp::trunk_pp_body<1> (two groups in flight).  The
// two schedules are built from the same CTA-pair pipeline pieces (trunk_pair.cuh): cta_group::2 MMAs on per-CTA weight
// halves, 19 warps, clusters of two CTAs and the same grid; shared memory is the larger footprint.  Batches above 7
// positions per pair are left to a second launch, trunk_pp_large_kernel (net_pp.cu).
#include "heads_fc.cuh"
#include "net_pp_kernel.cuh"
#include "net_tc2_kernel.cuh"

namespace uttt {

static_assert(tc2::Cfg<>::THREADS == pp::THREADS, "one block size for both bodies");
constexpr int AUTO_SMEM = tc2::Cfg<>::SMEM_BYTES > pp::Cfg<1>::SMEM_BYTES ? tc2::Cfg<>::SMEM_BYTES : pp::Cfg<1>::SMEM_BYTES;
static_assert(HEADS_SMEM_BYTES <= AUTO_SMEM, "the fused heads reuse the trunk's shared memory");

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(pp::THREADS, 1)
trunk_auto_kernel(const __nv_bfloat16* __restrict__ res_w8, const __nv_bfloat16* __restrict__ conv_in_w8,     // tc2: 8-block stages
                  const __nv_bfloat16* __restrict__ res_w18, const __nv_bfloat16* __restrict__ conv_in_w18,   // pp<1>: 18-block stages
                  const __nv_bfloat16* __restrict__ bias_2sm,     // the bias blocks of both (all per-CTA weight halves)
                  const __nv_bfloat16* __restrict__ planes, const float* __restrict__ headw, float* headfeat, uint4* skip,
                  const int32_t* __restrict__ count, int small_cap, int cap1, long long* dbg,
                  HeadsFC fc, float* policy, float* value /* null: the heads' FC layers are a separate kernel */) {
    extern __shared__ __align__(1024) uint8_t smem[];
    pdl_trigger();          // the next round's tree kernel may be scheduled (it waits for this grid's policy / value rows)
    pdl_wait();             // this round's tree kernel has finished: queue length and planes are visible
    const int n_pairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
    const int n_pos = *count;
    const bool small = n_pos <= small_cap;
    if (n_pos <= 0 || n_pos > cap1) return;        // (larger batches are trunk_pp_large_kernel's)
    tcx::count_batch(dbg, n_pos);
    // (at the 96-register cap ptxas spills 24 bytes here: n_pos and loop-invariant values of the bodies, stored once and
    // reloaded from L1, three of the loads in pp<1>'s issuer loop; no statement order tried avoids that)
    if (!small)
        pp::trunk_pp_body<1>(res_w18, conv_in_w18, bias_2sm, planes, headw, headfeat, skip, dbg, n_pos);
    else
        tc2::trunk_tc2_body<false>(res_w8, conv_in_w8, bias_2sm, planes, headw, headfeat, skip, dbg, n_pos, 0, false);
    if (policy == nullptr) return;
    // Fused heads (the host passes policy / value only if no batch can exceed one group per pair): the pair's head
    // features were written to global memory by both CTAs' last epilogues and ordered by the cluster barrier that ends
    // the body (release / acquire); they are read back with ld.global.cg.  The two CTAs take alternate positions of
    // the pair (at most 4 each); the body's shared memory is free now.
    const int P = small ? tc2::group_positions(n_pos, n_pairs) : pp::pair_positions<1>(n_pos, n_pairs);
    const int first = pair * P, last = min(n_pos, first + P);
    const int rank = (int)tcx::cluster_rank();
    const int row0 = first + rank;
    const int np = row0 < last ? (last - row0 + 1) >> 1 : 0;
    static_assert((pp::Cfg<1>::MAX_PA + pp::Cfg<1>::MAX_PB + 1) / 2 <= HEADS_P, "one heads call per CTA");
    if (np == 0) return;
    heads_fc_block(fc, headfeat, row0, 2, np, policy, value, 1, reinterpret_cast<float*>(smem));
}

cudaError_t trunk_auto_init() {
    return cudaFuncSetAttribute(trunk_auto_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AUTO_SMEM);
}

// batches of 1 .. 7 positions per CTA pair in one launch; larger ones are left to launch_trunk_pp_large.
// policy / value non-null: the heads' FC layers run in the kernel's tail (only valid if max_rows <= trunk_pp_cap1).
cudaError_t launch_trunk_auto(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count, int max_rows,
                              float* skip, int n_sm, cudaStream_t s, long long* dbg, float* policy, float* value) {
    int pairs = n_sm / 2;
    if (max_rows < pairs) pairs = max_rows < 1 ? 1 : max_rows;
    const int small_cap = (n_sm / 2) * tc2::Cfg<>::MAX_P;
    const int cap1 = (n_sm / 2) * (pp::Cfg<1>::MAX_PA + pp::Cfg<1>::MAX_PB);
    if (policy && max_rows > cap1) return cudaErrorInvalidValue;
    return launch_pdl(trunk_auto_kernel, dim3(2 * pairs), dim3(pp::THREADS), AUTO_SMEM, s, w.res_w_2sm, w.conv_in_w_2sm,
                      w.res_w_2sm18, w.conv_in_w_2sm18, w.bias_blk_2sm, planes, w.head_w, headfeat, reinterpret_cast<uint4*>(skip),
                      count, small_cap, cap1, dbg, heads_fc_of(w), policy, value);
}

}  // namespace uttt
