// net_auto.cu -- trunk_auto_kernel: ONE launch per evaluator round.  The queue length is only known on the device, and a
// kernel that exits at once still costs a full kernel boundary (3.4 us under ncu, ~6 us between dependent launches), so
// the bodies sit behind one device-side branch on the batch size: batches of up to one wave of 5-position groups run
// tc2::trunk_tc2_body (next layer overlaps the epilogue), larger ones pp::trunk_pp_body<1> (two groups in flight).  Both
// issue cta_group::2 MMAs on per-CTA weight halves and use 19 warps, clusters of two CTAs and the same grid; shared memory
// is the larger footprint.  Batches above 7 positions per pair are left to a second launch, trunk_pp_large_kernel
// (net_pp.cu).
#include "heads_fc.cuh"
#include "net_pp_kernel.cuh"
#include "net_tc2_kernel.cuh"

namespace uttt {

static_assert(tc2::Cfg<>::THREADS == pp::THREADS, "one block size for both bodies");
constexpr int AUTO_SMEM = tc2::Cfg<>::SMEM_BYTES > pp::Cfg<1>::SMEM_BYTES ? tc2::Cfg<>::SMEM_BYTES : pp::Cfg<1>::SMEM_BYTES;
static_assert(HEADS_SMEM_BYTES <= AUTO_SMEM, "the fused heads reuse the trunk's shared memory");

// Slot mode.  With an atomic counter the leaves of a round land in the evaluator queue in arrival order, which differs
// from run to run; that is harmless as long as every row is computed by the same arithmetic, but the one-tile group of
// trunk_pp_body<1> accumulates in another order (split K), so WHICH leaves fall into it must not depend on arrival order
// if a self-play run is to be reproducible.  In slot mode a leaf stays in the slot of its tree (planes[slot], policy[slot],
// value[slot]) and flags[slot] says whether the slot holds one this round; row i of the batch is the i-th flagged slot.
// Every CTA derives the batch size and the slots of its own <= 7 positions from the same scan (warp 0, one L2 round trip).
constexpr int SLOT_CHUNKS = 17;                                 // 544 slots >= one group per CTA pair on 148 SMs (518)
__device__ __forceinline__ void scan_slots(const uint8_t* __restrict__ flags, int n_slots, int n_pairs, int pair, int small_cap,
                                           int* s_npos, int* s_src) {
    const int lane = threadIdx.x & 31;
    uint32_t mine = 0;                                          // bit j: slot lane + 32 j holds a leaf
#pragma unroll
    for (int j = 0; j < SLOT_CHUNKS; j++) {
        const int idx = lane + 32 * j;
        if (idx < n_slots && flags[idx]) mine |= 1u << j;
    }
    uint32_t bal[SLOT_CHUNKS];
    int n_pos = 0;
#pragma unroll
    for (int j = 0; j < SLOT_CHUNKS; j++) {
        bal[j] = __ballot_sync(0xFFFFFFFFu, (mine >> j) & 1u);
        n_pos += __popc(bal[j]);
    }
    const int P = n_pos <= small_cap ? tc2::group_positions(n_pos, n_pairs) : pp::pair_positions<1>(n_pos, n_pairs);
    const int first = pair * P, last = min(n_pos, first + P);
    int run = 0;
#pragma unroll
    for (int j = 0; j < SLOT_CHUNKS; j++) {
        if ((bal[j] >> lane) & 1u) {
            const int rank = run + __popc(bal[j] & ((1u << lane) - 1u));
            if (rank >= first && rank < last) s_src[rank - first] = lane + 32 * j;
        }
        run += __popc(bal[j]);
    }
    if (lane == 0) *s_npos = n_pos;
}

constexpr int AUTO_SMEM_TOTAL = AUTO_SMEM + 64;                 // + the slot table of the pair and the batch size

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(pp::THREADS, 1)
trunk_auto_kernel(const __nv_bfloat16* __restrict__ res_w8, const __nv_bfloat16* __restrict__ conv_in_w8,     // tc2: 8-block stages
                  const __nv_bfloat16* __restrict__ res_w18, const __nv_bfloat16* __restrict__ conv_in_w18,   // pp<1>: 18-block stages
                  const __nv_bfloat16* __restrict__ bias_2sm,     // the bias blocks of both (all per-CTA weight halves)
                  const __nv_bfloat16* __restrict__ planes, const float* __restrict__ headw, float* headfeat, uint4* skip,
                  const int32_t* __restrict__ count, int small_cap, int cap1, long long* dbg,
                  HeadsFC fc, float* policy, float* value /* null: the heads' FC layers are a separate kernel */,
                  const uint8_t* __restrict__ slot_flags, int n_slots /* slot mode (needs the fused heads), else null */) {
    extern __shared__ __align__(1024) uint8_t smem[];
    pdl_trigger();          // the next round's tree kernel may be scheduled (it waits for this grid's policy / value rows)
    pdl_wait();             // this round's tree kernel has finished: slot flags / queue length and planes are visible
    const bool stamp = dbg && blockIdx.x == 0 && threadIdx.x == 0;          // diagnostics: phases of CTA 0
    if (stamp) dbg[200] = clock64();
    const int n_pairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
    int* s_src = reinterpret_cast<int*>(smem + AUTO_SMEM);                  // [8] slots of this pair's positions
    int* s_npos = s_src + 8;
    int n_pos;
    if (slot_flags) {
        if (threadIdx.x < 32) scan_slots(slot_flags, n_slots, n_pairs, pair, small_cap, s_npos, s_src);
        __syncthreads();
        n_pos = *s_npos;
    } else {
        n_pos = *count;
    }
    const int* src = slot_flags ? s_src : nullptr;
    const bool small = n_pos <= small_cap;
    if (n_pos <= 0 || n_pos > cap1) return;        // (larger batches are trunk_pp_large_kernel's)
    tcx::count_batch(dbg, n_pos);
    // (with the statements above and the branches below in this order ptxas fits the kernel into 96 registers without
    // spills; the other orders tried spill 32-64 bytes)
    if (!small)
        pp::trunk_pp_body<1>(res_w18, conv_in_w18, bias_2sm, planes, headw, headfeat, skip, dbg, n_pos, src);
    else
        tc2::trunk_tc2_body<false>(res_w8, conv_in_w8, bias_2sm, planes, headw, headfeat, skip, dbg, n_pos, src, 0, false);
    if (stamp) dbg[201] = clock64();
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
    heads_fc_block(fc, headfeat, row0, 2, np, policy, value, 1, reinterpret_cast<float*>(smem), stamp ? dbg + 203 : nullptr,
                   src ? src + rank : nullptr);
    if (stamp) dbg[202] = clock64();
}

cudaError_t trunk_auto_init() {
    return cudaFuncSetAttribute(trunk_auto_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AUTO_SMEM_TOTAL);
}

// batches of 1 .. 7 positions per CTA pair in one launch; larger ones are left to launch_trunk_pp_large.
// policy / value non-null: the heads' FC layers run in the kernel's tail (only valid if max_rows <= trunk_pp_cap1).
// slot_flags non-null: slot mode (see scan_slots; needs the fused heads and n_slots <= 32 * SLOT_CHUNKS)
cudaError_t launch_trunk_auto(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count, int max_rows,
                              float* skip, int n_sm, cudaStream_t s, long long* dbg, float* policy, float* value,
                              const uint8_t* slot_flags, int n_slots) {
    int pairs = n_sm / 2;
    if (max_rows < pairs) pairs = max_rows < 1 ? 1 : max_rows;
    const int small_cap = (n_sm / 2) * tc2::Cfg<>::MAX_P;
    const int cap1 = (n_sm / 2) * (pp::Cfg<1>::MAX_PA + pp::Cfg<1>::MAX_PB);
    if (policy && max_rows > cap1) return cudaErrorInvalidValue;
    if (slot_flags && (!policy || n_slots > 32 * SLOT_CHUNKS || n_slots > max_rows)) return cudaErrorInvalidValue;
    return launch_pdl(trunk_auto_kernel, dim3(2 * pairs), dim3(pp::THREADS), AUTO_SMEM_TOTAL, s, w.res_w_2sm, w.conv_in_w_2sm,
                      w.res_w_2sm18, w.conv_in_w_2sm18, w.bias_blk_2sm, planes, w.head_w, headfeat, reinterpret_cast<uint4*>(skip),
                      count, small_cap, cap1, dbg, heads_fc_of(w), policy, value, slot_flags, n_slots);
}

}  // namespace uttt
