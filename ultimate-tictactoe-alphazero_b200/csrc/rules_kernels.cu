// rules_kernels.cu -- bitboard rules kernels over arrays of packed states in HBM, and the
// host-side single-state helpers behind the `uttt_cpp.State` shim.
//
// Replaces UTTT::State (cpp/uttt_game.cpp:9-280).  All kernels are HBM-bound integer/byte work:
// one thread per 32-byte state, two 128-bit loads / stores per state, fully coalesced
// (a warp touches 1 KiB of contiguous states); grids are sized from n, no shared memory needed.
#include <stdarg.h>
#include <string.h>

#include <string>

#include "common.cuh"

namespace uttt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

__device__ __forceinline__ PackedState load_state(const PackedState* p) {
    PackedState s;
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    s.w[0] = a.x; s.w[1] = a.y; s.w[2] = a.z; s.w[3] = a.w;
    s.w[4] = b.x; s.w[5] = b.y; s.w[6] = b.z; s.w[7] = b.w;
    return s;
}
__device__ __forceinline__ void store_state(PackedState* p, const PackedState& s) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(s.w[0], s.w[1], s.w[2], s.w[3]);
    q[1] = make_uint4(s.w[4], s.w[5], s.w[6], s.w[7]);
}

// cpp/uttt_game.cpp:97-145
__global__ void __launch_bounds__(256) step_kernel(const PackedState* __restrict__ in, const int32_t* __restrict__ act,
                                                   PackedState* __restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PackedState s = load_state(in + i), o;
    next_state(s, __ldg(act + i), o);
    store_state(out + i, o);
}

// cpp/uttt_game.cpp:77-89,148-191
__global__ void __launch_bounds__(256) legal_kernel(const PackedState* __restrict__ in, uint4* __restrict__ masks,
                                                    uint8_t* __restrict__ status, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PackedState s = load_state(in + i);
    uint32_t lm[3];
    int cnt = legal_mask(s, lm);
    masks[i] = make_uint4(lm[0], lm[1], lm[2], (uint32_t)cnt);
    if (status) status[i] = (uint8_t)status_of(s, cnt);
}

// The 27 nine-bit picture rows of a position (3 planes x 9 rows), one per lane: lane 9*plane + R holds row R of
// plane (0 mover, 1 opponent, 2 legal).  Elements are then fetched with one shuffle each.
__device__ __forceinline__ uint32_t warp_picture_rows(const PackedState& s, int lane) {
    uint32_t lm[3];
    legal_mask(s, lm);
    int plane = lane / 9, R = lane - 9 * plane;
    uint32_t x[3];
#pragma unroll
    for (int j = 0; j < 3; j++) x[j] = (plane == 0) ? s.w[j] : (plane == 1 ? s.w[3 + j] : lm[j]);
    return (lane < 27) ? picture_row(x, R) : 0u;
}

// ---- encode / gather: bit string per block, 16-byte stores ----
// A position's planes are 243 cells that are 0 or 1, i.e. a 243-bit string; a block of PLANES_POS positions owns one
// contiguous, 16-byte aligned slice of the output.  Phase 1 (thread per position): build the position's bit string
// in output element order from the bitboards with word-parallel bit permutations and OR it into the block's
// string in shared memory at bit 243*t.  Phase 2 (all threads, position boundaries forgotten): every 16-byte output
// vector is a 4-bit (fp32) or 8-bit (bf16) slice of the string, expanded through a 16-entry table.  HBM traffic is
// the algorithmic 32 B in + 972 B (fp32 HWC) or 486 B (bf16 CHW) out per position.
constexpr int PLANES_POS = 256;                                  // positions per block
constexpr int PLANES_WORDS = (PLANES_POS * 243 + 31) / 32 + 8;   // block bit string (+ spill of the last position)

// 27-bit word of 3 sub-boards x 9 cells  ->  3 picture rows x 9 columns: transposes the 3x3 grid of 3-bit groups
__device__ __forceinline__ uint32_t rows27(uint32_t w) {
    uint32_t t = ((w >> 6) ^ w) & 0x00038038u;      // groups (board 0,row 1)<->(1,0) and (1,2)<->(2,1)
    w ^= t | (t << 6);
    t = ((w >> 12) ^ w) & 0x000001C0u;              // groups (0,2)<->(2,0)
    w ^= t | (t << 12);
    return w;
}
// bit i -> bit 3i for a 9-bit value
__device__ __forceinline__ uint32_t spread9x3(uint32_t x) {
    x = (x | (x << 16)) & 0x030000FFu;
    x = (x | (x << 8)) & 0x0300F00Fu;
    x = (x | (x << 4)) & 0x030C30C3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

// nine 27-bit chunks at bit 27*m -> the block string at bit 243*t
__device__ __forceinline__ void or_position_bits(uint32_t* S, const uint32_t chunk[9], int t) {
    uint32_t W[8];
#pragma unroll
    for (int k = 0; k < 8; k++) W[k] = 0u;
#pragma unroll
    for (int m = 0; m < 9; m++) {
        const int off = 27 * m, k = off >> 5, sh = off & 31;
        W[k] |= chunk[m] << sh;
        if (sh > 5) W[k + 1] |= chunk[m] >> (32 - sh);
    }
    int bit0 = 243 * t, b = bit0 >> 5, o = bit0 & 31;
#pragma unroll
    for (int k = 0; k <= 8; k++) {
        uint32_t hi = (k < 8) ? W[k] : 0u, lo = (k > 0) ? W[k - 1] : 0u;
        uint32_t v = __funnelshift_l(lo, hi, o);
        if (v) atomicOr(S + b + k, v);
    }
}

template <bool HWC>
__device__ __forceinline__ void position_chunks(const PackedState& s, uint32_t chunk[9]) {
    uint32_t lm[3];
    legal_mask(s, lm);
    if (HWC) {          // element (R*9 + C)*3 + plane: chunk R = the three planes' rows R interleaved bit by bit
#pragma unroll
        for (int j = 0; j < 3; j++) {
            uint32_t a = rows27(s.w[j]), b = rows27(s.w[3 + j]), c = rows27(lm[j]);
#pragma unroll
            for (int sr = 0; sr < 3; sr++)
                chunk[3 * j + sr] = spread9x3((a >> (9 * sr)) & 0x1FFu) | (spread9x3((b >> (9 * sr)) & 0x1FFu) << 1) |
                                    (spread9x3((c >> (9 * sr)) & 0x1FFu) << 2);
        }
    } else {            // element plane*81 + R*9 + C: chunk 3*plane + j = picture rows 3j..3j+2 of the plane
#pragma unroll
        for (int j = 0; j < 3; j++) {
            chunk[j] = rows27(s.w[j]);
            chunk[3 + j] = rows27(s.w[3 + j]);
            chunk[6 + j] = rows27(lm[j]);
        }
    }
}

template <bool HWC>
__device__ __forceinline__ void block_bit_string(uint32_t* S, const PackedState* __restrict__ in, int64_t pos0,
                                                 int npos) {
    for (int k = threadIdx.x; k < PLANES_WORDS; k += blockDim.x) S[k] = 0u;
    __syncthreads();
    if ((int)threadIdx.x < npos) {
        uint32_t chunk[9];
        position_chunks<HWC>(load_state(in + pos0 + threadIdx.x), chunk);
        or_position_bits(S, chunk, threadIdx.x);
    }
    __syncthreads();
}

// cpp/uttt_game.cpp:244-280: float HWC (9,9,3)
__global__ void __launch_bounds__(PLANES_POS) encode_kernel(const PackedState* __restrict__ in,
                                                            float* __restrict__ planes, int64_t n) {
    __shared__ uint32_t S[PLANES_WORDS];
    __shared__ float4 lut[16];
    if (threadIdx.x < 16) {
        int v = threadIdx.x;
        lut[v] = make_float4((float)(v & 1), (float)((v >> 1) & 1), (float)((v >> 2) & 1), (float)((v >> 3) & 1));
    }
    int64_t pos0 = (int64_t)blockIdx.x * PLANES_POS;
    int npos = (int)min((int64_t)PLANES_POS, n - pos0);
    block_bit_string<true>(S, in, pos0, npos);
    float* out = planes + pos0 * 243;
    int total = npos * 243, nvec = total >> 2;
    float4* out4 = reinterpret_cast<float4*>(out);
    for (int q = threadIdx.x; q < nvec; q += PLANES_POS) out4[q] = lut[(S[q >> 3] >> ((q & 7) * 4)) & 15u];
    int e = 4 * nvec + threadIdx.x;
    if (e < total) out[e] = (float)((S[e >> 5] >> (e & 31)) & 1u);
}

// leaf gather (pv_mcts_cpp.py:47-60): bf16 CHW (3,9,9) rows of the network's input batch
__global__ void __launch_bounds__(PLANES_POS) gather_planes_kernel(const PackedState* __restrict__ in,
                                                                   __nv_bfloat16* __restrict__ planes, int64_t n) {
    __shared__ uint32_t S[PLANES_WORDS];
    __shared__ uint2 lut[16];
    if (threadIdx.x < 16) {
        uint32_t v = threadIdx.x;
        lut[v] = make_uint2(((v & 1u) ? 0x3F80u : 0u) | ((v & 2u) ? 0x3F800000u : 0u),
                            ((v & 4u) ? 0x3F80u : 0u) | ((v & 8u) ? 0x3F800000u : 0u));
    }
    int64_t pos0 = (int64_t)blockIdx.x * PLANES_POS;
    int npos = (int)min((int64_t)PLANES_POS, n - pos0);
    block_bit_string<false>(S, in, pos0, npos);
    __nv_bfloat16* out = planes + pos0 * 243;
    int total = npos * 243, nvec = total >> 3;
    uint4* out4 = reinterpret_cast<uint4*>(out);
    for (int q = threadIdx.x; q < nvec; q += PLANES_POS) {
        uint32_t byte = (S[q >> 2] >> ((q & 3) * 8)) & 255u;
        uint2 lo = lut[byte & 15u], hi = lut[byte >> 4];
        out4[q] = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
    int e = 8 * nvec + threadIdx.x;
    if (e < total)
        out[e] = __ushort_as_bfloat16(((S[e >> 5] >> (e & 31)) & 1u) ? (unsigned short)0x3F80 : (unsigned short)0);
}

// Same outputs for a destination that is not 16-byte aligned (a caller's sub-view): one warp per position, 4-byte /
// 2-byte stores, every store instruction of the warp contiguous.
__global__ void __launch_bounds__(256) encode_unaligned_kernel(const PackedState* __restrict__ in,
                                                               float* __restrict__ planes, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (i >= n) return;
    uint32_t rows = warp_picture_rows(load_state(in + i), lane);
    float* out = planes + i * 243;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        int e = lane + 32 * k;                  // e = (R*9 + C)*3 + ch
        int cell = e / 3, ch = e - 3 * cell;
        int R = cell / 9, C = cell - 9 * R;
        uint32_t m = __shfl_sync(0xFFFFFFFFu, rows, (9 * ch + R) & 31);
        if (e < 243) out[e] = (float)((m >> C) & 1u);
    }
}
__global__ void __launch_bounds__(256) gather_planes_unaligned_kernel(const PackedState* __restrict__ in,
                                                                      __nv_bfloat16* __restrict__ planes, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (i >= n) return;
    uint32_t rows = warp_picture_rows(load_state(in + i), lane);
    __nv_bfloat16* out = planes + i * 243;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        int e = lane + 32 * k;                  // e = ch*81 + R*9 + C  ->  row index e/9 = 9*ch + R
        int row = e / 9, C = e - 9 * row;
        uint32_t m = __shfl_sync(0xFFFFFFFFu, rows, row & 31);
        if (e < 243) out[e] = __ushort_as_bfloat16(((m >> C) & 1u) ? (unsigned short)0x3F80 : (unsigned short)0);
    }
}

// Whole random games with the state in registers: HBM traffic is 16 B out per game, the kernel is
// integer-issue bound.  One thread per game (config 2 of BASELINE.json: 2^20 concurrent playouts).
__global__ void __launch_bounds__(128) playout_kernel(uint32_t seed, uint64_t game0, int64_t n,
                                                      uint64_t* __restrict__ digests, int32_t* __restrict__ plies,
                                                      int32_t* __restrict__ results) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t game = game0 + (uint64_t)i;
    PackedState s;
    init_state(s);
    uint64_t h = 0xCBF29CE484222325ull;
    int t = 0;
    for (;;) {
        uint32_t lm[3];
        int cnt = legal_mask(s, lm);      // 0 when the mover has already lost
        if (cnt == 0) break;
        Philox4 r = philox4x32(seed, 0u, (uint32_t)game, (uint32_t)(game >> 32), (uint32_t)t, 0u);
        int a = nth_legal(lm, (int)(r.x % (uint32_t)cnt));
        h = fnv64(h, (uint32_t)a);
        h = fnv64(h, lm[0]); h = fnv64(h, lm[1]); h = fnv64(h, lm[2]);
        h = fnv64(h, s.w[6]);
        PackedState o;
        next_state(s, a, o);
        s = o;
        t++;
    }
    bool lose = is_lose(s);
#pragma unroll
    for (int k = 0; k < 7; k++) h = fnv64(h, s.w[k]);
    h = fnv64(h, lose ? 1u : 2u);
    digests[i] = h;
    plies[i] = t;
    results[i] = lose ? (is_first_player(s) ? 2 : 1) : 0;
}

}  // namespace uttt

using namespace uttt;

extern "C" {

const char* uttt_last_error(void) { return g_err; }
int uttt_abi_version(void) { return UTTT_ABI_VERSION; }

int uttt_device_check(int device) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no CUDA device visible: libuttt_b200 has no CPU fallback");
        return 1;
    }
    UTTT_CHECK(device >= 0 && device < n, "device %d out of range (%d visible)", device, n);
    cudaDeviceProp p;
    UTTT_CUDA_OK(cudaGetDeviceProperties(&p, device));
    UTTT_CHECK(p.major == 10, "device %d is sm_%d%d; this library is built for sm_100a only", device, p.major, p.minor);
    return 0;
}

// ---- host single-state helpers -------------------------------------------------------------
int uttt_state_init(uint32_t* state) {
    memset(state, 0, 32);
    return 0;
}

int uttt_state_next(const uint32_t* state, int action, uint32_t* out) {
    UTTT_CHECK(action >= 0 && action < 81, "action %d out of range [0,81)", action);
    PackedState s, o;
    memcpy(s.w, state, 32);
    next_state(s, action, o);
    memcpy(out, o.w, 32);
    return 0;
}

int uttt_state_legal_actions(const uint32_t* state, int32_t* out81, int* n_out) {
    PackedState s;
    memcpy(s.w, state, 32);
    uint32_t lm[3];
    int n = legal_mask(s, lm), k = 0;
    for (int a = 0; a < 81; a++)
        if (legal_bit(lm, a)) out81[k++] = a;
    *n_out = n;
    return 0;
}

int uttt_state_flags(const uint32_t* state, int* flags_out) {
    PackedState s;
    memcpy(s.w, state, 32);
    uint32_t lm[3];
    int n = legal_mask(s, lm);
    bool lose = is_lose(s), draw = !lose && n == 0;
    *flags_out = (lose ? 1 : 0) | (draw ? 2 : 0) | ((lose || draw) ? 4 : 0) | (is_first_player(s) ? 8 : 0);
    return 0;
}

int uttt_state_encode(const uint32_t* state, float* out243) {
    PackedState s;
    memcpy(s.w, state, 32);
    uint32_t lm[3];
    legal_mask(s, lm);
    for (int R = 0; R < 9; R++)
        for (int C = 0; C < 9; C++) {
            int a = action_of_rc(R, C);
            float* o = out243 + (R * 9 + C) * 3;
            o[0] = stone_me(s, a) ? 1.0f : 0.0f;
            o[1] = stone_opp(s, a) ? 1.0f : 0.0f;
            o[2] = legal_bit(lm, a) ? 1.0f : 0.0f;
        }
    return 0;
}

int uttt_state_symmetry(const uint32_t* state, int g, uint32_t* out, int32_t* action_map81) {
    UTTT_CHECK(state && out, "null argument");
    UTTT_CHECK(g >= 0 && g < 8, "symmetry %d out of range [0,8)", g);
    PackedState s, o;
    memcpy(s.w, state, 32);
    sym_state(s, g, o);
    memcpy(out, o.w, 32);
    if (action_map81)
        for (int a = 0; a < 81; a++) action_map81[a] = sym_action(a, g);
    return 0;
}

// Debug rendering, same text as cpp/uttt_game.cpp:194-241.
int uttt_state_to_string(const uint32_t* state, char* buf, int cap, int* len_out) {
    PackedState s;
    memcpy(s.w, state, 32);
    const char* ox = is_first_player(s) ? "ox" : "xo";
    std::string out;
    for (int big_r = 0; big_r < 3; big_r++) {
        for (int sub_r = 0; sub_r < 3; sub_r++) {
            for (int big_c = 0; big_c < 3; big_c++) {
                int b = big_r * 3 + big_c;
                for (int sub_c = 0; sub_c < 3; sub_c++) {
                    int a = b * 9 + sub_r * 3 + sub_c;
                    out += stone_me(s, a) ? ox[0] : (stone_opp(s, a) ? ox[1] : '-');
                    out += ' ';
                }
                if (big_c < 2) out += "| ";
            }
            out += '\n';
        }
        if (big_r < 2) out += "---------------------\n";
    }
    out += "\nMain Board Status:\n";
    uint32_t M = main_me(s), E = main_opp(s);
    for (int b = 0; b < 9; b++) {
        bool m = (M >> b) & 1u, e = (E >> b) & 1u;
        out += (m && e) ? 'D' : (m ? ox[0] : (e ? ox[1] : '.'));
        if (b % 3 == 2) out += '\n';
    }
    out += "Next Player: ";
    out += ox[0];
    out += "\nActive Board: ";
    int act = active_board(s);
    out += (act < 0) ? std::string("Any") : std::to_string(act);
    out += '\n';
    if (len_out) *len_out = (int)out.size();
    if (buf && cap > 0) {
        int m = (int)out.size() < cap - 1 ? (int)out.size() : cap - 1;
        memcpy(buf, out.data(), (size_t)m);
        buf[m] = 0;
    }
    return 0;
}

// ---- device batch rules --------------------------------------------------------------------
int uttt_game_step(const uint32_t* states, const int32_t* actions, uint32_t* out, int64_t n, void* stream) {
    if (n <= 0) return 0;
    step_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>((const PackedState*)states, actions,
                                                                      (PackedState*)out, n);
    UTTT_CUDA_OK(cudaGetLastError());
    return 0;
}

int uttt_game_legal_mask(const uint32_t* states, uint32_t* masks, uint8_t* status, int64_t n, void* stream) {
    if (n <= 0) return 0;
    legal_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>((const PackedState*)states, (uint4*)masks,
                                                                       status, n);
    UTTT_CUDA_OK(cudaGetLastError());
    return 0;
}

int uttt_game_encode(const uint32_t* states, float* planes, int64_t n, void* stream) {
    if (n <= 0) return 0;
    if (((uintptr_t)planes & 15u) == 0)
        encode_kernel<<<ceil_div(n, PLANES_POS), PLANES_POS, 0, (cudaStream_t)stream>>>((const PackedState*)states,
                                                                                          planes, n);
    else
        encode_unaligned_kernel<<<ceil_div(n, 8), 256, 0, (cudaStream_t)stream>>>((const PackedState*)states, planes, n);
    UTTT_CUDA_OK(cudaGetLastError());
    return 0;
}

int uttt_game_gather_planes(const uint32_t* states, void* planes, int64_t n, void* stream) {
    if (n <= 0) return 0;
    if (((uintptr_t)planes & 15u) == 0)
        gather_planes_kernel<<<ceil_div(n, PLANES_POS), PLANES_POS, 0, (cudaStream_t)stream>>>(
            (const PackedState*)states, (__nv_bfloat16*)planes, n);
    else
        gather_planes_unaligned_kernel<<<ceil_div(n, 8), 256, 0, (cudaStream_t)stream>>>(
            (const PackedState*)states, (__nv_bfloat16*)planes, n);
    UTTT_CUDA_OK(cudaGetLastError());
    return 0;
}

int uttt_game_playout(uint32_t seed, uint64_t game0, int64_t n, uint64_t* digests, int32_t* plies,
                      int32_t* results, void* stream) {
    if (n <= 0) return 0;
    playout_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(seed, game0, n, digests, plies, results);
    UTTT_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
