// uttt_rules.cuh -- bitboard Ultimate Tic-Tac-Toe rules (host + device inline).
//
// Replaces the reference's UTTT::State (cpp/uttt_game.h:48-54, 181 ints = 724 B) with a
// 32-byte packed, mover-relative position that is loaded/stored as two 128-bit vectors:
//   w0..w2  mover's stones,   3 sub-boards per word, 9 bits per sub-board (bit = cell 3*row+col)
//   w3..w5  opponent's stones, same layout
//   w6      main_board_pieces | main_board_enemy_pieces<<9 | (active_board+1)<<18
//   w7      reserved (0)
// The 81-bit legal-move mask uses the same 3x27 layout, so action id = 27*word + bit = 9*board + cell
// and "ascending action id" (cpp/uttt_game.cpp:181-188, Q-G4) is ascending bit order.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define UTTT_HD __host__ __device__ __forceinline__
#else
#define UTTT_HD inline
#endif

namespace uttt {

struct alignas(16) PackedState {
    uint32_t w[8];
};

enum : uint32_t { STATUS_ONGOING = 0, STATUS_LOSE = 1, STATUS_DRAW = 2 };

UTTT_HD int popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// cpp/uttt_game.cpp:35-61 -- any of the 8 lines fully occupied in a 9-bit mask.
// Branch-free form of the 512-entry win table (rows, columns, two diagonals).
UTTT_HD bool win9(uint32_t m) {
    uint32_t rows = m & (m >> 1) & (m >> 2) & 0x049u;
    uint32_t cols = m & (m >> 3) & (m >> 6) & 0x007u;
    uint32_t diag = m & (m >> 4) & (m >> 8) & 0x001u;
    uint32_t anti = (m >> 2) & (m >> 4) & (m >> 6) & 0x001u;
    return (rows | cols | diag | anti) != 0u;
}

UTTT_HD uint32_t main_me(const PackedState& s) { return s.w[6] & 0x1FFu; }
UTTT_HD uint32_t main_opp(const PackedState& s) { return (s.w[6] >> 9) & 0x1FFu; }
UTTT_HD int active_board(const PackedState& s) { return (int)((s.w[6] >> 18) & 15u) - 1; }

UTTT_HD void init_state(PackedState& s) {
#pragma unroll
    for (int i = 0; i < 8; i++) s.w[i] = 0u;
}

// cpp/uttt_game.cpp:77-79
UTTT_HD bool is_lose(const PackedState& s) { return win9(main_opp(s)); }

// cpp/uttt_game.cpp:92-94
UTTT_HD bool is_first_player(const PackedState& s) {
    return popc32(s.w[0]) + popc32(s.w[1]) + popc32(s.w[2]) ==
           popc32(s.w[3]) + popc32(s.w[4]) + popc32(s.w[5]);
}

// spread the 3 candidate-board bits of one word into three 9-bit groups
UTTT_HD uint32_t spread3(uint32_t c3) {
    return ((c3 & 1u) ? 0x1FFu : 0u) | ((c3 & 2u) ? (0x1FFu << 9) : 0u) | ((c3 & 4u) ? (0x1FFu << 18) : 0u);
}

// cpp/uttt_game.cpp:148-191 -> 81-bit mask (3 x 27 bits). Returns the number of legal moves.
UTTT_HD int legal_mask(const PackedState& s, uint32_t lm[3]) {
    uint32_t M = main_me(s), E = main_opp(s);
    int act = active_board(s);
    uint32_t open = ~(M | E) & 0x1FFu;
    uint32_t cand = (act >= 0 && ((open >> act) & 1u)) ? (1u << act) : open;   // :158-178 (incl. Q-G3)
    if (win9(E)) cand = 0u;                                                    // :151-153
    int n = 0;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        uint32_t empty = ~(s.w[j] | s.w[3 + j]) & 0x7FFFFFFu;
        lm[j] = empty & spread3((cand >> (3 * j)) & 7u);
        n += popc32(lm[j]);
    }
    return n;
}

// cpp/uttt_game.cpp:77-89
UTTT_HD uint32_t status_of(const PackedState& s, int n_legal) {
    return is_lose(s) ? STATUS_LOSE : (n_legal == 0 ? STATUS_DRAW : STATUS_ONGOING);
}

// cpp/uttt_game.cpp:97-145 (no legality check, Q-G5). action in [0,81).
UTTT_HD void next_state(const PackedState& s, int action, PackedState& o) {
    int b = action / 9, c = action - 9 * b;
    int j = b / 3, sh = 9 * (b - 3 * j);
    uint32_t me0 = s.w[3], me1 = s.w[4], me2 = s.w[5];      // sides swap
    uint32_t op0 = s.w[0], op1 = s.w[1], op2 = s.w[2];
    uint32_t bit = 1u << (sh + c);
    op0 |= (j == 0) ? bit : 0u;
    op1 |= (j == 1) ? bit : 0u;
    op2 |= (j == 2) ? bit : 0u;
    uint32_t opw = (j == 0) ? op0 : (j == 1 ? op1 : op2);
    uint32_t mew = (j == 0) ? me0 : (j == 1 ? me1 : me2);
    uint32_t sub_op = (opw >> sh) & 0x1FFu;
    uint32_t sub_me = (mew >> sh) & 0x1FFu;
    uint32_t M = main_opp(s), E = main_me(s);
    if (win9(sub_op)) {
        E |= 1u << b;
    } else if ((sub_op | sub_me) == 0x1FFu) {              // drawn sub-board marks both (Q-G1)
        M |= 1u << b;
        E |= 1u << b;
    }
    uint32_t act1 = (((M | E) >> c) & 1u) ? 0u : (uint32_t)(c + 1);
    o.w[0] = me0; o.w[1] = me1; o.w[2] = me2;
    o.w[3] = op0; o.w[4] = op1; o.w[5] = op2;
    o.w[6] = M | (E << 9) | (act1 << 18);
    o.w[7] = 0u;
}

// rank-th (0-based) set bit of the 81-bit mask -> action id
UTTT_HD int nth_legal(const uint32_t lm[3], int rank) {
    int base = 0;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        int c = popc32(lm[j]);
        if (rank < c) {
            uint32_t m = lm[j];
            for (int k = 0; k < rank; k++) m &= m - 1u;
#if defined(__CUDA_ARCH__)
            return base + (__ffs((int)m) - 1);
#else
            return base + __builtin_ctz(m);
#endif
        }
        rank -= c;
        base += 27;
    }
    return -1;
}

UTTT_HD bool legal_bit(const uint32_t lm[3], int a) {
    int j = a / 27;
    uint32_t w = (j == 0) ? lm[0] : (j == 1 ? lm[1] : lm[2]);
    return (w >> (a - 27 * j)) & 1u;
}

// number of legal actions with id < a
UTTT_HD int legal_rank(const uint32_t lm[3], int a) {
    int j = a / 27, bit = a - 27 * j;
    int r = 0;
    if (j > 0) r += popc32(lm[0]);
    if (j > 1) r += popc32(lm[1]);
    uint32_t w = (j == 0) ? lm[0] : (j == 1 ? lm[1] : lm[2]);
    return r + popc32(w & ((1u << bit) - 1u));
}

// 9 cells of picture row R (bit C = column C) taken from three words holding 3 sub-boards x 9 cells each
// (the mover / opponent / legal-mask words): sub-board row R/3, cell row R%3 of its three sub-boards.
UTTT_HD uint32_t picture_row(const uint32_t x[3], int R) {
    int br = R / 3, sr = R - 3 * br;
    uint32_t w = (br == 0) ? x[0] : (br == 1 ? x[1] : x[2]);
    w >>= 3 * sr;
    return (w & 7u) | (((w >> 9) & 7u) << 3) | (((w >> 18) & 7u) << 6);
}

// cell (R,C) of the 9x9 picture <-> (board, cell): cpp/uttt_game.cpp:256-257
UTTT_HD int action_of_rc(int R, int C) { return ((R / 3) * 3 + (C / 3)) * 9 + (R % 3) * 3 + (C % 3); }

UTTT_HD bool stone_me(const PackedState& s, int a) {
    int j = a / 27;
    return (s.w[j] >> (a - 27 * j)) & 1u;
}
UTTT_HD bool stone_opp(const PackedState& s, int a) {
    int j = a / 27;
    return (s.w[3 + j] >> (a - 27 * j)) & 1u;
}

// ---- counter-based RNG: Philox4x32-10 (Salmon et al. 2011) ----
struct Philox4 {
    uint32_t x, y, z, w;
};
UTTT_HD Philox4 philox4x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox4 o = {c0, c1, c2, c3};
    return o;
}

UTTT_HD uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x85EBCA6Bu;
    x ^= x >> 13; x *= 0xC2B2AE35u;
    x ^= x >> 16;
    return x;
}

// Integer hash of a position (cells, main flags, active board): the key of the
// deterministic "oracle evaluator" used for search parity tests.
UTTT_HD uint32_t state_hash(const PackedState& s) {
    uint32_t h = 0x811C9DC5u;
    for (int a = 0; a < 81; a++) {
        uint32_t v = stone_me(s, a) ? 1u : (stone_opp(s, a) ? 2u : 0u);
        h = (h ^ v) * 0x01000193u;
    }
    uint32_t M = main_me(s), E = main_opp(s);
    for (int b = 0; b < 9; b++) {
        uint32_t v = ((M >> b) & 1u) | (((E >> b) & 1u) << 1);
        h = (h ^ v) * 0x01000193u;
    }
    h = (h ^ ((s.w[6] >> 18) & 15u)) * 0x01000193u;
    return h;
}

UTTT_HD uint64_t fnv64(uint64_t h, uint32_t x) { return (h ^ (uint64_t)x) * 0x100000001B3ull; }

// ---- board symmetries (include/uttt_b200.h, UTTT_SP_RANDOM_SYMMETRY) ----
// Symmetry g = 4f + r of the 9x9 picture (R, C): transpose if f, then numpy.rot90(picture, k=r).  It maps sub-board
// (R/3, C/3) and cell (R%3, C%3) by the same map of the 3x3 grid, so it acts on a 9-bit mask (bit 3y+x) of boards or
// cells.  On that grid rot90 is (y,x) -> (2-x,y) = transpose, then flip rows; every g is therefore "transpose, then
// flip rows (y -> 2-y), then flip columns (x -> 2-x)", each step present or not -- bits 0, 1, 2 of nibble g of
// SYM_STEPS:  g0 -, g1 T V, g2 V H, g3 T H, g4 T, g5 V, g6 T V H, g7 H.
constexpr uint32_t SYM_STEPS = 0x47215630u;

UTTT_HD uint32_t sym9(uint32_t m, int g) {
    const uint32_t steps = (SYM_STEPS >> (4 * g)) & 7u;
    if (steps & 1u) m = (m & 0x111u) | ((m & 0x022u) << 2) | ((m & 0x088u) >> 2) | ((m & 0x004u) << 4) | ((m & 0x040u) >> 4);
    if (steps & 2u) m = ((m & 0x007u) << 6) | (m & 0x038u) | ((m >> 6) & 0x007u);
    if (steps & 4u) m = ((m & 0x049u) << 2) | (m & 0x092u) | ((m >> 2) & 0x049u);
    return m;
}

// image of index i (0..8) of the 3x3 grid
UTTT_HD int sym_index(int i, int g) {
#if defined(__CUDA_ARCH__)
    return __ffs((int)sym9(1u << i, g)) - 1;
#else
    return __builtin_ctz(sym9(1u << i, g));
#endif
}

// sigma_g(a): the action at the image of action a's cell
UTTT_HD int sym_action(int a, int g) {
    const int b = a / 9;
    return 9 * sym_index(b, g) + sym_index(a - 9 * b, g);
}

// the image of a position: stones, main-board flags and the forced board moved by the map (-1 stays -1)
UTTT_HD void sym_state(const PackedState& s, int g, PackedState& o) {
#pragma unroll
    for (int i = 0; i < 8; i++) o.w[i] = 0u;
#pragma unroll
    for (int b = 0; b < 9; b++) {
        const int nb = sym_index(b, g), j = b / 3, sh = 9 * (b - 3 * j), nj = nb / 3, nsh = 9 * (nb - 3 * nj);
        const uint32_t me = sym9((s.w[j] >> sh) & 0x1FFu, g), op = sym9((s.w[3 + j] >> sh) & 0x1FFu, g);
        o.w[0] |= (nj == 0) ? me << nsh : 0u; o.w[1] |= (nj == 1) ? me << nsh : 0u; o.w[2] |= (nj == 2) ? me << nsh : 0u;
        o.w[3] |= (nj == 0) ? op << nsh : 0u; o.w[4] |= (nj == 1) ? op << nsh : 0u; o.w[5] |= (nj == 2) ? op << nsh : 0u;
    }
    const int act = active_board(s);
    o.w[6] = sym9(main_me(s), g) | (sym9(main_opp(s), g) << 9) | ((uint32_t)(act < 0 ? 0 : sym_index(act, g) + 1) << 18);
}

// the symmetry a leaf is evaluated under: Philox key (seed, 2), counter (game, ply, j = evaluation of the move's search)
UTTT_HD int sym_draw(uint32_t seed, uint64_t game, uint32_t ply, uint32_t j) {
    return (int)(philox4x32(seed, 2u, (uint32_t)game, (uint32_t)(game >> 32), ply, j).x >> 29);
}

}  // namespace uttt
