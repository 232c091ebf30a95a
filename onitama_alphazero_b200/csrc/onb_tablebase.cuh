// onb_tablebase.cuh -- the index of the endgame tablebase (DESIGN.md §5g) and its lookup, shared by the solver (onb_tablebase.cu)
// and the searches that probe the table at their leaves (onb_mcts.cu, DESIGN.md §5i).
#pragma once
#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {

constexpr uint32_t kTbPairs = 600;      // ordered king pairs on distinct squares

// C(n, k) for n <= 24, k <= 4 at [5 n + k]
struct BinomTable {
    uint32_t b[25 * 5];
};
constexpr BinomTable make_binom() {
    BinomTable t{};
    for (int n = 0; n < 25; ++n)
        for (int k = 0; k < 5; ++k) {
            uint64_t v = 1;
            for (int i = 0; i < k && i < n; ++i) v = v * (uint64_t)(n - i) / (uint64_t)(i + 1);
            t.b[n * 5 + k] = k > n ? 0u : (uint32_t)v;
        }
    return t;
}
constexpr BinomTable kBinomHost = make_binom();
static __device__ BinomTable g_binom = make_binom();

__host__ __device__ __forceinline__ uint32_t low_bit(uint32_t x) {
#ifdef __CUDA_ARCH__
    return (uint32_t)(__ffs(x) - 1);
#else
    return (uint32_t)__builtin_ctz(x);
#endif
}
__host__ __device__ __forceinline__ uint32_t below(uint32_t s) { return (1u << s) - 1u; }

// colex rank of the squares of `set` among the squares not in `occ` (a square's position there is s - popc(occ below s))
__host__ __device__ __forceinline__ uint32_t colex_rank(const uint32_t* B, uint32_t set, uint32_t occ) {
    uint32_t r = 0, i = 1;
    while (set) {
        const uint32_t s = low_bit(set);
        set &= set - 1;
        r += B[(s - popc32(occ & below(s))) * 5 + i];
        ++i;
    }
    return r;
}

// card configuration 6 j + r of a neutral card and a red hand (ids) within the set `setmask`
__host__ __device__ __forceinline__ uint32_t card_cfg(uint32_t setmask, uint32_t neutral, uint32_t ra, uint32_t rb) {
    const uint32_t j = popc32(setmask & below(neutral));
    uint32_t a = popc32(setmask & below(ra)), b = popc32(setmask & below(rb));
    a -= a > j;
    b -= b > j;
    const uint32_t lo = a < b ? a : b, hi = a < b ? b : a;
    return 6u * j + lo + hi * (hi - 1u) / 2u;
}

__host__ __device__ __forceinline__ uint64_t class_subsets(const uint32_t* B, uint32_t p, uint32_t q) {
    return (uint64_t)B[23 * 5 + p] * B[(23 - p) * 5 + q];
}
// entry of a position within its class (p, q); pr, pb internal-layout pawn boards, kr, kb king squares
__host__ __device__ __forceinline__ uint64_t tb_entry(const uint32_t* B, uint32_t pr, uint32_t pb, uint32_t kr, uint32_t kb, uint32_t cfg,
                                                      uint32_t side, uint32_t p, uint32_t q) {
    const uint32_t kings = (1u << kr) | (1u << kb);
    const uint64_t sb = B[(23 - p) * 5 + q];
    const uint64_t pair = (uint64_t)(cfg * 2u + side) * kTbPairs + 24u * kr + kb - (kb > kr ? 1u : 0u);
    return pair * ((uint64_t)B[23 * 5 + p] * sb) + (uint64_t)colex_rank(B, pr, kings) * sb + colex_rank(B, pb, kings | pr);
}

// Kernel parameters of the solver (by value): the table (TbTable, onb_internal.h) and the card configurations of the set
struct TbParams : TbTable {
    uint8_t cards[30][4];   // hand cards of configuration cfg in slots red lo, red hi, blue lo, blue hi
    uint8_t child[30][4];   // configuration after the mover plays hand card u (it becomes the neutral card)
};

// value of a game, ONB_TB_NONE when it is decided or not a position of the table
__device__ __forceinline__ int32_t tb_lookup(const TbTable& P, const uint32_t* B, const Game& g) {
    if (g.result != 0 || current_state(g) != 0) return ONB_TB_NONE;
    uint32_t seen = 0;
    for (uint32_t s = 0; s < 5; ++s) seen |= 1u << card_at(g.cards, s);
    if (seen != P.setmask) return ONB_TB_NONE;
    if (popc32(g.king_r) != 1 || popc32(g.king_b) != 1 || (g.king_r & g.king_b) || (g.pawn_r & g.pawn_b) ||
        ((g.pawn_r | g.pawn_b) & (g.king_r | g.king_b)))
        return ONB_TB_NONE;
    const uint32_t p = popc32(g.pawn_r), q = popc32(g.pawn_b);
    if (p + q > P.max_pawns) return ONB_TB_NONE;
    const uint32_t cfg = card_cfg(P.setmask, card_at(g.cards, 4), card_at(g.cards, 0), card_at(g.cards, 1));
    return P.tab[5 * p + q][tb_entry(B, g.pawn_r, g.pawn_b, low_bit(g.king_r), low_bit(g.king_b), cfg, g.side, p, q)];
}

}  // namespace onb
