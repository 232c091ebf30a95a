// onb_rules.cuh -- Onitama rules for the GPU: bit layout, the 16-card attack table, packed game state,
// move generation, move application, terminal detection, the counter RNG.
//
// Internal bit layout: square n (row-major, n = row*5 + col, (0,0) = a5) is bit n of a 25-bit word.
// The reference layout (onitama-game/src/common/mod.rs:2-4: square n = bit 31-n) is exactly
// __brev() of this one, so the conversion at the ABI is a single instruction.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace onb {

constexpr uint32_t kAll25 = 0x01FFFFFFu;
constexpr int kRed = 0, kBlue = 1;

// ---------------------------------------------------------------------------------------------
// Card table. Each card is the list of (d_row, d_col) steps for Red (Red moves towards row 0);
// Blue uses the 180-degree rotation. Restates the patterns of onitama-game/src/game/card.rs:17-463
// (checked against the reference's hex masks by tests/test_abi_cpu.py via onb_attack_maps()).
// ---------------------------------------------------------------------------------------------
struct CardDef {
    int n;
    int dr[4];
    int dc[4];
};
constexpr CardDef kCards[16] = {
    {2, {-2, 1, 0, 0}, {0, 0, 0, 0}},      //  0 Tiger
    {4, {-1, -1, 1, 1}, {-2, 2, -1, 1}},   //  1 Dragon
    {3, {-1, 0, 1, 0}, {-1, -2, 1, 0}},    //  2 Frog
    {3, {-1, 0, 1, 0}, {1, 2, -1, 0}},     //  3 Rabbit
    {3, {-1, 0, 0, 0}, {0, -2, 2, 0}},     //  4 Crab
    {4, {-1, -1, 0, 0}, {-1, 1, -1, 1}},   //  5 Elephant
    {4, {-1, 0, 0, 1}, {-1, -1, 1, 1}},    //  6 Goose
    {4, {-1, 0, 0, 1}, {1, -1, 1, -1}},    //  7 Rooster
    {4, {-1, -1, 1, 1}, {-1, 1, -1, 1}},   //  8 Monkey
    {3, {-1, -1, 1, 0}, {-1, 1, 0, 0}},    //  9 Mantis
    {3, {-1, 1, 1, 0}, {0, -1, 1, 0}},     // 10 Crane
    {3, {-1, 0, 1, 0}, {0, -1, 0, 0}},     // 11 Horse
    {3, {-1, 0, 1, 0}, {0, 1, 0, 0}},      // 12 Ox
    {3, {-1, 0, 0, 0}, {0, -1, 1, 0}},     // 13 Boar
    {3, {-1, 0, 1, 0}, {-1, 1, -1, 0}},    // 14 Eel
    {3, {-1, 0, 1, 0}, {1, -1, 1, 0}},     // 15 Cobra
};
// bit i set = card i carries the Blue stamp (card.rs player_color fields); the neutral card's stamp
// decides the first mover (game_state.rs:34-41).
constexpr uint32_t kBlueStampMask = 0x5551u;

struct alignas(16) AttackTable {
    uint32_t t[2 * 16 * 25];  // [colour][card][from] -> to-mask (internal layout)
};
constexpr AttackTable make_attack_table() {
    AttackTable a{};
    for (int color = 0; color < 2; ++color)
        for (int card = 0; card < 16; ++card)
            for (int from = 0; from < 25; ++from) {
                uint32_t m = 0;
                const int r = from / 5, c = from % 5;
                for (int j = 0; j < kCards[card].n; ++j) {
                    const int dr = color == kRed ? kCards[card].dr[j] : -kCards[card].dr[j];
                    const int dc = color == kRed ? kCards[card].dc[j] : -kCards[card].dc[j];
                    const int rr = r + dr, cc = c + dc;
                    if (rr >= 0 && rr < 5 && cc >= 0 && cc < 5) m |= 1u << (rr * 5 + cc);
                }
                a.t[(color * 16 + card) * 25 + from] = m;
            }
    return a;
}
constexpr AttackTable kAttackHost = make_attack_table();
// The 16-card move table (3 200 B) lives in device memory and is staged into shared memory once per CTA
// (load_attack_table_to_smem): lanes index it divergently (one `from` square per lane), which would serialise in the
// constant cache, whereas the staging copy reads consecutive words (coalesced, L1/L2 resident).
static __device__ AttackTable g_attack = make_attack_table();

__device__ __forceinline__ void load_attack_table_to_smem(uint32_t* s_att) {
    const uint4* src = reinterpret_cast<const uint4*>(g_attack.t);
    uint4* dst = reinterpret_cast<uint4*>(s_att);
    for (int i = threadIdx.x; i < 200; i += blockDim.x) dst[i] = src[i];
}

// ---------------------------------------------------------------------------------------------
// Packed game: 16 bytes, one 128-bit load/store per game (structure-of-arrays: one uint4 array).
//   x = pawns[Red]  | card[0] << 25 | (card[4] & 7) << 29
//   y = pawns[Blue] | card[1] << 25 | (card[4] >> 3) << 29 | side << 30 | passed << 31
//   z = kings[Red]  | card[2] << 25 | result << 29
//   w = kings[Blue] | card[3] << 25
// Four separate bitboards are kept (rather than pieces + king index) because make_move performs no
// legality check (state.rs:144) and the Random agent can fabricate pieces (ai/random.rs:26-34).
// ---------------------------------------------------------------------------------------------
struct Game {
    uint32_t pawn_r, pawn_b, king_r, king_b;
    uint32_t cards;   // 5 nibbles, slot k at bits 4k..4k+3
    uint32_t side;    // side to move
    uint32_t result;  // 0 in progress, 1 Red won, 2 Blue won
    uint32_t passed;  // sticky: a pass happened since reset
};

__host__ __device__ __forceinline__ Game unpack(const uint4 v) {
    Game g;
    g.pawn_r = v.x & kAll25; g.pawn_b = v.y & kAll25; g.king_r = v.z & kAll25; g.king_b = v.w & kAll25;
    g.cards = ((v.x >> 25) & 15u) | (((v.y >> 25) & 15u) << 4) | (((v.z >> 25) & 15u) << 8) | (((v.w >> 25) & 15u) << 12) |
              ((((v.x >> 29) & 7u) | (((v.y >> 29) & 1u) << 3)) << 16);
    g.side = (v.y >> 30) & 1u;
    g.passed = v.y >> 31;
    g.result = (v.z >> 29) & 3u;
    return g;
}
__host__ __device__ __forceinline__ uint4 pack(const Game& g) {
    uint4 v;
    const uint32_t c4 = (g.cards >> 16) & 15u;
    v.x = g.pawn_r | ((g.cards & 15u) << 25) | ((c4 & 7u) << 29);
    v.y = g.pawn_b | (((g.cards >> 4) & 15u) << 25) | ((c4 >> 3) << 29) | (g.side << 30) | (g.passed << 31);
    v.z = g.king_r | (((g.cards >> 8) & 15u) << 25) | (g.result << 29);
    v.w = g.king_b | (((g.cards >> 12) & 15u) << 25);
    return v;
}
__host__ __device__ __forceinline__ uint32_t card_at(uint32_t cards, uint32_t slot) { return (cards >> (4u * slot)) & 15u; }
// Deck::rotate (deck.rs:87-90): swap hand slot `idx` with the neutral slot 4.
__host__ __device__ __forceinline__ uint32_t rotate_cards(uint32_t cards, uint32_t idx) {
    const uint32_t sh = 4u * idx;
    const uint32_t d = ((cards >> sh) ^ (cards >> 16)) & 15u;  // xor-swap of the two nibbles
    return cards ^ (d << sh) ^ (d << 16);
}

// start position (state.rs:24-45) in the internal layout
constexpr uint32_t kRedKingStart = 1u << 22, kBlueKingStart = 1u << 2;
constexpr uint32_t kRedPawnsStart = (1u << 20) | (1u << 21) | (1u << 23) | (1u << 24);
constexpr uint32_t kBluePawnsStart = (1u << 0) | (1u << 1) | (1u << 3) | (1u << 4);
constexpr uint32_t kBlueTemple = 2, kRedTemple = 22;

__host__ __device__ __forceinline__ Game start_game(uint32_t cards) {
    Game g;
    g.pawn_r = kRedPawnsStart; g.pawn_b = kBluePawnsStart; g.king_r = kRedKingStart; g.king_b = kBlueKingStart;
    g.cards = cards;
    g.side = (kBlueStampMask >> ((cards >> 16) & 15u)) & 1u;
    g.result = 0; g.passed = 0;
    return g;
}

// ---------------------------------------------------------------------------------------------
// Counter RNG shared with the oracle (restated there independently): splitmix64 finaliser keyed by
// (seed, global game id) then (step, draw). Index = mulhi32(r, n).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return z;
}
__host__ __device__ __forceinline__ uint64_t game_key(uint64_t seed, uint64_t game) {
    return mix64(seed + 0x9E3779B97F4A7C15ull * (game + 1));
}
__host__ __device__ __forceinline__ uint32_t rand_from_key(uint64_t key, uint32_t step, uint32_t draw) {
    return (uint32_t)(mix64(key ^ (((uint64_t)step << 32) | draw)) >> 32);
}
__host__ __device__ __forceinline__ uint32_t rand_index(uint32_t r, uint32_t n) {
#ifdef __CUDA_ARCH__
    return __umulhi(r, n);
#else
    return (uint32_t)(((uint64_t)r * n) >> 32);
#endif
}
enum : uint32_t { kDrawMove = 0, kDrawPass = 1, kDrawAgentSlot = 2, kDrawAgentMove = 3, kDrawDeal = 8 };

// first 5 of a Fisher-Yates shuffle of the 16 card ids, as 5 nibbles
__host__ __device__ __forceinline__ uint32_t deal_cards(uint64_t key, uint32_t epoch) {
    uint64_t ids = 0xFEDCBA9876543210ull;  // nibble i = i
    for (uint32_t i = 0; i < 5; ++i) {
        const uint32_t j = i + rand_index(rand_from_key(key, epoch, kDrawDeal + i), 16u - i);
        const uint64_t a = (ids >> (4 * i)) & 15ull, b = (ids >> (4 * j)) & 15ull;
        ids &= ~((15ull << (4 * i)) | (15ull << (4 * j)));
        ids |= (b << (4 * i)) | (a << (4 * j));
    }
    return (uint32_t)(ids & 0xFFFFFull);
}

// ---------------------------------------------------------------------------------------------
// Action code (include/onb.h): to | from<<5 | used_card_idx<<10 | piece<<12 | pass<<13
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t make_action(uint32_t card_idx, uint32_t from, uint32_t to, uint32_t king) {
    return to | (from << 5) | (card_idx << 10) | (king << 12);
}
constexpr uint32_t kPassBit = 1u << 13;

// ---------------------------------------------------------------------------------------------
// Move application. State::make_move (state.rs:145-202): no legality check; pawn capture is tested
// before king capture; a king stepping on the enemy temple wins (overrides Capture); the used card is
// swapped with the neutral one. Returns the game result code (0 = in progress).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t apply_move(Game& g, uint32_t action) {
    const uint32_t to = action & 31u, from = (action >> 5) & 31u, idx = (action >> 10) & 3u, king = (action >> 12) & 1u;
    const uint32_t side = g.side;
    uint32_t res = 0;
    if (action & kPassBit) {  // State::pass (state.rs:139-142)
        g.cards = rotate_cards(g.cards, idx);
        g.passed = 1;
    } else {
        const uint32_t fb = 1u << from, tb = 1u << to;
        uint32_t own_p = side ? g.pawn_b : g.pawn_r, own_k = side ? g.king_b : g.king_r;
        uint32_t en_p = side ? g.pawn_r : g.pawn_b, en_k = side ? g.king_r : g.king_b;
        if (king) own_k &= ~fb; else own_p &= ~fb;
        if (en_p & tb) en_p &= ~tb;
        else if (en_k & tb) { en_k &= ~tb; res = 1u + side; }
        if (king) own_k |= tb; else own_p |= tb;
        if (king && to == (side ? kRedTemple : kBlueTemple)) res = 1u + side;
        g.pawn_r = side ? en_p : own_p; g.pawn_b = side ? own_p : en_p;
        g.king_r = side ? en_k : own_k; g.king_b = side ? own_k : en_k;
        g.cards = rotate_cards(g.cards, idx);
    }
    g.side = side ^ 1u;
    g.result = res;
    return res;
}

// The same transition on a mover-relative view (own / enemy boards instead of Red / Blue), used by the search descent where
// the per-ply colour selects of apply_move would dominate: after the move the roles are swapped, so the view is again
// relative to the side to move.
struct RelGame {
    uint32_t op, ok, ep, ek;  // own pawns, own king, enemy pawns, enemy king (of the side to move)
    uint32_t cards, side;
};
__host__ __device__ __forceinline__ RelGame to_rel(const Game& g) {
    RelGame r;
    r.op = g.side ? g.pawn_b : g.pawn_r; r.ok = g.side ? g.king_b : g.king_r;
    r.ep = g.side ? g.pawn_r : g.pawn_b; r.ek = g.side ? g.king_r : g.king_b;
    r.cards = g.cards; r.side = g.side;
    return r;
}
__host__ __device__ __forceinline__ Game from_rel(const RelGame& r) {
    Game g;
    g.pawn_r = r.side ? r.ep : r.op; g.king_r = r.side ? r.ek : r.ok;
    g.pawn_b = r.side ? r.op : r.ep; g.king_b = r.side ? r.ok : r.ek;
    g.cards = r.cards; g.side = r.side; g.result = 0; g.passed = 0;
    return g;
}
__host__ __device__ __forceinline__ uint32_t apply_move_rel(RelGame& g, uint32_t action) {
    const uint32_t to = action & 31u, from = (action >> 5) & 31u, idx = (action >> 10) & 3u, king = (action >> 12) & 1u;
    uint32_t res = 0;
    if (!(action & kPassBit)) {
        const uint32_t fb = 1u << from, tb = 1u << to;
        const uint32_t km = 0u - king;  // all ones if the mover is the king
        g.ok = (g.ok & ~(fb & km)) | (tb & km);
        g.op = (g.op & ~(fb & ~km)) | (tb & ~km);
        const uint32_t hit_p = g.ep & tb;
        g.ep &= ~tb;
        const uint32_t hit_k = hit_p ? 0u : (g.ek & tb);
        g.ek &= ~hit_k;
        if (hit_k || (king && to == (g.side ? kRedTemple : kBlueTemple))) res = 1u + g.side;
    }
    g.cards = rotate_cards(g.cards, idx);
    uint32_t t = g.op; g.op = g.ep; g.ep = t;
    t = g.ok; g.ok = g.ek; g.ek = t;
    g.side ^= 1u;
    return res;
}

// State::current_state (state.rs:120-134): 0 in progress, 1 RedWin, 2 BlueWin (BlueWin tested first).
__host__ __device__ __forceinline__ uint32_t current_state(const Game& g) {
    if (g.king_r == 0 || g.king_b == kRedKingStart) return 2;
    if (g.king_b == 0 || g.king_r == kBlueKingStart) return 1;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Leaf evaluation of the alpha-beta agent (project-defined, DESIGN.md §5d; restated square by square in
// tests/alphabeta_oracle.cpp). E = V(mover) - V(opponent), for one side
//   V = sum over pawns (100 + 4 adv(q) + 2 ctr(q)) + sum over kings 6 (6 - manhattan(king, enemy temple)),
// q = 5 row + col, adv = 4 - row for Red and row for Blue, ctr = 2 - |col - 2|, enemy temple = 2 for Red, 22 for Blue.
// The per-square sums are taken with popcounts over row / column masks: sum(row) = #(row >= 1) + ... + #(row >= 4),
// sum(ctr) = #(col in 1..3) + #(col == 2); the king term is 6 (4 - row + ctr) for Red and 6 (row + ctr) for Blue.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t popc32(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __popc(x);
#else
    return (uint32_t)__builtin_popcount(x);
#endif
}
constexpr uint32_t each_row(uint32_t pattern5) { return pattern5 * 0x108421u; }  // the 5-bit row pattern repeated on all five rows
constexpr uint32_t kRowGe1 = kAll25 & ~0x1Fu, kRowGe2 = kAll25 & ~0x3FFu, kRowGe3 = kAll25 & ~0x7FFFu, kRowGe4 = kAll25 & ~0xFFFFFu;
constexpr uint32_t kColMid3 = each_row(0x0Eu), kCol2 = each_row(0x04u);
constexpr int32_t kAlphaBetaWin = 1000000;
__host__ __device__ __forceinline__ int32_t sum_rows(uint32_t b) {
    return (int32_t)(popc32(b & kRowGe1) + popc32(b & kRowGe2) + popc32(b & kRowGe3) + popc32(b & kRowGe4));
}
__host__ __device__ __forceinline__ int32_t sum_ctr(uint32_t b) { return (int32_t)(popc32(b & kColMid3) + popc32(b & kCol2)); }
__host__ __device__ __forceinline__ int32_t side_value(uint32_t pawns, uint32_t kings, uint32_t color) {
    const int32_t np = (int32_t)popc32(pawns), nk = (int32_t)popc32(kings);
    if (color == kRed) return 116 * np - 4 * sum_rows(pawns) + 2 * sum_ctr(pawns) + 24 * nk - 6 * sum_rows(kings) + 6 * sum_ctr(kings);
    return 100 * np + 4 * sum_rows(pawns) + 2 * sum_ctr(pawns) + 6 * sum_rows(kings) + 6 * sum_ctr(kings);
}
__host__ __device__ __forceinline__ int32_t eval_position(const RelGame& g) {
    return side_value(g.op, g.ok, g.side) - side_value(g.ep, g.ek, g.side ^ 1u);
}

// ---------------------------------------------------------------------------------------------
// Move generation for one thread (State::generate_all_legal_moves, state.rs:301-378).
// Enumeration order: hand slot ascending, from ascending, to ascending. A piece is a Pawn if the pawn
// bit is set, else a King (state.rs:345-358). T points at the 800-word attack table (shared memory).
// ---------------------------------------------------------------------------------------------
struct MoveSummary {
    uint32_t n0, n1;  // number of moves of own hand slot 0 / 1
    uint32_t m0, m1;  // union of destination squares per slot (policy-shaped legal mask, internal layout)
};
__device__ __forceinline__ MoveSummary summarize_moves(const uint32_t* T, const Game& g, uint32_t side) {
    const uint32_t own_p = side ? g.pawn_b : g.pawn_r, own_k = side ? g.king_b : g.king_r;
    const uint32_t own = own_p | own_k;
    const uint32_t base = side * 2u;
    const uint32_t* T0 = T + (side * 16u + card_at(g.cards, base)) * 25u;
    const uint32_t* T1 = T + (side * 16u + card_at(g.cards, base + 1u)) * 25u;
    MoveSummary s{0, 0, 0, 0};
    uint32_t rem = own;
    while (rem) {
        const int f = __ffs(rem) - 1;
        rem &= rem - 1;
        const uint32_t a0 = T0[f] & ~own, a1 = T1[f] & ~own;
        s.n0 += __popc(a0); s.n1 += __popc(a1);
        s.m0 |= a0; s.m1 |= a1;
    }
    return s;
}
// r-th move (0-based, r < count) of hand slot `slot01` in reference order -> action code
__device__ __forceinline__ uint32_t nth_move_of_slot(const uint32_t* T, const Game& g, uint32_t side, uint32_t slot01, uint32_t r) {
    const uint32_t own_p = side ? g.pawn_b : g.pawn_r, own_k = side ? g.king_b : g.king_r;
    const uint32_t own = own_p | own_k;
    const uint32_t idx = side * 2u + slot01;
    const uint32_t* Ts = T + (side * 16u + card_at(g.cards, idx)) * 25u;
    uint32_t rem = own;
    while (rem) {
        const int f = __ffs(rem) - 1;
        rem &= rem - 1;
        uint32_t a = Ts[f] & ~own;
        const uint32_t c = __popc(a);
        if (r < c) {
            for (; r; --r) a &= a - 1;
            const uint32_t to = __ffs(a) - 1;
            return make_action(idx, (uint32_t)f, to, ((own_p >> f) & 1u) ^ 1u);
        }
        r -= c;
    }
    return 0xFFFFu;  // unreachable when r < count
}

// 21 plane words of create_tensor_from_state (alphazero-training/src/common.rs:26-80), internal layout:
// 0 red pawns, 1 red king, 2 blue pawns, 3 blue king, 4+card for the mover's two cards, 20 = Blue to move.
__device__ __forceinline__ uint32_t plane_word(const Game& g, uint32_t side, uint32_t p) {
    if (p == 0) return g.pawn_r;
    if (p == 1) return g.king_r;
    if (p == 2) return g.pawn_b;
    if (p == 3) return g.king_b;
    if (p == 20) return side ? kAll25 : 0u;
    const uint32_t c0 = card_at(g.cards, side * 2u), c1 = card_at(g.cards, side * 2u + 1u);
    return (p - 4u == c0 || p - 4u == c1) ? kAll25 : 0u;
}

}  // namespace onb
