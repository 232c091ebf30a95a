// onb_tablebase.cu -- endgame tablebases (DESIGN.md §5g): exact win / loss / draw and distance to win for every position of one
// five-card set with at most max_pawns pawns, solved on the GPU, plus the probe and best-move kernels.
//
// Classes (p red pawns, q blue pawns) are solved in ascending p + q: a capture leads to a class of lower material, whose values are
// final. Within a class the solve is a layered forward iteration over a work list of the unresolved entries. Iteration k reads
// only values of magnitude below k, so the table does not depend on the order in which threads resolve entries. A win in n has n
// odd and a loss in n has n even, so an odd iteration only looks for a child that holds -(k-1) and an even one only for a position
// whose every child is a win. During the solve 0 means "unresolved"; the entries still unresolved at the end are the draws.
#include <cstring>

#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {

constexpr int kTbThreads = 256;
constexpr uint32_t kTbPairs = 600;      // ordered king pairs on distinct squares
constexpr uint32_t kTbDecided = 47;     // of them with the red king on square 2 or the blue king on square 22

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
// the k squares outside `occ` whose colex rank is r
__host__ __device__ __forceinline__ uint32_t colex_unrank(const uint32_t* B, uint32_t r, uint32_t k, uint32_t occ) {
    uint32_t set = 0;
    for (uint32_t i = k; i >= 1; --i) {
        uint32_t c = i - 1;
        while (c < 23 && B[(c + 1) * 5 + i] <= r) ++c;
        r -= B[c * 5 + i];
        uint32_t f = kAll25 & ~occ;
        for (uint32_t t = 0; t < c; ++t) f &= f - 1;
        set |= 1u << low_bit(f);
    }
    return set;
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
struct TbPos {
    uint32_t pr, pb, kr, kb, cfg, side;
};
// (every class of at most four pawns has fewer than 2^32 entries)
__host__ __device__ __forceinline__ TbPos tb_unrank(const uint32_t* B, uint32_t e, uint32_t p, uint32_t q) {
    const uint32_t sb = B[(23 - p) * 5 + q];
    const uint32_t s = B[23 * 5 + p] * sb;
    const uint32_t sub = e % s;
    const uint32_t rest = e / s;
    TbPos x;
    const uint32_t kp = rest % kTbPairs, cs = rest / kTbPairs;
    x.side = cs & 1u;
    x.cfg = cs >> 1;
    x.kr = kp / 24u;
    const uint32_t t = kp % 24u;
    x.kb = t + (t >= x.kr ? 1u : 0u);
    const uint32_t kings = (1u << x.kr) | (1u << x.kb);
    x.pr = colex_unrank(B, sub / sb, p, kings);
    x.pb = colex_unrank(B, sub % sb, q, kings | x.pr);
    return x;
}

// Kernel parameters (by value): the class tables and the card configurations of the set
struct TbParams {
    int16_t* tab[25];       // class 5 p + q; nullptr: not in the table
    uint32_t setmask, max_pawns;
    uint8_t cards[30][4];   // hand cards of configuration cfg in slots red lo, red hi, blue lo, blue hi
    uint8_t child[30][4];   // configuration after the mover plays hand card u (it becomes the neutral card)
};

__device__ __forceinline__ void tb_load_smem(uint32_t* s_att, uint32_t* s_b) {
    load_attack_table_to_smem(s_att);
    for (int i = threadIdx.x; i < 125; i += blockDim.x) s_b[i] = g_binom.b[i];
}

// appends the flagged entries of a warp to out (order within the list is irrelevant: each entry is examined by one thread)
__device__ __forceinline__ void warp_append(bool keep, uint32_t e, uint32_t* out, unsigned long long* cnt) {
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, keep);
    if (!bal) return;
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long base = 0;
    if (lane == (uint32_t)(__ffs(bal) - 1)) base = atomicAdd(cnt, (unsigned long long)__popc(bal));
    base = __shfl_sync(0xFFFFFFFFu, base, __ffs(bal) - 1);
    if (keep) out[base + __popc(bal & below(lane))] = e;
}
__device__ __forceinline__ void warp_count(bool hit, unsigned long long* cnt) {
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, hit);
    if (bal && (threadIdx.x & 31u) == (uint32_t)(__ffs(bal) - 1)) atomicAdd(cnt, (unsigned long long)__popc(bal));
}

// iteration 1 over every entry of class (p, q): ONB_TB_NONE for decided king pairs, +1 for immediate wins, else 0 (and onto the list)
__global__ void __launch_bounds__(kTbThreads) k_tb_init(const TbParams P, uint32_t p, uint32_t q, uint64_t entries, uint32_t* list,
                                                        unsigned long long* cnt) {
    __shared__ __align__(16) uint32_t s_att[800];
    __shared__ uint32_t s_b[125];
    tb_load_smem(s_att, s_b);
    __syncthreads();
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool win = false, open = false;
    if (e < entries) {
        const TbPos x = tb_unrank(s_b, (uint32_t)e, p, q);
        int16_t v = ONB_TB_NONE;
        if (x.kr != kBlueTemple && x.kb != kRedTemple) {
            const uint32_t c0 = P.cards[x.cfg][x.side * 2u], c1 = P.cards[x.cfg][x.side * 2u + 1u];
            const uint32_t op = x.side ? x.pb : x.pr, ok = 1u << (x.side ? x.kb : x.kr);
            const uint32_t ek = 1u << (x.side ? x.kr : x.kb);
            const uint32_t own = op | ok;
            const uint32_t* T0 = s_att + (x.side * 16u + c0) * 25u;
            const uint32_t* T1 = s_att + (x.side * 16u + c1) * 25u;
            const uint32_t temple = 1u << (x.side ? kRedTemple : kBlueTemple);
            const uint32_t fk = low_bit(ok);
            // the king captures the enemy king or reaches the temple; a pawn captures the enemy king (never shared with a pawn here)
            uint32_t wins = (T0[fk] | T1[fk]) & ~own & (ek | temple);
            for (uint32_t rem = op; rem; rem &= rem - 1) {
                const uint32_t f = low_bit(rem);
                wins |= (T0[f] | T1[f]) & ek;
            }
            win = wins != 0;
            open = !win;
            v = win ? (int16_t)1 : (int16_t)0;
        }
        P.tab[5 * p + q][e] = v;
    }
    warp_count(win, cnt);
    warp_append(open, (uint32_t)e, list, cnt + 1);
}

// iteration k >= 2 over the work list: odd k resolves +k (a child holds -(k-1)), even k resolves -k (every child is a win, the
// largest +(k-1)). Entries resolved by earlier iterations but not yet compacted away are skipped.
__global__ void __launch_bounds__(kTbThreads) k_tb_iter(const TbParams P, uint32_t p, uint32_t q, const uint32_t* __restrict__ list, uint32_t m,
                                                        int32_t k, unsigned long long* cnt) {
    __shared__ __align__(16) uint32_t s_att[800];
    __shared__ uint32_t s_b[125];
    tb_load_smem(s_att, s_b);
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool hit = false;
    int16_t* const T = P.tab[5 * p + q];
    uint32_t e = 0;
    if (i < m) {
        e = list[i];
        if (T[e] == 0) {
            const TbPos x = tb_unrank(s_b, e, p, q);
            const bool odd = (k & 1) != 0;
            const int32_t target = odd ? 1 - k : k - 1;
            const uint32_t side = x.side;
            const uint32_t op = side ? x.pb : x.pr, ok = 1u << (side ? x.kb : x.kr);
            const uint32_t ep = side ? x.pr : x.pb;
            const uint32_t own = op | ok;
            const uint32_t ksq_e = side ? x.kr : x.kb;
            bool any = false, stop = false;
            int32_t maxv = 0;
            // value of the child in which the mover's pieces are (cp, ck) and the enemy's (cep, enemy king unchanged)
            auto child = [&](uint32_t cp, uint32_t ck, uint32_t cep, uint32_t ccfg) -> int32_t {
                const uint32_t rp = side ? cep : cp, bp = side ? cp : cep;
                const uint32_t rk = side ? ksq_e : low_bit(ck), bk = side ? low_bit(ck) : ksq_e;
                const uint32_t cpn = popc32(rp), cqn = popc32(bp);
                return P.tab[5 * cpn + cqn][tb_entry(s_b, rp, bp, rk, bk, ccfg, side ^ 1u, cpn, cqn)];
            };
            auto judge = [&](int32_t v) {
                if (odd) {
                    if (v == target) { hit = true; stop = true; }
                } else if (v <= 0) {
                    stop = true;
                } else if (v > maxv) {
                    maxv = v;
                }
            };
            for (uint32_t s = 0; s < 2 && !stop; ++s) {
                const uint32_t* Ts = s_att + (side * 16u + P.cards[x.cfg][side * 2u + s]) * 25u;
                const uint32_t ccfg = P.child[x.cfg][side * 2u + s];
                for (uint32_t rem = own; rem && !stop; rem &= rem - 1) {
                    const uint32_t f = low_bit(rem);
                    const uint32_t fb = 1u << f;
                    const bool king = (ok & fb) != 0;
                    for (uint32_t a = Ts[f] & ~own; a && !stop; a &= a - 1) {
                        const uint32_t tb = a & (0u - a);
                        any = true;
                        judge(child(king ? op : ((op & ~fb) | tb), king ? tb : ok, ep & ~tb, ccfg));
                    }
                }
            }
            if (!any)  // no legal move: the two pass children
                for (uint32_t s = 0; s < 2 && !stop; ++s) judge(child(op, ok, ep, P.child[x.cfg][side * 2u + s]));
            if (!odd && !stop && maxv == k - 1) hit = true;
            if (hit) T[e] = (int16_t)(odd ? k : -k);
        }
    }
    warp_count(hit, cnt);
}

__global__ void __launch_bounds__(kTbThreads) k_tb_compact(const int16_t* __restrict__ T, const uint32_t* __restrict__ in, uint32_t m,
                                                           uint32_t* __restrict__ out, unsigned long long* cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t e = i < m ? in[i] : 0u;
    warp_append(i < m && T[e] == 0, e, out, cnt);
}

// value of a game, ONB_TB_NONE when it is decided or not a position of the table
__device__ __forceinline__ int32_t tb_lookup(const TbParams& P, const uint32_t* B, const Game& g) {
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

// values [n] (optional) and the number of undecided games outside the table (optional)
__global__ void __launch_bounds__(kTbThreads) k_tb_probe(const TbParams P, const uint4* __restrict__ states, int64_t n, int16_t* values,
                                                         unsigned long long* missing) {
    __shared__ uint32_t s_b[125];
    for (int j = threadIdx.x; j < 125; j += blockDim.x) s_b[j] = g_binom.b[j];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool out = false;
    if (i < n) {
        const Game g = unpack(states[i]);
        const int32_t v = tb_lookup(P, s_b, g);
        if (values) values[i] = (int16_t)v;
        out = v == ONB_TB_NONE && g.result == 0 && current_state(g) == 0;
    }
    if (missing) warp_count(out, missing);
}

// the move onb_tb_best defines for games[i] (nullptr: game i), in generation order of the game's own card slots
__global__ void __launch_bounds__(kTbThreads) k_tb_best(const TbParams P, const uint4* __restrict__ states, const int32_t* __restrict__ games,
                                                        int64_t m, uint16_t* __restrict__ out) {
    __shared__ __align__(16) uint32_t s_att[800];
    __shared__ uint32_t s_b[125];
    tb_load_smem(s_att, s_b);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int64_t game = games ? (int64_t)games[i] : i;
    const Game g = unpack(states[game]);
    const int32_t v = tb_lookup(P, s_b, g);
    uint32_t best = 0xFFFFu;
    if (v != ONB_TB_NONE) {
        const int32_t target = v > 0 ? 1 - v : v < 0 ? -v - 1 : 0;
        const uint32_t side = g.side;
        const uint32_t own_p = side ? g.pawn_b : g.pawn_r, own = own_p | (side ? g.king_b : g.king_r);
        bool any = false;
        for (uint32_t s = 0; s < 2 && best == 0xFFFFu; ++s) {
            const uint32_t* Ts = s_att + (side * 16u + card_at(g.cards, side * 2u + s)) * 25u;
            for (uint32_t rem = own; rem && best == 0xFFFFu; rem &= rem - 1) {
                const uint32_t f = low_bit(rem);
                for (uint32_t a = Ts[f] & ~own; a; a &= a - 1) {
                    any = true;
                    const uint32_t action = make_action(side * 2u + s, f, low_bit(a), ((own_p >> f) & 1u) ^ 1u);
                    Game ch = g;
                    const uint32_t res = apply_move(ch, action);
                    if (v == 1 ? res != 0 : (res == 0 && tb_lookup(P, s_b, ch) == target)) {
                        best = action;
                        break;
                    }
                }
            }
        }
        if (!any)
            for (uint32_t s = 0; s < 2 && best == 0xFFFFu; ++s) {
                const uint32_t action = kPassBit | ((side * 2u + s) << 10);
                Game ch = g;
                apply_move(ch, action);
                if (tb_lookup(P, s_b, ch) == target) best = action;
            }
    }
    out[game] = (uint16_t)best;
}

// ------------------------------------------------------------------------------------------------ host side
static bool tb_cards_ok(const uint8_t cards5[5], uint32_t* setmask) {
    uint32_t m = 0;
    for (int i = 0; i < 5; ++i) {
        if (cards5[i] > 15 || (m >> cards5[i]) & 1u) return false;
        m |= 1u << cards5[i];
    }
    *setmask = m;
    return true;
}
// the cards of configuration cfg: red lo, red hi, blue lo, blue hi, neutral
static void tb_cfg_cards(uint32_t setmask, uint32_t cfg, uint8_t out[5]) {
    uint8_t s[5];
    for (uint32_t id = 0, n = 0; id < 16; ++id)
        if ((setmask >> id) & 1u) s[n++] = (uint8_t)id;
    const uint32_t j = cfg / 6u, r = cfg % 6u;
    static const uint8_t kPair[6][2] = {{0, 1}, {0, 2}, {1, 2}, {0, 3}, {1, 3}, {2, 3}};
    uint8_t rem[4];
    for (uint32_t t = 0, n = 0; t < 5; ++t)
        if (t != j) rem[n++] = s[t];
    const uint8_t a = kPair[r][0], b = kPair[r][1];
    uint8_t blue[2];
    for (uint32_t t = 0, n = 0; t < 4; ++t)
        if (t != a && t != b) blue[n++] = rem[t];
    out[0] = rem[a]; out[1] = rem[b]; out[2] = blue[0]; out[3] = blue[1]; out[4] = s[j];
}
static TbParams tb_params(const Ctx* c) {
    TbParams P;
    memset(&P, 0, sizeof(P));
    for (int k = 0; k < 25; ++k) P.tab[k] = c->tb_len[k] ? c->d_tb + c->tb_off[k] : nullptr;
    P.setmask = c->tb_setmask;
    P.max_pawns = (uint32_t)c->tb_max_pawns;
    for (uint32_t cfg = 0; cfg < 30; ++cfg) {
        uint8_t cc[5];
        tb_cfg_cards(c->tb_setmask, cfg, cc);
        for (int u = 0; u < 4; ++u) {
            P.cards[cfg][u] = cc[u];
            // the used card becomes the neutral one, the old neutral card joins the mover's hand
            const uint32_t red_a = u < 2 ? (u == 0 ? cc[4] : cc[0]) : cc[0];
            const uint32_t red_b = u < 2 ? (u == 1 ? cc[4] : cc[1]) : cc[1];
            P.child[cfg][u] = (uint8_t)card_cfg(c->tb_setmask, cc[u], red_a, red_b);
        }
    }
    return P;
}

void tb_free(Ctx* c) {
    if (c->d_tb) cudaFree(c->d_tb);
    c->d_tb = nullptr;
    c->tb_live = 0;
    memset(c->tb_off, 0, sizeof(c->tb_off));
    memset(c->tb_len, 0, sizeof(c->tb_len));
}

static uint64_t tb_class_entries(uint32_t p, uint32_t q) { return 36000ull * class_subsets(kBinomHost.b, p, q); }

int32_t tb_solve(Ctx* c, const uint8_t cards5[5], int32_t max_pawns, onb_tb_class out[25], char* err, size_t err_len) {
    uint32_t setmask = 0;
    if (!cards5 || !tb_cards_ok(cards5, &setmask) || max_pawns < 0 || max_pawns > ONB_TB_MAX_PAWNS) {
        snprintf(err, err_len, "onb_tb_solve: need five distinct card ids 0..15 and 0 <= max_pawns <= %d", ONB_TB_MAX_PAWNS);
        return ONB_E_INVALID;
    }
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        snprintf(err, err_len, "onb_tb_solve: %s", cudaGetErrorString(e));
        return ONB_E_CUDA;
    }
    tb_free(c);
    uint64_t total = 0, max_cls = 0;
    for (uint32_t p = 0; p <= 4; ++p)
        for (uint32_t q = 0; p + q <= (uint32_t)max_pawns; ++q) {
            const uint64_t en = tb_class_entries(p, q);
            c->tb_off[5 * p + q] = (int64_t)total;
            c->tb_len[5 * p + q] = (int64_t)en;
            total += en;
            if (en > max_cls) max_cls = en;
        }
    uint32_t* lists = nullptr;
    unsigned long long* cnt = nullptr;
    const size_t need = (size_t)total * 2 + (size_t)max_cls * 8 + 16;
    e = cudaMalloc(&c->d_tb, (size_t)total * 2);
    if (e == cudaSuccess) e = cudaMalloc(&lists, (size_t)max_cls * 8);
    if (e == cudaSuccess) e = cudaMalloc(&cnt, 16);
    auto cleanup = [&]() {
        if (lists) cudaFree(lists);
        if (cnt) cudaFree(cnt);
    };
    if (e != cudaSuccess) {
        cleanup();
        tb_free(c);
        cudaGetLastError();
        snprintf(err, err_len, "onb_tb_solve: cannot allocate %zu bytes of device memory (table %zu, work lists %zu): %s", need, (size_t)total * 2,
                 (size_t)max_cls * 8, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;
    }
    c->tb_setmask = setmask;
    c->tb_max_pawns = max_pawns;
    const TbParams P = tb_params(c);
    if (out) memset(out, 0, 25 * sizeof(onb_tb_class));
    int32_t level_max[ONB_TB_MAX_PAWNS + 1] = {0, 0, 0, 0, 0};  // largest |value| of the classes with p + q = level
    int32_t rc = ONB_OK;
#define TB(call)                                                                   \
    do {                                                                           \
        e = (call);                                                                \
        if (e != cudaSuccess) {                                                    \
            snprintf(err, err_len, "onb_tb_solve: %s: %s", #call, cudaGetErrorString(e)); \
            rc = ONB_E_CUDA;                                                       \
            goto done;                                                             \
        }                                                                          \
    } while (0)
    for (uint32_t level = 0; level <= (uint32_t)max_pawns; ++level) {
        int32_t L = 0;
        for (uint32_t l = 0; l < level; ++l) L = level_max[l] > L ? level_max[l] : L;
        for (uint32_t p = 0; p <= level; ++p) {
            const uint32_t q = level - p, cls = 5 * p + q;
            const uint64_t en = (uint64_t)c->tb_len[cls];
            const uint64_t invalid = (uint64_t)kTbDecided * 60u * class_subsets(kBinomHost.b, p, q);
            uint32_t* list = lists;
            uint32_t* spare = lists + max_cls;
            unsigned long long h = 0;
            onb_tb_class st;
            memset(&st, 0, sizeof(st));
            st.entries = (int64_t)en;
            st.invalid = (int64_t)invalid;
            TB(cudaMemsetAsync(cnt, 0, 16, c->stream));
            k_tb_init<<<(unsigned)((en + kTbThreads - 1) / kTbThreads), kTbThreads, 0, c->stream>>>(P, p, q, en, list, cnt);
            TB(cudaGetLastError());
            TB(cudaMemcpyAsync(&h, cnt, 8, cudaMemcpyDeviceToHost, c->stream));
            TB(cudaStreamSynchronize(c->stream));
            st.wins = (int64_t)h;
            st.max_win = h ? 1 : 0;
            st.iterations = 1;
            st.examined = (int64_t)en;
            uint64_t live = en - invalid - h, m = live;
            for (int32_t k = 2; live > 0; ++k) {
                if (k > 32767) {
                    snprintf(err, err_len, "onb_tb_solve: class (%u,%u) needs values beyond int16 (%llu entries unresolved after iteration 32767)",
                             p, q, (unsigned long long)live);
                    rc = ONB_E_OVERFLOW;
                    goto done;
                }
                TB(cudaMemsetAsync(cnt, 0, 8, c->stream));
                k_tb_iter<<<(unsigned)((m + kTbThreads - 1) / kTbThreads), kTbThreads, 0, c->stream>>>(P, p, q, list, (uint32_t)m, k, cnt);
                TB(cudaGetLastError());
                TB(cudaMemcpyAsync(&h, cnt, 8, cudaMemcpyDeviceToHost, c->stream));
                TB(cudaStreamSynchronize(c->stream));
                st.iterations = k;
                st.examined += (int64_t)m;
                if (h) {
                    if (k & 1) { st.wins += (int64_t)h; st.max_win = k; }
                    else { st.losses += (int64_t)h; st.max_loss = k; }
                }
                live -= h;
                if (h == 0 && k > L) break;
                if (live * 4 < m * 3) {  // the list has shrunk by a quarter: keep only the unresolved entries
                    TB(cudaMemsetAsync(cnt + 1, 0, 8, c->stream));
                    k_tb_compact<<<(unsigned)((m + kTbThreads - 1) / kTbThreads), kTbThreads, 0, c->stream>>>(P.tab[cls], list, (uint32_t)m, spare, cnt + 1);
                    TB(cudaGetLastError());
                    uint32_t* t = list; list = spare; spare = t;
                    m = live;
                }
            }
            st.draws = st.entries - st.invalid - st.wins - st.losses;
            st.solved = 1;
            if (st.max_win > level_max[level]) level_max[level] = st.max_win;
            if (st.max_loss > level_max[level]) level_max[level] = st.max_loss;
            if (out) out[cls] = st;
        }
    }
#undef TB
done:
    cudaStreamSynchronize(c->stream);
    cleanup();
    if (rc != ONB_OK) {
        tb_free(c);
        return rc;
    }
    c->tb_live = 1;
    return ONB_OK;
}

cudaError_t launch_tb_probe(Ctx* c, int16_t* d_values, unsigned long long* d_missing) {
    const TbParams P = tb_params(c);
    k_tb_probe<<<(unsigned)((c->n + kTbThreads - 1) / kTbThreads), kTbThreads, 0, c->stream>>>(P, c->d_states, c->n, d_values, d_missing);
    return cudaGetLastError();
}
cudaError_t launch_tb_best(Ctx* c, const int32_t* d_games, int64_t m, uint16_t* d_out) {
    if (m <= 0) return cudaSuccess;
    const TbParams P = tb_params(c);
    k_tb_best<<<(unsigned)((m + kTbThreads - 1) / kTbThreads), kTbThreads, 0, c->stream>>>(P, c->d_states, d_games, m, d_out);
    return cudaGetLastError();
}

}  // namespace onb

using namespace onb;

static uint32_t brev32(uint32_t x) {
    uint32_t r = 0;
    for (int i = 0; i < 32; ++i) r |= ((x >> i) & 1u) << (31 - i);
    return r;
}

extern "C" {

int32_t onb_tb_index(const uint8_t cards5[5], const onb_state* s, int64_t n, int32_t* cls, int64_t* idx) {
    uint32_t setmask = 0;
    if (!cards5 || !tb_cards_ok(cards5, &setmask) || n < 0 || (n && (!s || !cls || !idx))) return ONB_E_INVALID;
    const uint32_t* B = kBinomHost.b;
    for (int64_t i = 0; i < n; ++i) {
        cls[i] = -1;
        idx[i] = -1;
        const uint32_t pr = brev32(s[i].pawns[0]) & kAll25, pb = brev32(s[i].pawns[1]) & kAll25;
        const uint32_t kr = brev32(s[i].kings[0]) & kAll25, kb = brev32(s[i].kings[1]) & kAll25;
        uint32_t seen = 0;
        for (int k = 0; k < 5; ++k) seen |= s[i].cards[k] < 16 ? 1u << s[i].cards[k] : 0x10000u;
        if (seen != setmask || s[i].side > 1 || popc32(kr) != 1 || popc32(kb) != 1 || (kr & kb) || (pr & pb) || ((pr | pb) & (kr | kb))) continue;
        const uint32_t p = popc32(pr), q = popc32(pb);
        if (p + q > ONB_TB_MAX_PAWNS) continue;
        cls[i] = (int32_t)(5 * p + q);
        idx[i] = (int64_t)tb_entry(B, pr, pb, low_bit(kr), low_bit(kb), card_cfg(setmask, s[i].cards[4], s[i].cards[0], s[i].cards[1]), s[i].side, p, q);
    }
    return ONB_OK;
}

int32_t onb_tb_state(const uint8_t cards5[5], int32_t cls, const int64_t* idx, int64_t n, onb_state* out) {
    uint32_t setmask = 0;
    if (!cards5 || !tb_cards_ok(cards5, &setmask) || cls < 0 || cls >= 25 || cls / 5 + cls % 5 > ONB_TB_MAX_PAWNS || n < 0 ||
        (n && (!idx || !out)))
        return ONB_E_INVALID;
    const uint32_t p = (uint32_t)cls / 5, q = (uint32_t)cls % 5;
    const int64_t en = (int64_t)tb_class_entries(p, q);
    for (int64_t i = 0; i < n; ++i)
        if (idx[i] < 0 || idx[i] >= en) return ONB_E_INVALID;
    for (int64_t i = 0; i < n; ++i) {
        const TbPos x = tb_unrank(kBinomHost.b, (uint32_t)idx[i], p, q);
        onb_state& o = out[i];
        memset(&o, 0, sizeof(o));
        o.pawns[0] = brev32(x.pr);
        o.pawns[1] = brev32(x.pb);
        o.kings[0] = brev32(1u << x.kr);
        o.kings[1] = brev32(1u << x.kb);
        tb_cfg_cards(setmask, x.cfg, o.cards);
        o.side = (uint8_t)x.side;
    }
    return ONB_OK;
}

}  // extern "C"
