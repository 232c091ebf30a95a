// =====================================================================================
// tests/tablebase_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of the endgame tablebase (onb_tb_*, DESIGN.md §5g) in the shape of the reference: positions are `State`s, moves
// come from generate_all_legal_moves and are played with make_move / pass on copies (oracle/onb_oracle.cpp, included below). The
// index is restated from the text of include/onb.h square by square and shares no code with csrc/onb_tablebase.cu.
//
//   orc_tb_solve        the layered forward iteration of the definition, one std::vector<int16_t> per class, host threads
//   orc_tb_check_local  local consistency: an entry equals the rule applied to its children, looked up in the given table
//   orc_tb_check_swap   the colour-swap identity (square n -> 24 - n, boards and hands swapped, neutral kept, side flipped)
//   orc_tb_probe        the value of a game as onb_tb_probe defines it
//   orc_tb_best         the move onb_tb_best defines
// Tables cross this boundary as 25 pointers (class 5 p + q, NULL: not in the table).
// =====================================================================================
#include "../oracle/onb_oracle.cpp"

namespace orc_tb {
using namespace orc;

static const int16_t NONE = -32768;
static const uint16_t ACTION_NONE = 0xFFFF;

static uint64_t binom(int n, int k) {
    if (k < 0 || k > n) return 0;
    uint64_t r = 1;
    for (int i = 0; i < k; ++i) r = r * (uint64_t)(n - i) / (uint64_t)(i + 1);
    return r;
}
static uint64_t subsets(int p, int q) { return binom(23, p) * binom(23 - p, q); }
static uint64_t class_entries(int p, int q) { return 36000ull * subsets(p, q); }

struct Set {
    uint8_t s[5];  // ascending card ids
    bool ok;
};
static Set make_set(const uint8_t cards[5]) {
    Set st;
    st.ok = true;
    for (int i = 0; i < 5; ++i) st.s[i] = cards[i];
    std::sort(st.s, st.s + 5);
    for (int i = 0; i < 5; ++i)
        if (st.s[i] > 15 || (i && st.s[i] == st.s[i - 1])) st.ok = false;
    return st;
}
static int pos_in(const uint8_t* arr, int n, uint8_t id) {
    for (int i = 0; i < n; ++i)
        if (arr[i] == id) return i;
    return -1;
}
// the five deck slots of configuration cfg: red hand ascending, blue hand ascending, neutral
static void cfg_deck(const Set& set, int cfg, uint8_t deck[5]) {
    const int j = cfg / 6, r = cfg % 6;
    uint8_t rem[4];
    for (int i = 0, n = 0; i < 5; ++i)
        if (i != j) rem[n++] = set.s[i];
    // colex order of the pairs {a < b}: rank = C(a, 1) + C(b, 2)
    int a = 0, b = 1;
    for (int bb = 1; bb < 4; ++bb)
        for (int aa = 0; aa < bb; ++aa)
            if ((int)(binom(aa, 1) + binom(bb, 2)) == r) { a = aa; b = bb; }
    deck[0] = rem[a]; deck[1] = rem[b];
    for (int i = 0, n = 2; i < 4; ++i)
        if (i != a && i != b) deck[n++] = rem[i];
    deck[4] = set.s[j];
}
// configuration of a deck, -1 if its five slots are not the set
static int deck_cfg(const Set& set, const uint8_t deck[5]) {
    for (int i = 0; i < 5; ++i)
        if (pos_in(set.s, 5, deck[i]) < 0) return -1;
    for (int i = 0; i < 5; ++i)
        for (int k = 0; k < i; ++k)
            if (deck[i] == deck[k]) return -1;
    const int j = pos_in(set.s, 5, deck[4]);
    uint8_t rem[4];
    for (int i = 0, n = 0; i < 5; ++i)
        if (i != j) rem[n++] = set.s[i];
    int a = pos_in(rem, 4, deck[0]), b = pos_in(rem, 4, deck[1]);
    if (a > b) std::swap(a, b);
    return 6 * j + (int)(binom(a, 1) + binom(b, 2));
}

struct Pos {
    State st;
    int side;
};
static int count_bits(uint32_t b) {
    int c = 0;
    for (unsigned n = 0; n < 25; ++n) c += (int)get_bit(b, n);
    return c;
}
static int only_square(uint32_t b) {
    for (unsigned n = 0; n < 25; ++n)
        if (get_bit(b, n)) return (int)n;
    return -1;
}
// class and entry of a position; false if it is no position of the set's classes with at most max_pawns pawns
static bool index_of(const Set& set, int max_pawns, const State& st, int side, int& cls, uint64_t& idx) {
    const int cfg = deck_cfg(set, st.deck);
    if (cfg < 0 || count_bits(st.kings[RED]) != 1 || count_bits(st.kings[BLUE]) != 1) return false;
    const int kr = only_square(st.kings[RED]), kb = only_square(st.kings[BLUE]);
    if (kr == kb) return false;
    uint32_t all = 0;
    for (int c = 0; c < 2; ++c) {
        if (st.pawns[c] & (st.kings[0] | st.kings[1])) return false;
        all |= st.pawns[c];
    }
    if (st.pawns[RED] & st.pawns[BLUE]) return false;
    const int p = count_bits(st.pawns[RED]), q = count_bits(st.pawns[BLUE]);
    if (p + q > max_pawns) return false;
    // the red pawns' positions among the squares without a king, the blue pawns' among the squares left
    uint64_t rank_r = 0, rank_b = 0;
    int free_r = 0, free_b = 0, i_r = 0, i_b = 0;
    for (unsigned n = 0; n < 25; ++n) {
        if ((int)n == kr || (int)n == kb) continue;
        if (get_bit(st.pawns[RED], n)) rank_r += binom(free_r, ++i_r);
        ++free_r;
        if (get_bit(st.pawns[RED], n)) continue;
        if (get_bit(st.pawns[BLUE], n)) rank_b += binom(free_b, ++i_b);
        ++free_b;
    }
    const uint64_t pair = (uint64_t)(24 * kr + kb - (kb > kr ? 1 : 0));
    idx = (((uint64_t)cfg * 2 + (uint64_t)side) * 600 + pair) * subsets(p, q) + rank_r * binom(23 - p, q) + rank_b;
    cls = 5 * p + q;
    (void)all;
    return true;
}
// the `k` positions (ascending) of colex rank r
static void colex_positions(uint64_t r, int k, int* out) {
    for (int i = k; i >= 1; --i) {
        int c = i - 1;
        while (binom(c + 1, i) <= r) ++c;
        out[i - 1] = c;
        r -= binom(c, i);
    }
}
static Pos position_of(const Set& set, int p, int q, uint64_t e) {
    const uint64_t s = subsets(p, q), sb = binom(23 - p, q);
    const uint64_t sub = e % s, rest = e / s;
    const int kp = (int)(rest % 600), cs = (int)(rest / 600);
    Pos x;
    x.side = cs % 2;
    cfg_deck(set, cs / 2, x.st.deck);
    const int kr = kp / 24, t = kp % 24, kb = t + (t >= kr ? 1 : 0);
    x.st.kings[RED] = x.st.kings[BLUE] = x.st.pawns[RED] = x.st.pawns[BLUE] = 0;
    set_bit(x.st.kings[RED], (unsigned)kr);
    set_bit(x.st.kings[BLUE], (unsigned)kb);
    int pr[4], pb[4];
    colex_positions(sub / sb, p, pr);
    colex_positions(sub % sb, q, pb);
    std::vector<unsigned> fr, fb;
    for (unsigned n = 0; n < 25; ++n)
        if ((int)n != kr && (int)n != kb) fr.push_back(n);
    for (int i = 0; i < p; ++i) set_bit(x.st.pawns[RED], fr[(size_t)pr[i]]);
    for (unsigned n : fr)
        if (!get_bit(x.st.pawns[RED], n)) fb.push_back(n);
    for (int i = 0; i < q; ++i) set_bit(x.st.pawns[BLUE], fb[(size_t)pb[i]]);
    return x;
}

// the children of a position in generation order (passes for a position without a legal move); win = the move wins at once
struct Child {
    uint16_t action;
    State st;
    bool win;
};
static std::vector<Child> children(const State& st, int side) {
    std::vector<Child> out;
    for (const auto& cm : st.generate_all_legal_moves(side)) {
        Child c{encode_action(cm.first, cm.second), st, false};
        c.win = is_win(c.st.make_move(cm.second, side, cm.first));
        out.push_back(c);
    }
    if (out.empty())
        for (unsigned s = 0; s < 2; ++s) {
            Child c{encode_pass((side == RED ? 0u : 2u) + s), st, false};
            c.st.pass((side == RED ? 0u : 2u) + s);
            out.push_back(c);
        }
    return out;
}

struct Tables {
    const Set* set;
    int max_pawns;
    int16_t* const* t;  // [25]
    int16_t value(const State& st, int side) const {
        int cls;
        uint64_t idx;
        if (!index_of(*set, max_pawns, st, side, cls, idx) || !t[cls]) return NONE;
        return t[cls][idx];
    }
};

template <class F>
static void parallel(int64_t n, int threads, F f) {
    std::atomic<int64_t> next{0};
    const int64_t chunk = 4096;
    auto work = [&]() {
        for (int64_t b; (b = next.fetch_add(chunk)) < n;)
            for (int64_t i = b; i < n && i < b + chunk; ++i) f(i);
    };
    if (threads < 1) threads = 1;
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work);
    work();
    for (auto& th : pool) th.join();
}

// the rule of the definition applied to a position's children (the value a consistent table holds)
static int32_t rule(const Tables& T, const Pos& x) {
    const int kr = only_square(x.st.kings[RED]), kb = only_square(x.st.kings[BLUE]);
    if (kr == (int)BLUE_TEMPLE || kb == (int)RED_TEMPLE) return NONE;
    const std::vector<Child> ch = children(x.st, x.side);
    int32_t shortest_loss = 0, longest_win = 0;
    bool all_win = true;
    for (const Child& c : ch) {
        if (c.win) return 1;
        const int32_t v = T.value(c.st, enemy(x.side));
        if (v < 0 && (shortest_loss == 0 || v > shortest_loss)) shortest_loss = v;
        if (v <= 0) all_win = false;
        else if (v > longest_win) longest_win = v;
    }
    if (shortest_loss) return 1 - shortest_loss;
    if (all_win) return -(longest_win + 1);
    return 0;
}

}  // namespace orc_tb

using namespace orc_tb;

extern "C" {

uint64_t orc_tb_entries(int p, int q) { return class_entries(p, q); }

// solves every class with p + q <= max_pawns into tables[5 p + q] (caller-allocated, E(p, q) entries each);
// stats[4 * cls + 0..3] = iterations, longest win, longest loss, solved. Returns 0, or -1 for a bad set.
int orc_tb_solve(const uint8_t cards[5], int max_pawns, int threads, int16_t* const* tables, int32_t* stats) {
    const Set set = make_set(cards);
    if (!set.ok || max_pawns < 0 || max_pawns > 4) return -1;
    const Tables T{&set, max_pawns, tables};
    int32_t level_max[5] = {0, 0, 0, 0, 0};
    for (int level = 0; level <= max_pawns; ++level) {
        int32_t L = 0;
        for (int l = 0; l < level; ++l) L = std::max(L, level_max[l]);
        for (int p = 0; p <= level; ++p) {
            const int q = level - p, cls = 5 * p + q;
            int16_t* tab = tables[cls];
            const int64_t n = (int64_t)class_entries(p, q);
            // iteration 1: decided king pairs, immediate wins
            parallel(n, threads, [&](int64_t e) {
                const Pos x = position_of(set, p, q, (uint64_t)e);
                const int kr = only_square(x.st.kings[RED]), kb = only_square(x.st.kings[BLUE]);
                int16_t v = 0;
                if (kr == (int)BLUE_TEMPLE || kb == (int)RED_TEMPLE) v = NONE;
                else
                    for (const Child& c : children(x.st, x.side))
                        if (c.win) { v = 1; break; }
                tab[e] = v;
            });
            std::vector<uint32_t> open;
            for (int64_t e = 0; e < n; ++e)
                if (tab[e] == 0) open.push_back((uint32_t)e);
            int32_t k = 1, max_win = 0, max_loss = 0;
            for (int64_t e = 0; e < n; ++e)
                if (tab[e] == 1) max_win = 1;
            while (!open.empty()) {
                ++k;
                std::vector<int16_t> next(open.size(), 0);
                parallel((int64_t)open.size(), threads, [&](int64_t i) {
                    const Pos x = position_of(set, p, q, open[(size_t)i]);
                    int32_t longest = 0;
                    bool all_win = true, hit = false;
                    for (const Child& c : children(x.st, x.side)) {
                        const int32_t v = T.value(c.st, enemy(x.side));
                        if (v == 1 - k) hit = true;  // a child lost in k - 1
                        if (v <= 0) all_win = false;
                        else longest = std::max(longest, v);
                    }
                    if (k % 2 == 1 && hit) next[(size_t)i] = (int16_t)k;
                    if (k % 2 == 0 && all_win && longest == k - 1) next[(size_t)i] = (int16_t)-k;
                });
                // the iteration's results become visible together: it read only the values of the earlier iterations
                std::vector<uint32_t> still;
                int64_t resolved = 0;
                for (size_t i = 0; i < open.size(); ++i) {
                    if (next[i]) { tab[open[i]] = next[i]; ++resolved; }
                    else still.push_back(open[i]);
                }
                if (resolved) (k % 2 ? max_win : max_loss) = k;
                open.swap(still);
                if (resolved == 0 && k > L) break;
            }
            stats[4 * cls + 0] = k;
            stats[4 * cls + 1] = max_win;
            stats[4 * cls + 2] = max_loss;
            stats[4 * cls + 3] = 1;
            level_max[level] = std::max(level_max[level], std::max(max_win, max_loss));
        }
    }
    return 0;
}

// entries idx[0 .. n) of class cls (idx NULL: every entry) that differ from the rule; the first `cap` offenders go to bad
int64_t orc_tb_check_local(const uint8_t cards[5], int max_pawns, int16_t* const* tables, int cls, const int64_t* idx, int64_t n,
                           int threads, int64_t* bad, int64_t cap) {
    const Set set = make_set(cards);
    const Tables T{&set, max_pawns, tables};
    const int p = cls / 5, q = cls % 5;
    if (!idx) n = (int64_t)class_entries(p, q);
    std::atomic<int64_t> nbad{0};
    parallel(n, threads, [&](int64_t i) {
        const int64_t e = idx ? idx[i] : i;
        if (rule(T, position_of(set, p, q, (uint64_t)e)) != tables[cls][e]) {
            const int64_t b = nbad.fetch_add(1);
            if (b < cap) bad[b] = e;
        }
    });
    return nbad.load();
}

// entries of class cls whose colour-swapped position (class 5 q + p) holds another value
int64_t orc_tb_check_swap(const uint8_t cards[5], int max_pawns, int16_t* const* tables, int cls, const int64_t* idx, int64_t n, int threads) {
    const Set set = make_set(cards);
    const Tables T{&set, max_pawns, tables};
    const int p = cls / 5, q = cls % 5;
    if (!idx) n = (int64_t)class_entries(p, q);
    std::atomic<int64_t> nbad{0};
    parallel(n, threads, [&](int64_t i) {
        const int64_t e = idx ? idx[i] : i;
        const Pos x = position_of(set, p, q, (uint64_t)e);
        State w;
        w.kings[RED] = w.kings[BLUE] = w.pawns[RED] = w.pawns[BLUE] = 0;
        for (unsigned s = 0; s < 25; ++s)
            for (int c = 0; c < 2; ++c) {
                if (get_bit(x.st.kings[c], s)) set_bit(w.kings[enemy(c)], 24 - s);
                if (get_bit(x.st.pawns[c], s)) set_bit(w.pawns[enemy(c)], 24 - s);
            }
        w.deck[0] = x.st.deck[2]; w.deck[1] = x.st.deck[3]; w.deck[2] = x.st.deck[0]; w.deck[3] = x.st.deck[1]; w.deck[4] = x.st.deck[4];
        if (T.value(w, enemy(x.side)) != tables[cls][e]) nbad.fetch_add(1);
    });
    return nbad.load();
}

// onb_tb_probe's value of each game
void orc_tb_probe(const uint8_t cards[5], int max_pawns, int16_t* const* tables, const orc_state* g, int64_t n, int16_t* out) {
    const Set set = make_set(cards);
    const Tables T{&set, max_pawns, tables};
    for (int64_t i = 0; i < n; ++i) {
        const State st = to_state(g[i]);
        out[i] = (g[i].result != 0 || st.current_state() != IN_PROGRESS) ? NONE : T.value(st, g[i].side);
    }
}

// onb_tb_best's move for each game
void orc_tb_best(const uint8_t cards[5], int max_pawns, int16_t* const* tables, const orc_state* g, int64_t n, int threads, uint16_t* out) {
    const Set set = make_set(cards);
    const Tables T{&set, max_pawns, tables};
    parallel(n, threads, [&](int64_t i) {
        const State st = to_state(g[i]);
        out[i] = ACTION_NONE;
        if (g[i].result != 0 || st.current_state() != IN_PROGRESS) return;
        const int32_t v = T.value(st, g[i].side);
        if (v == NONE) return;
        const int32_t want = v > 0 ? 1 - v : v < 0 ? -v - 1 : 0;
        for (const Child& c : children(st, g[i].side)) {
            if (v == 1 ? c.win : (!c.win && T.value(c.st, enemy(g[i].side)) == want)) {
                out[i] = c.action;
                return;
            }
        }
    });
}

}  // extern "C"
