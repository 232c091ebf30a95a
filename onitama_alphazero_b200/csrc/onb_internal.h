// onb_internal.h -- context layout and launcher prototypes shared by the translation units of libonb.so.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>
#include <string>

#include "../../include/onb.h"

namespace onb {

// One search-tree node: exactly one 32-byte sector. A node's children occupy CONTIGUOUS slots (the
// reference pushes them back to back into its arena, mcts_arena.rs:231-260), so a warp reads a whole
// children block with one coalesced request and every lane gets (N, W, P, header) of its child at once.
struct __align__(32) Node {
    double w;              // MctsNode::reward (sum of backed-up values)      mcts_arena.rs:366-367
    double p;              // MctsNode::probability                           mcts_arena.rs:372
    uint32_t n;            // MctsNode::visits                                mcts_arena.rs:364-365
    uint32_t first_child;  // index of child 0 in this tree's pool
    uint32_t parent;       // 0xFFFFFFFF for the root
    uint16_t action;       // move that leads here (onb_action)
    uint8_t n_child;
    uint8_t flags;         // bit0 expanded, bit1 terminal, bit2 pass pseudo-child, bit3 proven win, bit4 proven loss (DESIGN.md §5k)
};
static_assert(sizeof(Node) == 32, "node must be one sector");
constexpr uint8_t kNodeExpanded = 1, kNodeTerminal = 2, kNodePass = 4;
// MCTS solver (onb_mcts_set_solver, DESIGN.md §5k): the side that moved into the node wins / loses with best play
constexpr uint8_t kNodeWin = ONB_NODE_WIN, kNodeLoss = ONB_NODE_LOSS, kNodeProven = ONB_NODE_WIN | ONB_NODE_LOSS;
constexpr uint8_t kTreePassSeen = 1, kTreeOverflow = 2;
constexpr int kMaxDepth = 32;  // path entries kept in registers (lane l <-> level l); deeper paths spill to the parent chain

// Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f). Every onb_mcts_begin with the switch on rewrites this device struct, so
// a captured simulation round (CUDA graph) reads the current search's step and table instead of baking them into its launches.
constexpr int kGbStride = 64;  // per-tree root-child slots: 8 pieces x 2 cards x 4 moves, the most the lane-group expansion writes
struct GumbelDev {
    double c_visit, c_scale, scale;
    uint64_t seed;
    uint32_t step, m, n_tab, interior;  // n_tab = sims - 1 descents; interior: the search runs the interior-selection kernels
    const uint32_t* tab;                // [m][n_tab]: row m_eff - 1 = seq_halving(m_eff, n_tab)
    double* base;                       // [n][kGbStride] g(a) + (logit(a) - L), written by the root's first descent
    double* p;                          // [n][kGbStride] max(DBL_MIN, P(a) / sum P)
    double* r0;                         // [n] the reward the root's own evaluation backed up into the root
    float* rx;                          // [n][node_cap] r_x: the reward the expanding simulation backed up into node x (interior only)
};

// The resident endgame tablebase as the kernels that probe it take it (by value): class 5 p + q at tab[5 p + q] (nullptr: not in the
// table), the set's cards (bit id) and the largest p + q solved. onb_tablebase.cuh holds the index and the lookup.
struct TbTable {
    int16_t* tab[25];
    uint32_t setmask, max_pawns;
};

// Everything a search is begun with (begin_search). onb_mcts_begin builds it from the context's switches, onb_self_play from its
// config, onb_fight from the agent; the launchers read only the copy in Ctx::search, so a switch changed after the begin does not
// reach the search already running.
struct SearchPlan {
    double c_puct;
    uint32_t sims;
    const int32_t* d_games;  // tree t searches game d_games[t] (device, ascending), t < m; nullptr: every game
    int64_t m;
    bool reuse;              // keep the remembered trees (onb_reuse.cu): the trees are laid out by remaining budget
    bool game_order;         // ... and onb_mcts_finish puts its outputs back into game order (the public onb_mcts_begin)
    bool noise;              // train-mode root noise (onb_mcts_set_noise)
    double noise_eps, noise_alpha;
    uint64_t noise_seed;
    bool gumbel;             // the Gumbel root search (onb_mcts_set_gumbel); gb_cfg.interior: Gumbel MuZero below the root
    onb_gumbel_config gb_cfg;
    uint32_t gb_step;
    uint32_t leaves;         // K >= 2: leaf parallelism with virtual loss (onb_mcts_set_virtual_loss), 0: one descent per round
    double vloss;
    bool tb;                 // tablebase leaves (onb_mcts_set_tablebase, DESIGN.md §5i): begin_search copies the table into tb_table
    TbTable tb_table;
    uint32_t tb_serial;      // Ctx::tb_serial at the begin: the search continues only while that table is resident
    bool solver;             // the MCTS solver (onb_mcts_set_solver, DESIGN.md §5k)
};
// Descents of the next round of a search with virtual loss (DESIGN.md §5h), from the descents done so far (= the root's visits) and
// the target the round counts against: 1 for round 0, then min(K, target - done). The kernels derive it from the root's visit count,
// so a captured round (CUDA graph) runs the right number of descents on every replay.
__host__ __device__ inline uint32_t vl_descents(uint32_t done, uint32_t leaves, uint32_t target) {
    if (done >= target) return 0u;
    if (done == 0u) return 1u;
    return target - done < leaves ? target - done : leaves;
}
// the search begun last
struct ActiveSearch {
    SearchPlan plan;
    uint32_t sims_done;
    int phase;  // 0 idle, 1 begun/after expand, 2 after select
    // the first n_act trees search the games listed in d_tree_game (device, ascending); n_act == 0: every game is searched by the
    // tree of the same index. A subset plan sets them, launch_reuse_begin fills them for a reuse begin.
    int64_t n_act;
    const int32_t* d_tree_game;
    bool finished;       // onb_mcts_finish has run since the last simulation (onb_mcts_choose reads its best)
    uint32_t vl_target;  // with virtual loss: the descent count the current round is counted against (onb_mcts_run's end, or plan.sims)
};

struct Ctx {
    onb_config cfg;
    cudaStream_t stream;
    bool own_stream;
    int64_t n;
    // env
    uint4* d_states;
    uint32_t* d_masks;
    float* d_planes;
    uint16_t* d_actions;
    unsigned long long* d_stats;
    int32_t fixed_cards;  // -1: auto-reset deals from the RNG, else the nibble-packed deck every reset re-deals (onb_env_reset with one deck)
    // scratch for host<->device transfers of boundary structs
    onb_state* d_io_states;
    uint16_t* d_moves;  // [n][40]
    uint8_t* d_counts;  // [n]
    // mcts
    Node* d_nodes;          // [n][node_cap]
    uint32_t node_cap;
    uint32_t* d_tree_size;  // [n]
    uint8_t* d_tree_flags;  // [n]
    uint4* d_roots;         // [n] root states captured by mcts_begin
    uint32_t* d_leaf_node;  // [n] leaf reached by the last select
    uint4* d_leaf_state;    // [n]
    float* d_leaf_planes;   // [n][525]
    float* d_policy;        // [n][50]
    float* d_value;         // [n]
    float* d_pi;            // [n][50]
    uint16_t* d_best;       // [n]
    uint32_t* d_root_visits;
    double* d_root_q;
    uint32_t* d_child_visits;  // [n][40]
    ActiveSearch search;
    int noise_on;           // the switch of onb_mcts_set_noise: Dirichlet-like exploration noise at the root (mcts_arena.rs:186-202)
    double noise_eps, noise_alpha;
    uint64_t noise_seed;
    float* d_ln_table;  // logf(i) for the plain UCT search (filled by the host: the libm call behind Rust's f32::ln)
    uint32_t ln_cap;
    // policy/value network (onb_net.cu): weights in tensor-core operand layout, folded biases, head parameters
    struct NetSlot {
        float* w;     // conv taps in operand layout
        float* bias;  // folded biases
        float* head;  // head parameters
        int blocks, loaded, f16, x3;  // f16: f16 operands (else tf32); x3: split-operand f32-faithful mode (ONB_NET_F32)
        int hid;                      // hidden channels: 64 (the k_net_forward family) or 128 (k_net_wide)
        size_t pair_off;              // x3: byte offset in w of the taps in CTA-pair order (onb_net.cu, k_net_forward_x3p<true>)
    } net[2];         // two networks can be resident (an arena pits the new model against the previous one, evaluator.rs:355-399)
    void* sp_buf[32];          // grow-only buffers of onb_self_play (slots 0-15) and onb_fight (16-31), see onb_selfplay.cu
    size_t sp_cap[32];
    int fight_valid;           // an onb_fight has left its per-game results on the device (onb_fight_statistics)
    int net_cur;      // slot used by onb_net_load / onb_net_forward / ONB_EVAL_NET (onb_net_select)
    int net_tf32;     // requested arithmetic for the next onb_net_load: ONB_NET_F16 (default) | ONB_NET_TF32 | ONB_NET_F32
    // grow-only device scratch reused across onb_perft calls (counters, cursor, two ping-pong frontiers): repeated
    // cudaMalloc/cudaFree of several hundred MB made the call time vary by +-50 %
    void* scratch[16];
    size_t scratch_cap[16];
    // onb_alphabeta_run: per-game root score and node count (allocated on first use)
    int32_t* d_ab_score;
    unsigned long long* d_ab_nodes;
    // tree reuse (onb_reuse.cu, onb_mcts_set_reuse); buffers allocated by the first enabling call
    int reuse_on;         // the switch
    int ru_live;          // the pools hold the remembered trees of the last reuse search (slot layout of d_ru_game / d_ru_slot)
    int64_t ru_m;         // trees of the current reuse search
    Node* d_nodes_alt;    // second pool: the kept subtrees are compacted into it, then the pools swap
    uint4* d_roots_alt;
    uint32_t* d_tree_size_alt;
    int32_t* d_ru_game;   // [n] game searched by slot t (slots ordered by remaining budget, descending)
    int32_t* d_ru_slot;   // [n] slot holding game g's remembered tree, -1: none
    uint4* d_ru_plan;     // [n] per searched game: old slot, kept node, budget, new slot
    uint32_t* d_ru_mat;   // [(mcts_max_sims + 1) * blocks] counting-sort matrix
    uint32_t* d_ru_off;   // [mcts_max_sims + 1] off[r] = trees with budget > r
    uint32_t* h_ru_off;   // host copy (round r of the search runs trees [0, off[r]))
    float* d_ru_pi;       // finish outputs in slot order before onb_mcts_finish puts them into game order
    uint16_t* d_ru_best;
    uint32_t* d_ru_rv;
    double* d_ru_q;
    uint32_t* d_ru_cv;
    uint64_t ru_stats[4];
    // Gumbel root search (onb_mcts_set_gumbel); buffers allocated by the first enabling call
    int gb_on;                // the switch
    onb_gumbel_config gb_cfg;
    uint32_t gb_serial;       // step of the next Gumbel onb_mcts_begin
    GumbelDev* d_gb;          // the device struct every Gumbel begin rewrites
    uint32_t* d_gb_tab;       // [40][mcts_max_sims]
    double* d_gb_base;
    double* d_gb_p;
    double* d_gb_r0;
    float* d_gb_rx;           // [n][node_cap], allocated by the first call that turns interior selection on
    uint32_t gb_tab_m, gb_tab_n;  // the table d_gb_tab holds (gb_tab_m = 0: none)
    // leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h); buffers allocated by the first enabling call
    uint32_t vl_leaves;       // the switch: K (2..32), 0 off
    double vl_loss;
    uint32_t vl_cap;          // K the row buffers are sized for: n * vl_cap rows, row t * K + j = descent j of tree t
    int vl_dirty;             // a select left virtual counts that no expand/backup has cleared (the next begin clears them)
    uint8_t* d_vl_cnt;        // [n][node_cap] virtual visits of the current round (zero between rounds)
    uint32_t* d_vl_leaf_node; // rows: leaf node, packed leaf state, planes [21][5][5], policy [50], value
    uint4* d_vl_leaf_state;
    float* d_vl_planes;
    float* d_vl_policy;
    float* d_vl_value;
    // endgame tablebase (onb_tablebase.cu, onb_tb_solve)
    int16_t* d_tb;            // every solved class, class 5 p + q at d_tb + tb_off[5 p + q]
    int64_t tb_off[25], tb_len[25];  // tb_len = 0: class not in the table
    uint32_t tb_setmask;      // bit id set for the five cards of the set
    int32_t tb_max_pawns;
    int tb_live;              // a solved table is resident
    int tb_search;            // the switch of onb_mcts_set_tablebase (tablebase leaves); tb_free switches it off
    uint32_t tb_serial;       // raised by every tb_free, so a search begun with an earlier table knows it is gone
    int16_t* d_tb_values;     // [n] onb_tb_probe's output, and ONB_AGENT_PUCT_TB's table moves (allocated on first use)
    // self-play move protocol (onb_self_play_set_protocol, DESIGN.md §5j)
    onb_selfplay_protocol sp_proto;  // all zero: off
    double* d_root_m;         // [n] ONB_BUF_ROOT_M, written by k_mcts_choose
    uint8_t* d_choose_mask;   // [n] onb_mcts_choose's sample mask
    int sp_ran;               // an onb_self_play has run (its protocol stats are readable)
    onb_selfplay_protocol_stats sp_stats;
    // MCTS solver (onb_mcts_set_solver, DESIGN.md §5k)
    int solver_on;            // the switch
    int8_t* d_root_proof;     // [n] ONB_BUF_ROOT_PROOF, written by the solver's finish; allocated by the first enabling call
    char err[512];
};

inline int64_t trees(const Ctx* c) { return c->search.n_act > 0 ? c->search.n_act : c->n; }

// env (onb_env.cu)
cudaError_t launch_env_reset(Ctx* c, const uint8_t* d_decks5, int64_t n_decks, uint32_t epoch);
cudaError_t launch_env_reset_where(Ctx* c, const uint8_t* d_mask, uint32_t epoch, unsigned long long* d_count);
cudaError_t launch_states_export(Ctx* c, onb_state* d_out, int64_t first, int64_t n);
cudaError_t launch_states_import(Ctx* c, const onb_state* d_in, int64_t first, int64_t n);
cudaError_t launch_legal_moves(Ctx* c);
cudaError_t launch_observe(Ctx* c, uint32_t out_flags);
cudaError_t launch_env_step(Ctx* c, int mode, uint32_t step, int auto_reset, uint32_t out_flags);
// the same on games [first, first + count) and a stream of the caller's choice (first % 64 == 0); done_bits: [count/32][2] or nullptr
cudaError_t launch_env_step_slice(Ctx* c, int mode, uint32_t step, int auto_reset, uint32_t out_flags, int64_t first, int64_t count,
                                  cudaStream_t stream, uint32_t* done_bits);
// perft (onb_perft.cu)
int32_t run_perft(Ctx* c, const onb_state* roots_host, int64_t n, int depth, uint64_t* nodes, uint64_t* wins, uint64_t* zero);
// mcts (onb_mcts.cu)
cudaError_t launch_selftest_div(Ctx* c, unsigned long long* d_mismatches);
cudaError_t launch_mcts_begin(Ctx* c);
cudaError_t launch_mcts_select(Ctx* c);
cudaError_t launch_mcts_expand_backup(Ctx* c);
cudaError_t launch_mcts_eval(Ctx* c, int evaluator);
cudaError_t launch_mcts_run(Ctx* c, int evaluator, uint32_t sims);
cudaError_t launch_uct_run(Ctx* c, float exploration_c, uint32_t min_node_visits, uint32_t sims);
cudaError_t launch_mcts_finish(Ctx* c, float* pi, uint16_t* best, uint32_t* root_visits, double* root_q, uint32_t* child_visits);
cudaError_t launch_mcts_play_best(Ctx* c, uint32_t out_flags);
cudaError_t launch_mcts_scatter_best(Ctx* c, uint16_t* dst_actions);  // dst[game of tree t] = best[t]
// the self-play protocol's move and m (include/onb.h onb_self_play_set_protocol) of every tree after launch_mcts_finish, into
// dst_actions / d_root_m [game of tree t]. best: the finish's best in tree order. The tree of game i samples iff mask[i] != 0 (mask)
// or plies[i] < temp_plies (plies); both nullptr: no tree samples.
cudaError_t launch_mcts_choose(Ctx* c, const uint16_t* best, uint64_t seed, uint32_t step, double temperature, const uint8_t* mask,
                               const int32_t* plies, uint32_t temp_plies, uint16_t* dst_actions);
// the search launchers take their kernel from c->search.plan: noise, Gumbel at the root (select, run, finish) and Gumbel MuZero
// below it (select, run, expand_backup), virtual loss (select, eval, expand_backup over the K rows of every tree, round target
// search.vl_target), tablebase leaves (expand_backup), the solver (select, run, expand_backup, finish; finish also writes d_root_proof)

// network (onb_net.cu)
int32_t net_load(Ctx* c, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel, std::string& err);
cudaError_t launch_net_forward(Ctx* c, const float* planes, float* policy, float* value, int64_t count);  // count positions

// alpha-beta agent (onb_alphabeta.cu): searches games d_games[0 .. m) (nullptr: games 0 .. m) to `depth` plies; d_out[game] = the best
// action (ONB_ACTION_NONE for a decided game), d_score / d_nodes [game] (optional) = root score and positions entered
cudaError_t launch_alphabeta(Ctx* c, int depth, const int32_t* d_games, int64_t m, uint16_t* d_out, int32_t* d_score, unsigned long long* d_nodes);

// endgame tablebase (onb_tablebase.cu)
int32_t tb_solve(Ctx* c, const uint8_t cards5[5], int32_t max_pawns, onb_tb_class out[25], char* err, size_t err_len);
void tb_free(Ctx* c);
// values [n] of every game (optional) and the number of undecided games outside the table (optional, accumulated)
cudaError_t launch_tb_probe(Ctx* c, int16_t* d_values, unsigned long long* d_missing);
// d_out[game] = onb_tb_best's move for the games d_games[0 .. m) (nullptr: games 0 .. m)
cudaError_t launch_tb_best(Ctx* c, const int32_t* d_games, int64_t m, uint16_t* d_out);
// the same for the listed games in the table only (the others keep d_out[game]), through d_tmp [n]
cudaError_t launch_tb_best_in_table(Ctx* c, const int32_t* d_games, int64_t m, uint16_t* d_out, uint16_t* d_tmp);
TbTable tb_table(const Ctx* c);  // the resident table as the search kernels take it

// tree reuse (onb_reuse.cu)
cudaError_t reuse_alloc(Ctx* c);
void reuse_free(Ctx* c);
// reroot the remembered trees of the m games d_games (nullptr: all games) for a search to `sims` visits, swap the pools, fill
// h_ru_off; leaves search.n_act = m, search.d_tree_game = d_ru_game
cudaError_t launch_reuse_begin(Ctx* c, const int32_t* d_games, int64_t m, uint32_t sims);
cudaError_t launch_reuse_unpermute(Ctx* c);  // d_ru_* (slot order) -> d_pi / d_best / ... (game order)

// native self-play driver (onb_selfplay.cu)
int32_t run_self_play(Ctx* c, const onb_selfplay_config* cfg, onb_selfplay_result* out,
                      int32_t (*search)(Ctx*, const onb_selfplay_config*, uint32_t ply, const int32_t* d_games, int64_t m), char* err,
                      size_t err_len);

int32_t run_fight(Ctx* c, const onb_agent* a, const onb_agent* b, const uint8_t* a_is_red_host, uint32_t max_plies, onb_fight_result* out,
                  int32_t (*move)(Ctx*, const onb_agent*, uint32_t ply, const int32_t* d_games, int64_t m, uint16_t* d_out), char* err, size_t err_len);
int32_t run_fight_statistics(Ctx* c, double rating_a, double rating_b, onb_fight_statistics* out, double* history_host, char* err, size_t err_len);

constexpr int kModeActions = 2;  // env step modes: 0 = ONB_POLICY_UNIFORM, 1 = ONB_POLICY_AGENT, 2 = explicit actions

}  // namespace onb
