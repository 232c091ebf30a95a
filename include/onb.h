/*
 * onb.h -- C ABI of the B200-native Onitama self-play hot path (libonb.so).
 *
 * The reference (cyoq/onitama-alphazero) has no FFI of its own: its seam is Rust-level. Every entry
 * point below names the reference interface it replaces (file:line relative to the reference root).
 * The Rust-side `extern "C"` block a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every call returns int32_t: 0 = ONB_OK, < 0 = ONB_E*; onb_last_error(ctx) gives a message.
 *     No C++ exception crosses this boundary. There is NO CPU fallback: without a CUDA device
 *     onb_create fails with ONB_E_CUDA.
 *   - a context owns one CUDA device, one stream and all device memory; it is single-threaded
 *     (one host thread per context, mirroring the reference's one-thread-per-replica self-play,
 *     alphazero-training/src/train.rs:218-245).
 *   - board words at this boundary use the reference bit layout: square n (row-major, (0,0) = a5)
 *     is bit (31 - n) of a uint32_t, low 7 bits zero (onitama-game/src/common/mod.rs:2-4).
 *   - pointers named *_host are host memory; the call copies. Device buffers are exposed through
 *     onb_buffer() as borrowed pointers valid until onb_destroy().
 */
#ifndef ONB_H_
#define ONB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ONB_VERSION 200 /* 200: round 2 (onb_actor_*, onb_comm_*, onb_fight_stats, onb_fight_result.moves_chosen, ONB_NET_F32) */

#if defined(__GNUC__)
#define ONB_API __attribute__((visibility("default")))
#else
#define ONB_API
#endif

/* ---- error codes ---- */
#define ONB_OK 0
#define ONB_E_INVALID (-1)   /* bad argument */
#define ONB_E_CUDA (-2)      /* CUDA runtime error (message has the CUDA error string) */
#define ONB_E_NOMEM (-3)     /* device allocation failed */
#define ONB_E_STATE (-4)     /* call out of sequence (e.g. mcts_select before mcts_begin) */
#define ONB_E_OVERFLOW (-5)  /* a node pool or output buffer was too small */

/* ---- colours, pieces, results (player_color.rs:6-9, piece.rs:6-9, move_result.rs:4-9) ---- */
#define ONB_RED 0
#define ONB_BLUE 1
#define ONB_PAWN 0
#define ONB_KING 1
#define ONB_RESULT_IN_PROGRESS 0
#define ONB_RESULT_RED_WIN 1
#define ONB_RESULT_BLUE_WIN 2

/* ---- action code (replaces DoneMove{mov: Move{from,to,piece}, used_card_idx}, done_move.rs:4-7) ----
 *   bits 0-4 to, 5-9 from, 10-11 used_card_idx (deck slot 0..3), bit 12 piece (1 = King),
 *   bit 13 pass (State::pass(card_idx), state.rs:139-142; only `used_card_idx` is meaningful). */
typedef uint16_t onb_action;
#define ONB_ACTION(card_idx, from, to, piece) \
    ((onb_action)((to) | ((from) << 5) | ((card_idx) << 10) | ((piece) << 12)))
#define ONB_ACTION_PASS(card_idx) ((onb_action)(((card_idx) << 10) | (1u << 13)))
#define ONB_ACTION_NONE ((onb_action)0xFFFFu)

/* ---- one game at the boundary (replaces State + GameState::curr_player_color,
 *      state.rs:51-56, game_state.rs:5-13). 24 bytes. ---- */
typedef struct onb_state {
    uint32_t pawns[2]; /* [Red, Blue], reference bit layout */
    uint32_t kings[2];
    uint8_t cards[5];  /* card ids 0..15 in deck slots RED1, RED2, BLUE1, BLUE2, NEUTRAL (deck.rs:14-18) */
    uint8_t side;      /* side to move */
    uint8_t result;    /* ONB_RESULT_* of the last transition */
    uint8_t flags;     /* bit0: a pass (zero-legal-move turn) happened since the last reset */
} onb_state;

/* ---- random policies for onb_env_step_random ---- */
#define ONB_POLICY_UNIFORM 0 /* uniform over all legal moves, pass if none (ai/mcts/mcts_arena.rs:190-241) */
#define ONB_POLICY_AGENT 1   /* the `Random` agent incl. its quirks (ai/random.rs:12-43) */

/* ---- outputs of a step ---- */
#define ONB_OUT_MASKS 1u   /* policy-shaped legal mask of the NEW state, 2 x uint32 per game */
#define ONB_OUT_PLANES 2u  /* [n,21,5,5] f32 planes of the NEW state (alphazero-training/src/common.rs:26-80) */
#define ONB_OUT_ACTIONS 4u /* the action taken (random policies) */

/* ---- evaluators that live on the device ---- */
#define ONB_EVAL_UNIFORM 0 /* policy = f32(1/50) everywhere, value = 0 (BASELINE config 4) */
#define ONB_EVAL_HASH 1    /* deterministic pseudo-random policy/value from a hash of the planes (parity tests) */
#define ONB_EVAL_NET 2     /* the ConvResNet loaded with onb_net_load, evaluated on the tensor cores */

/* ---- device buffers (onb_buffer) ---- */
#define ONB_BUF_STATES 0      /* packed internal states, 16 B per game (layout in DESIGN.md) */
#define ONB_BUF_MASKS 1       /* uint32[n][2] */
#define ONB_BUF_PLANES 2      /* float[n][21][5][5] */
#define ONB_BUF_ACTIONS 3     /* uint16[n] */
#define ONB_BUF_LEAF_PLANES 4 /* float[n][21][5][5]   written by onb_mcts_select */
#define ONB_BUF_POLICY 5      /* float[n][2][25]      read by onb_mcts_expand_backup */
#define ONB_BUF_VALUE 6       /* float[n]             read by onb_mcts_expand_backup */
#define ONB_BUF_PI 7          /* float[n][2][25]      written by onb_mcts_finish */
#define ONB_BUF_BEST 8        /* uint16[n]            written by onb_mcts_finish */
#define ONB_BUF_STATS 9       /* uint64[ONB_STAT_COUNT] */
/* the rows of a search with virtual loss (onb_mcts_set_virtual_loss), row t * K + j = descent j of tree t, n_games * K' rows with K'
 * the largest K enabled so far (a search with K uses the first n_games * K rows). They exist after the first enabling call (before:
 * ONB_E_STATE); an enabling call with a larger K reallocates them, which invalidates pointers taken earlier (and captured graphs). */
#define ONB_BUF_VL_PLANES 10  /* float[n K'][21][5][5] written by onb_mcts_select */
#define ONB_BUF_VL_POLICY 11  /* float[n K'][2][25]    read by onb_mcts_expand_backup */
#define ONB_BUF_VL_VALUE 12   /* float[n K']           read by onb_mcts_expand_backup */
#define ONB_BUF_ROOT_M 13     /* double[n]            written by onb_mcts_choose: max(v_root, q_best) */
#define ONB_BUF_ROOT_PROOF 14 /* int8[n]              written by onb_mcts_finish of a solver search (onb_mcts_set_solver) */

#define ONB_STAT_STEPS 0     /* transitions applied */
#define ONB_STAT_RED_WINS 1
#define ONB_STAT_BLUE_WINS 2
#define ONB_STAT_PASSES 3
#define ONB_STAT_RESETS 4
#define ONB_STAT_BAD_ACTIONS 5 /* host actions rejected by onb_env_step / onb_actor_submit (from or to square > 24) */
#define ONB_STAT_COUNT 8

typedef struct onb_ctx onb_ctx;

typedef struct onb_config {
    int32_t device;         /* CUDA device ordinal */
    uint32_t flags;         /* reserved, 0 */
    int64_t n_games;        /* games (= search trees) owned by this context */
    uint64_t game_id_base;  /* global id of local game 0; the RNG is keyed by the GLOBAL id, so results
                               do not depend on how games are sharded over GPUs */
    uint64_t seed;
    void* stream;           /* cudaStream_t to launch on; NULL = the context creates its own */
    uint32_t mcts_max_sims; /* 0 = no search-tree pools */
    uint32_t mcts_node_cap; /* nodes per tree; 0 = hard bound 1 + 40 * mcts_max_sims */
    uint32_t alloc_planes;  /* 0/1: allocate the [n,21,5,5] plane buffer */
    uint32_t reserved;
} onb_config;

/* ------------------------------------------------------------------------------------------------
 * lifecycle
 * ------------------------------------------------------------------------------------------------ */
ONB_API int32_t onb_version(void);
ONB_API int32_t onb_create(const onb_config* cfg, onb_ctx** out);
ONB_API int32_t onb_destroy(onb_ctx* ctx);
ONB_API const char* onb_last_error(const onb_ctx* ctx);
ONB_API int32_t onb_sync(onb_ctx* ctx);
/* the cudaStream_t every call of this context launches on (so the network and copies can be ordered with it) */
ONB_API int32_t onb_get_stream(onb_ctx* ctx, void** stream);
ONB_API int32_t onb_buffer(onb_ctx* ctx, int32_t which, void** dev_ptr, int64_t* bytes);

/* copy a whole device buffer to / from host memory on the context's stream (synchronous). Lets a host-side evaluator
 * (the reference's ConvResNet::forward on CPU tensors, net.rs:215-232) sit between onb_mcts_select and
 * onb_mcts_expand_backup without any CUDA code on the caller's side. bytes must not exceed the buffer size. */
ONB_API int32_t onb_read_buffer(onb_ctx* ctx, int32_t which, void* host, int64_t bytes);
ONB_API int32_t onb_write_buffer(onb_ctx* ctx, int32_t which, const void* host, int64_t bytes);

/* host-side helpers (pure C, no device): */
/* State::with_deck (state.rs:67-73) + first mover = neutral card's stamp (game_state.rs:34-41) */
ONB_API int32_t onb_start_states(const uint8_t* decks5, int64_t n, onb_state* out);
/* the shared counter RNG (project-defined; the reference uses rand::thread_rng) */
ONB_API uint32_t onb_rand_u32(uint64_t seed, uint64_t game, uint32_t step, uint32_t draw);
/* random deal = first 5 of a shuffle of the 16 cards (replaces Deck::default, deck.rs:139-151) */
ONB_API int32_t onb_deal(uint64_t seed, uint64_t game, uint32_t epoch, uint8_t out5[5]);
/* ATTACK_MAPS[2][16][25] in the reference layout (card.rs:476): the table the kernels stage into shared memory */
ONB_API int32_t onb_attack_maps(uint32_t out800[800]);

/* ------------------------------------------------------------------------------------------------
 * env: lockstep batched game dynamics
 * ------------------------------------------------------------------------------------------------ */
/* (re)start every game. n_decks = 0: deal from the RNG with `epoch`; 1: the same deck for all games;
 * n_games: one deck per game. Replaces State::with_deck / GameState::with_deck (train.rs:44-49). */
ONB_API int32_t onb_env_reset(onb_ctx* ctx, const uint8_t* decks5_host, int64_t n_decks, uint32_t epoch);
/* Re-deals selected games in place (start position, cards from the counter RNG at `epoch`, or the fixed deck of the last
 * onb_env_reset): mask_host[i] != 0 selects game i; mask_host == NULL selects every game that is over. *n_reset (optional)
 * receives the number of games restarted. This is what keeps every slot of a lockstep self-play busy: a worker of the
 * reference starts its next game as soon as one ends (train.rs:44-98 inside the per-thread loop of :218-245). */
ONB_API int32_t onb_env_reset_games(onb_ctx* ctx, const uint8_t* mask_host, uint32_t epoch, int64_t* n_reset);
ONB_API int32_t onb_env_set_states(onb_ctx* ctx, const onb_state* states_host, int64_t first, int64_t n);
ONB_API int32_t onb_env_get_states(onb_ctx* ctx, onb_state* states_host, int64_t first, int64_t n);
/* State::generate_all_legal_moves (state.rs:301-378) for the side to move of every game.
 * moves_host: [n][40] action codes in reference order, counts_host: [n]; either may be NULL. */
ONB_API int32_t onb_env_legal_moves(onb_ctx* ctx, onb_action* moves_host, uint8_t* counts_host);
/* policy-shaped mask (word s = union of `to` of own hand slot s); masks_host [n][2] may be NULL
 * (result stays in ONB_BUF_MASKS). */
ONB_API int32_t onb_env_legal_masks(onb_ctx* ctx, uint32_t* masks_host);
/* create_tensor_from_state (common.rs:26-80) for every game into ONB_BUF_PLANES; planes_host may be NULL */
ONB_API int32_t onb_env_encode(onb_ctx* ctx, float* planes_host);
/* State::make_move / State::pass + side switch (state.rs:139-202, game_state.rs:65-80) with the given
 * actions. actions_host NULL = use ONB_BUF_ACTIONS as already filled on the device. Finished games and games
 * whose action is ONB_ACTION_NONE are left untouched; so is a game whose action names a from or to square above 24 (the reference
 * would index out of its 25-square board: such actions are counted in ONB_STAT_BAD_ACTIONS instead of corrupting the packed state). auto_reset: a game that ends is replaced by a fresh deal (RNG epoch step+1; `step` is only
 * used for that). out_flags selects which observation buffers of the new state are written. */
ONB_API int32_t onb_env_step(onb_ctx* ctx, const onb_action* actions_host, uint32_t step, int32_t auto_reset,
                             uint32_t out_flags);
/* one lockstep step of every unfinished game with a random policy drawn from the counter RNG keyed by
 * (seed, global game id, step). auto_reset: a game that ends is replaced by a fresh deal (epoch step+1). */
ONB_API int32_t onb_env_step_random(onb_ctx* ctx, uint32_t step, int32_t policy, int32_t auto_reset, uint32_t out_flags);
/* the same random policies as agents for the arena loop: write the chosen action of every unfinished game to
 * ONB_BUF_ACTIONS without playing it (Agent::generate_move of `Random`, ai/random.rs:12-43) */
ONB_API int32_t onb_env_choose_random(onb_ctx* ctx, uint32_t step, int32_t policy);
/* `n_steps` steps back to back starting at `step0` (no host round trip in between) */
ONB_API int32_t onb_env_run_random(onb_ctx* ctx, uint32_t step0, uint32_t n_steps, int32_t policy, int32_t auto_reset,
                           uint32_t out_flags);
/* BASELINE config 1: every game is played from its current state until it ends or max_plies more plies were
 * made, entirely in registers (no per-step launch). Equivalent to onb_env_step_random(step0), (step0+1), ...
 * plies_host [n] and trace_host [n] (a hash chain over the action codes, defined in DESIGN.md) may be NULL.
 * Replaces the random-vs-random game loop of evaluator.rs:355-399 / ai/mcts/mcts_arena.rs:190-241. */
ONB_API int32_t onb_env_playout(onb_ctx* ctx, uint32_t step0, uint32_t max_plies, int32_t policy, uint32_t* plies_host,
                        uint64_t* trace_host);
ONB_API int32_t onb_env_stats(onb_ctx* ctx, uint64_t stats_host[ONB_STAT_COUNT], int32_t clear);

/* ---- host-acted stepping, pipelined inside the library ------------------------------------------------------------------
 * The env loop of a self-play driver whose policy lives on the HOST (train.rs:55-80 with generate_move on the Rust side): per
 * step the actions go in and "what happened" comes out. The context's games are cut into n_sub contiguous sub-batches
 * (boundaries on multiples of 64 games); each has its own stream, pinned host staging and completion event, so while the host
 * consumes sub-batch j the other n_sub - 1 are copying or stepping and PCIe never idles behind a kernel (4 is a good n_sub).
 *   onb_actor_create(ctx, n_sub, out_flags, host_flags, &actor)
 *       out_flags  = ONB_OUT_* observation buffers written ON THE DEVICE every step (planes stay in HBM for the network);
 *       host_flags = what is copied back to pinned host memory every step:
 *         ONB_HOST_MASKS  uint32[count][2]     policy-shaped legal masks of the new states (8 B / game)
 *         ONB_HOST_DONE   uint32[count/32][2]  per 32 games one word pair: bit j of [w][0] = game first+32w+j was WON BY RED in this
 *                                              step, bit j of [w][1] = won by Blue (2 bits / game: all a z back-fill needs)
 *         ONB_HOST_STATS  uint64[ONB_STAT_COUNT] the context's counters as of this sub-batch's step
 *   onb_actor_get_view(actor, j, &view)    the sub-batch's range and its pinned host buffers (library-owned, valid until destroy)
 *   onb_actor_submit(actor, j, actions_host, step, auto_reset)
 *       asynchronous: H2D of the sub-batch's `count` actions (actions_host, or view.actions when NULL; pinned memory keeps the
 *       copy asynchronous) -> onb_env_step semantics on the slice -> D2H of the host_flags outputs -> event. actions_host must
 *       stay untouched until onb_actor_wait.
 *   onb_actor_wait(actor, j)               blocks on that ONE event; afterwards view.masks / done / stats hold the step's outputs
 *   onb_actor_replay(actor, trace, stride, step0, n_steps, auto_reset)
 *       the same ring driven by the library: action of game g at step t = trace[t * stride + g] (replay of recorded games)
 *   onb_actor_join(actor)                  orders the context's own stream after everything submitted (no host block); the next
 *                                          submit re-forks. Other context calls must not overlap with sub-batches in flight.
 * Results equal onb_env_step on the whole context (tests/test_gpu_parity.py::test_actor_pipeline_*). */
#define ONB_HOST_MASKS 1u
#define ONB_HOST_DONE 2u
#define ONB_HOST_STATS 4u
typedef struct onb_actor onb_actor;
typedef struct onb_actor_view {
    int64_t first, count;
    onb_action* actions; /* [count]        pinned staging the host may fill (optional: submit accepts any host pointer) */
    uint32_t* masks;     /* [count][2]     NULL unless ONB_HOST_MASKS */
    uint32_t* done;      /* [count/32][2]  NULL unless ONB_HOST_DONE */
    uint64_t* stats;     /* [ONB_STAT_COUNT] NULL unless ONB_HOST_STATS */
} onb_actor_view;
ONB_API int32_t onb_actor_create(onb_ctx* ctx, int32_t n_sub, uint32_t out_flags, uint32_t host_flags, onb_actor** out);
ONB_API int32_t onb_actor_destroy(onb_actor* actor);
ONB_API int32_t onb_actor_get_view(onb_actor* actor, int32_t sub, onb_actor_view* view);
ONB_API int32_t onb_actor_submit(onb_actor* actor, int32_t sub, const onb_action* actions_host, uint32_t step, int32_t auto_reset);
ONB_API int32_t onb_actor_wait(onb_actor* actor, int32_t sub);
ONB_API int32_t onb_actor_join(onb_actor* actor);
ONB_API int32_t onb_actor_replay(onb_actor* actor, const onb_action* trace_host, int64_t stride, uint32_t step0, uint32_t n_steps,
                                 int32_t auto_reset);

/* ------------------------------------------------------------------------------------------------
 * perft-style enumeration (BASELINE config 2)
 * nodes/wins/zero are host arrays [n][depth]: positions reached by exactly d+1 plies (a line stops at
 * a win), how many of them are wins, and non-terminal positions at depth d that have no legal move.
 * ------------------------------------------------------------------------------------------------ */
ONB_API int32_t onb_perft(onb_ctx* ctx, const onb_state* roots_host, int64_t n, int32_t depth, uint64_t* nodes_host,
                  uint64_t* wins_host, uint64_t* zero_host);

/* ------------------------------------------------------------------------------------------------
 * batched AlphaZero PUCT search, one tree per game, rooted at the current env states
 * (replaces MctsArena::{new,search,playout,select,expand,evaluate,back_propagate},
 *  alphazero-training/src/alphazero_mcts/mcts_arena.rs:48-323). Eval mode only.
 * Split phase so the network stays outside:
 *   onb_mcts_begin; repeat sims times { onb_mcts_select; <evaluator writes POLICY/VALUE from LEAF_PLANES>;
 *   onb_mcts_expand_backup }; onb_mcts_finish.
 * or fused with a device evaluator: onb_mcts_begin; onb_mcts_run; onb_mcts_finish.
 * ------------------------------------------------------------------------------------------------ */
ONB_API int32_t onb_mcts_begin(onb_ctx* ctx, double c_puct, uint32_t sims);
/* train mode (AlphaZeroMctsConfig::train, alphazero_mcts/mod.rs:26-43): at the ROOT every uct() evaluation uses
 * P' = P (1 - epsilon) + noise epsilon with a fresh Dirichlet(alpha; k) component (a Beta(alpha, (k-1) alpha) variate) per evaluation and a left-to-right max_by
 * fold (mcts_arena.rs:186-220). The reference draws from thread_rng (not reproducible); here the draws come from the counter RNG
 * keyed by (seed, global tree id, root visit count), so a run is repeatable. Reference values: epsilon 0.25, alpha 0.03.
 * Applies to the searches started after the call; enabled = 0 restores eval mode. Statistical parity only (DESIGN.md). */
ONB_API int32_t onb_mcts_set_noise(onb_ctx* ctx, int32_t enabled, double epsilon, double alpha, uint64_t seed);
/* Tree reuse between moves (off by default; with it off every entry point behaves exactly as without this call).
 * On: onb_mcts_begin and every ply of onb_self_play keep, per game, the subtree of the last reuse-enabled search whose root
 * position equals the game's current state: a child of that search's root is kept when the game is undecided and its boards,
 * five card slots and side to move equal the position the child's action leads to (siblings always lead to different positions,
 * so no action of the caller is needed, and onb_env_reset / onb_env_set_states / any move stay sound). No match: a fresh root.
 * The kept subtree is the played child and all its descendants in arena order (a stable filter of the old pool; parent and
 * first_child renumbered, the new root has no parent, every other field -- N, W, P, action, n_child, flags -- unchanged). Root W
 * is carried over as it is: later backups keep the same alternating sign, so root Q stays consistent.
 * `sims` becomes a visit TARGET: a tree runs max(0, sims - N_root) simulations, so a root never exceeds sims visits and the node
 * bound 1 + 40 * mcts_max_sims still holds. onb_mcts_run after a reuse begin must be given the begin's sims. onb_mcts_finish reports
 * over all of the root's visits, kept ones included. Outputs (finish, play_best, dump_tree, tree_info) stay in game order; the
 * pools are laid out internally by remaining budget. Train-mode noise is keyed by (seed, game, root visit count) as before.
 * Refused after a reuse begin (ONB_E_STATE): the caller-driven split phase (onb_mcts_select / _eval / _expand_backup) and
 * onb_uct_run. onb_fight ignores the switch (its two agents share the pools). Remembered trees are forgotten by any search without
 * reuse (onb_mcts_begin with reuse off, onb_fight), by onb_self_play's start and by switching reuse off.
 * Memory: the first enabling call allocates a second node pool of n_games * node_cap * 32 bytes (the kept subtrees are compacted
 * into it, then the pools swap), doubling node memory: 2 x 16.8 GB for 16 384 games x 800 simulations. */
ONB_API int32_t onb_mcts_set_reuse(onb_ctx* ctx, int32_t enabled);
/* counters of the reuse-enabled searches since the last clear: out[ONB_REUSE_TREES] trees searched, [ONB_REUSE_KEPT] trees that
 * started with kept visits, [ONB_REUSE_KEPT_VISITS] root visits carried over (counted up to the target), [ONB_REUSE_SIMS]
 * simulations run (= leaf evaluations). clear != 0 zeroes them after the read; out may be NULL. */
#define ONB_REUSE_TREES 0
#define ONB_REUSE_KEPT 1
#define ONB_REUSE_KEPT_VISITS 2
#define ONB_REUSE_SIMS 3
ONB_API int32_t onb_mcts_reuse_stats(onb_ctx* ctx, uint64_t out[4], int32_t clear);
/* Gumbel root search (Danihelka et al., "Policy improvement by planning with Gumbel", ICLR 2022; the root part of mctx's
 * gumbel_muzero_policy). Off by default; with it off every entry point behaves exactly as without this call. On: the searches begun
 * afterwards select at the ROOT by sequential halving over Gumbel-Top-k samples and report the improved policy; below the root the
 * PUCT descent is unchanged unless interior = 1 (interior selection, below). Definition (exact to the bit, DESIGN.md §5f), per tree, with k root children (pass pseudo-children
 * included), P(a) the stored prior, N(a), W(a) visits and reward sum, q(a) = W(a) / N(a), r0 = the reward the root's own evaluation
 * (simulation 0) backed up into the root and v = -r0:
 *   logit(a) = onb_log(P(a)) (-inf for P = 0), L = max logit, p(a) = max(DBL_MIN, P(a) / sum P); if every prior is 0, every P counts as 1;
 *   g(a) = gumbel_scale * (-onb_log(-onb_log(u))), u = (r + 0.5) 2^-32, r = onb_rand_u32(seed, global game id, step, 0x10000 + a);
 *   v_mix = (v + sum N * (sum_{N>0} p q / sum_{N>0} p)) / (sum N + 1)  (the quotient is 0 when no child is visited);
 *   qhat(a) = q(a) if N(a) > 0 else v_mix; sigma(a) = ((c_visit + max N) * c_scale) * ((qhat - min qhat) / max(max qhat - min qhat, 1e-8));
 *   score(a) = max(-1e9, (g(a) + (logit(a) - L)) + sigma(a)).
 * Descent i (i = N_root - 1) chooses the FIRST child of maximal score among those with N(a) = seq(min(m, k), sims - 1)[i] (child 0 if
 * none), seq being mctx's sequential-halving table; onb_mcts_finish's best = the same with N(a) = max N, and pi = softmax over the
 * children of logit + sigma (onb_exp of the difference to the maximum) summed per policy index (hand slot & 1, to) in f64, then f32.
 * All f64 sums run in child order. onb_log / onb_exp are the project's own f64 log / exp from IEEE basic operations (fdlibm's
 * algorithms), so the CPU and the GPU agree to the bit. root_visits, root_q and child_visits are reported as before.
 * step: onb_mcts_begin uses a serial that this call sets to step0 and every Gumbel begin increments; onb_self_play uses step = ply,
 * onb_fight step = ply for ONB_AGENT_GUMBEL and ONB_AGENT_GUMBEL_MUZERO agents (both leave the serial as they found it).
 * Checks: 1 <= max_considered <= 40, finite c_visit, c_scale, gumbel_scale >= 0, else ONB_E_INVALID. cfg NULL or enabled = 0: off.
 * Refused with ONB_E_STATE at onb_mcts_begin: Gumbel together with tree reuse or train-mode noise; after a Gumbel begin: onb_uct_run
 * and more simulations than the begin's sims. onb_self_play while Gumbel is on: ONB_E_STATE with tree reuse on, ONB_E_INVALID with train != 0. onb_fight searches
 * without reuse, so its Gumbel agents play whatever the reuse switch says. Every begin decides anew: a search begun with the switch
 * off is a PUCT search. The caller-driven split phase is supported.
 * Memory: the first enabling call allocates n_games * 1 KB of per-tree root data and a 40 x mcts_max_sims table; the first call with
 * interior = 1 also n_games * mcts_node_cap * 4 B for r_x (16 384 games x 800 simulations: 2.1 GB).
 *
 * Interior selection (interior = 1; the rest of mctx's gumbel_muzero_policy, gumbel_muzero_interior_action_selection): every descent
 * step at depth >= 1 at an expanded, non-terminal node x chooses by the rule below instead of the PUCT argmax. The root keeps the
 * sequential halving above, and onb_mcts_finish's best and pi are unchanged. With k children of x, P(a) the stored prior (the
 * per-card renormalised prior, as at the root; mctx's raw network logits differ from its log by a constant per card), N(a), W(a),
 * q(a) = W(a) / N(a):
 *   r_x = the reward the expanding simulation backed up into x (stored when the expansion succeeds), v = -r_x;
 *   p(a), v_mix, sigma(a) exactly as at the root with r_x in place of r0 (the all-priors-0 rule, the sums in child order, c_visit,
 *     c_scale, the 1e-8 floor: mctx's qtransform_completed_by_mix_value with the node's raw value);
 *   z(a) = logit(a) + sigma(a), logit(a) = onb_log(P(a)) (-inf for P = 0; P counts as 1 when every prior of x is 0);
 *   e(a) = onb_exp(z(a) - max z), pi'(a) = e(a) / sum e (the sum in child order);
 *   choice = the FIRST child maximising pi'(a) - N(a) / (1 + sum N), sum N over x's children (mctx's _prepare_argmax_input + argmax).
 * All f64 with IEEE basic operations (no FMA contraction), so the CPU oracle gives the same bits. It needs no c_puct. interior = 0
 * keeps PUCT below the root; any other value than 0 or 1: ONB_E_INVALID. The refusals above hold unchanged. If allocating r_x fails the
 * call returns ONB_E_NOMEM and leaves the switch as it was. */
typedef struct onb_gumbel_config {
    int32_t enabled;
    uint32_t max_considered; /* m, the number of root actions sampled without replacement (mctx default 16) */
    double c_visit, c_scale, gumbel_scale; /* 50, 0.1, 1 (0: a deterministic search) */
    uint64_t seed;
    uint32_t step0;
    uint32_t interior; /* 0: PUCT below the root, 1: interior selection below the root (Gumbel MuZero) */
} onb_gumbel_config;
ONB_API int32_t onb_mcts_set_gumbel(onb_ctx* ctx, const onb_gumbel_config* cfg);
/* Leaf parallelism with virtual loss (the remedy of AlphaGo Zero, Leela and KataGo for searches over few trees; DESIGN.md §5h). Off by
 * default; leaves <= 1 switches it off, and every entry point then computes what it computes without this call. 2 <= leaves <= 32
 * with a finite virtual_loss >= 0 switches it on for the searches begun afterwards; any other value: ONB_E_INVALID. With K = leaves,
 * vl = virtual_loss, a search begun with the switch on runs in ROUNDS (exact to the bit):
 *   descents: round 0 has b = 1 descent (it evaluates the root), every later round b = min(K, descents left), counted against the
 *     current onb_mcts_run call's sims or, in the split phase, against the begin's sims; the search never runs more than the begin's
 *     sims (beyond: ONB_E_STATE). Every descent is a visit, so the root ends with exactly sims visits and at most 1 + 40 sims nodes.
 *   descent j (0 <= j < b) of a tree starts at the root and goes on while the node is expanded and not terminal. At node x it
 *     chooses the LAST child c maximising u = q' + (c_puct P) (sqrt(Np') / (N' + 1)), q' = W' / N' (0 if N' = 0), with
 *     v(c) = the earlier descents 0 .. j-1 of this round whose path contains c (the leaf included; v = j at the root),
 *     N' = N(c) + v(c), W' = W(c) if v(c) = 0, else W(c) - vl v(c) (W is kept from the view of the side that moved into c, so a
 *     pending descent counts as a lost visit for the chooser), Np' = N(x) + v(x); f64, IEEE basic operations, no FMA contraction.
 *     With v = 0 this is the PUCT selection bit for bit. Terminal marking during the descent is unchanged.
 *   leaves: the leaf of descent j of tree t is row t K + j of ONB_BUF_VL_PLANES / _POLICY / _VALUE. The evaluator runs over
 *     trees x K rows (rows j >= b are no descents, their output is ignored; the rows are zeroed at allocation, so they are finite).
 *   expand/backup: per tree, for j = 0 .. b-1 in order: a leaf still unexpanded and not terminal is expanded with row j's policy
 *     (a leaf an earlier descent of the round expanded is not expanded again); then row j's reward is backed up along the parent
 *     chain as without virtual loss. All virtual counts are zero after every round.
 * onb_mcts_select fills the rows, onb_mcts_eval evaluates them (ONB_EVAL_NET included), onb_mcts_expand_backup consumes them; every
 * onb_mcts_select / _eval / _expand_backup triple is one round. onb_mcts_run runs the same rounds (device evaluators too). Outputs
 * (onb_mcts_finish, play_best, dump_tree, tree_info) read the tree as before.
 * Refused with ONB_E_STATE: a begin with the switch on together with train-mode noise, the Gumbel root search or tree reuse;
 * onb_uct_run after such a begin; onb_self_play while the switch is on. onb_fight searches with virtual loss only for
 * ONB_AGENT_PUCT_VL agents, whatever the switch says, and leaves the switch as it found it.
 * Memory: the first enabling call allocates n_games * mcts_node_cap bytes of virtual counts and n_games * K rows of about 2.3 KB;
 * a later call with a larger K reallocates the rows. A failed allocation returns ONB_E_NOMEM and leaves the switch as it was. */
ONB_API int32_t onb_mcts_set_virtual_loss(onb_ctx* ctx, uint32_t leaves, double virtual_loss);
ONB_API int32_t onb_mcts_select(onb_ctx* ctx);
ONB_API int32_t onb_mcts_expand_backup(onb_ctx* ctx);
ONB_API int32_t onb_mcts_eval(onb_ctx* ctx, int32_t evaluator); /* fills POLICY/VALUE from LEAF_PLANES on the device */
ONB_API int32_t onb_mcts_run(onb_ctx* ctx, int32_t evaluator, uint32_t sims);
/* calculate_priors + best child (mcts_arena.rs:83-124). Any host pointer may be NULL.
 * best [n], pi [n][2][25], root_visits [n], root_q [n], child_visits [n][40] (zero padded, child order) */
ONB_API int32_t onb_mcts_finish(onb_ctx* ctx, onb_action* best_host, float* pi_host, uint32_t* root_visits_host,
                        double* root_q_host, uint32_t* child_visits_host);
/* apply the best action of every tree to its game (self_play: state.make_move(&mov.mov, ...), train.rs:70-72) */
ONB_API int32_t onb_mcts_play_best(onb_ctx* ctx, uint32_t out_flags);

typedef struct onb_tree_dump { /* host arrays of length cap */
    uint32_t* visits;
    double* reward;
    double* prior;
    onb_action* action;
    int32_t* parent;
    uint32_t* first_child;
    uint32_t* n_child;
    uint8_t* flags; /* bit0 expanded, bit1 terminal, bit2 pass child, ONB_NODE_WIN, ONB_NODE_LOSS (onb_mcts_set_solver) */
} onb_tree_dump;
/* copies tree `tree` (arena order == reference arena order); *n_nodes receives the node count */
ONB_API int32_t onb_mcts_dump_tree(onb_ctx* ctx, int64_t tree, int64_t cap, onb_tree_dump* out, int64_t* n_nodes);
/* per-tree summary: node counts [n], flags [n] (bit0: a zero-legal-move node was expanded -> parity with the
 * reference is undefined for that tree, bit1: node pool overflow) */
ONB_API int32_t onb_mcts_tree_info(onb_ctx* ctx, uint32_t* n_nodes_host, uint8_t* flags_host);

/* ---- self_play (alphazero-training/src/train.rs:35-98) for all games of the context, natively -------------------------------
 * Plays exactly max(n_games, slots) games, every one of them TO ITS END: per ply { planes of every slot (train.rs:58); search of
 * the slots with a game in progress (evaluator = ONB_EVAL_*, ONB_EVAL_NET for the loaded network; train != 0: root exploration
 * noise, epsilon 0.25 / alpha 0.03); record (planes, pi, colour); play the best move; finished games (a win, or max_plies + 2
 * plies: the ply cap of train.rs:74-79) get their z = reward(result, sample colour); their slots -- in slot order -- start the
 * next game at once while games remain to be started and go idle afterwards }. No game is abandoned when the quota is reached
 * (dropping the games still running would drop the LONG ones and bias z / pi; a worker of the reference plays its
 * self_play_game_amnt games to completion). Two 8-byte counters per ply cross PCIe.
 * The result points at device buffers owned by the context (valid until the next onb_self_play / onb_destroy): sample
 * i = ply * n_games_of_ctx + slot; valid_idx[0 .. n_valid) lists, ascending, the samples of the completed games (all games
 * unless truncated). serial = slot + n * (games finished before in that slot).
 * sample_cap bounds the buffers (samples; >= one ply); truncated = 1 if it was reached first (running games are then dropped).
 * Requires onb_config.alloc_planes and mcts_max_sims >= sims. Every game is dealt from the counter RNG (epoch = ply + 1). */
typedef struct onb_selfplay_config {
    double c_puct;
    uint32_t sims;
    int32_t evaluator;
    int64_t n_games;
    uint32_t max_plies; /* train.rs: 150 */
    int32_t train;
    uint64_t noise_seed;
    int64_t sample_cap;
} onb_selfplay_config;
typedef struct onb_selfplay_result {
    int64_t n_samples, n_valid, n_games, plies_run;
    int32_t truncated, reserved;
    float* planes;      /* [n_samples][21][5][5] */
    float* pi;          /* [n_samples][2][25] */
    float* z;           /* [n_samples] */
    uint8_t* color;     /* [n_samples] side to move */
    int64_t* serial;    /* [n_samples] */
    int64_t* valid_idx; /* [n_valid] */
} onb_selfplay_result;
ONB_API int32_t onb_self_play(onb_ctx* ctx, const onb_selfplay_config* cfg, onb_selfplay_result* out);

/* ---- AlphaZero's self-play move protocol: opening temperature and resignation (DESIGN.md §5j) -------------------------------
 * A context setting read by every later onb_self_play; NULL or an all-zero struct switches it off, and with it off onb_self_play
 * computes exactly what it computes without this call. Per searched tree of game slot s, with p = plies already played in the slot's
 * current game, tick = the loop's ply, gen = the slot's generation, g = game_id_base + s, N(c) / W(c) = the root children's visits
 * and reward sums in child order (pass children included), best = onb_mcts_finish's best child:
 *   move: p >= temp_plies: best. p < temp_plies: w(c) = onb_exp(onb_log(N(c)) / temperature) for N(c) > 0, else 0; S = the sum of
 *     w in child order; u = (r + 0.5) 2^-32 with r = onb_rand_u32(seed, g, tick, 0x20000); the move is the first child whose
 *     inclusive running sum exceeds u S, else (rounding) the last child with N > 0, else (no visited child) best. All f64, IEEE basic
 *     operations, no FMA contraction, the same onb_log / onb_exp on the CPU and the GPU. pi stays the visit distribution.
 *   value: m = max(v_root, q_best) with v_root = -W_root / N_root (the root's value from the side to move's view; W_root is stored
 *     from the other side's) and q_best = W(best) / N(best); m = v_root when N(best) = 0.
 *   held out: onb_rand_u32(seed, g, gen, 0x20001) < floor(resign_holdout 2^32), compared as uint64 (h = 1 holds out every game).
 *   resignation (resign = 1): a game that is not held out ends at the first search with m < resign_below (strict). That ply's sample
 *     is recorded, no move is played, the side to move loses (z = -1 on its samples, +1 on the opponent's) and the slot restarts or
 *     goes idle exactly as after a win. Held-out games play to their end.
 * For every completed held-out game the run keeps (in the order the games end, slot order within a ply) its serial, its result (0 a
 * draw at the ply cap, 1 Red, 2 Blue) and min m over Red's and over Blue's searches (+inf for a side that never searched).
 * Checks: temperature finite and > 0 when temp_plies > 0, resign 0 or 1, resign_below finite and resign_holdout in [0, 1] when
 * resign = 1; otherwise ONB_E_INVALID and the setting stays as it was. onb_self_play with temp_plies > 0 while the Gumbel root
 * search is on: ONB_E_STATE (Gumbel plays its sequential-halving winner); resignation combines with every search. */
typedef struct onb_selfplay_protocol {
    uint32_t temp_plies; /* T: plies of a game that sample their move, 0 = off (AlphaGo Zero: 30) */
    uint32_t resign;     /* 1: resignation on */
    double temperature;  /* tau */
    double resign_below; /* v_resign */
    double resign_holdout; /* h: fraction of games that never resign */
    uint64_t seed;
} onb_selfplay_protocol;
ONB_API int32_t onb_self_play_set_protocol(onb_ctx* ctx, const onb_selfplay_protocol* protocol);
/* after an onb_self_play: games that ended by resignation, completed held-out games and their records (device pointers, valid until
 * the next onb_self_play, like onb_selfplay_result). ONB_E_STATE before the first onb_self_play. */
typedef struct onb_selfplay_protocol_stats {
    int64_t resigned, held_out;
    int64_t* serial;  /* [held_out] */
    uint8_t* result;  /* [held_out] 0 draw, 1 Red, 2 Blue */
    double* min_m;    /* [held_out][2] min m over Red's, Blue's searches */
} onb_selfplay_protocol_stats;
ONB_API int32_t onb_self_play_protocol_stats(onb_ctx* ctx, onb_selfplay_protocol_stats* out);
/* the protocol's move and value for the trees of the last search, after its onb_mcts_finish: tree of game i samples its move at
 * temperature `temperature` with r = onb_rand_u32(seed, game_id_base + i, step, 0x20000) when sample_mask_host[i] != 0 (NULL: no
 * game samples) and plays best otherwise. The moves go to ONB_BUF_ACTIONS, m to ONB_BUF_ROOT_M (game order). Games no tree searched
 * keep both. ONB_E_STATE without a finished search, ONB_E_INVALID for a temperature that is not finite and > 0. */
ONB_API int32_t onb_mcts_choose(onb_ctx* ctx, uint64_t seed, uint32_t step, double temperature, const uint8_t* sample_mask_host);
/* host copy of a borrowed device pointer (onb_buffer, onb_selfplay_result), ordered after the work queued on the context's stream */
ONB_API int32_t onb_copy_to_host(onb_ctx* ctx, void* host, const void* device, int64_t bytes);

/* ---- fight (alphazero-training/src/evaluator.rs:355-399) for all games of the context in lockstep -----------------------------
 * Two agents, each game played from its current position (call onb_env_reset first) until it is decided or max_plies + 2 plies
 * were played (the ply cap of evaluator.rs:386-392; such games count as draws). a_is_red_host[i] != 0: agent A plays Red in game
 * i (the reference swaps colours every game). Agents: ONB_AGENT_RANDOM = the `Random` agent (ai/random.rs, draws keyed by the
 * ply); ONB_AGENT_PUCT = AlphaZeroMcts (evaluator = ONB_EVAL_*, for ONB_EVAL_NET the resident network net_slot, sims, c);
 * ONB_AGENT_UCT = `Mcts` (sims playouts, c, min_node_visits); ONB_AGENT_ALPHABETA = `AlphaBeta` (onb_alphabeta_run below, depth in
 * plies = sims, 1 <= sims <= ONB_ALPHABETA_MAX_DEPTH; needs no search-tree pools). results (device, [n]: 0 undecided, 1 Red won, 2 Blue won) stays
 * valid until the next onb_fight; results_host (optional) receives a copy. The Elo update of evaluator.rs:58-110 is a fold over
 * these per-game results in game order: onb_fight_stats below. */
#define ONB_AGENT_RANDOM 0
#define ONB_AGENT_PUCT 1
#define ONB_AGENT_UCT 2
#define ONB_AGENT_ALPHABETA 3
/* ONB_AGENT_GUMBEL: the Gumbel root search (onb_mcts_set_gumbel) with evaluator / net_slot / sims as ONB_AGENT_PUCT, m = min_node_visits
 * (0: 16, at most 40), c_scale = c, c_visit = 50, gumbel_scale = 1, seed = onb_config.seed, step = ply, and c_puct = 2 for the PUCT
 * descent below the root. ONB_AGENT_PUCT agents search with
 * PUCT whatever the context's Gumbel switch says; onb_fight leaves that switch as it found it. */
#define ONB_AGENT_GUMBEL 4
/* ONB_AGENT_GUMBEL_MUZERO: as ONB_AGENT_GUMBEL (the same fields and defaults) with interior = 1: Gumbel MuZero, interior selection
 * below the root instead of PUCT. ONB_AGENT_GUMBEL agents search with interior = 0 whatever the context's setting says. */
#define ONB_AGENT_GUMBEL_MUZERO 6
/* ONB_AGENT_PUCT_VL: as ONB_AGENT_PUCT with virtual loss (onb_mcts_set_virtual_loss): K = min_node_visits (2 .. 32, else
 * ONB_E_INVALID) descents per round and vl = 1. Every other agent searches without virtual loss, whatever the switch says. */
#define ONB_AGENT_PUCT_VL 7
typedef struct onb_agent {
    int32_t kind;
    int32_t evaluator;
    int32_t net_slot;
    uint32_t sims;
    double c;
    uint32_t min_node_visits;
    uint32_t reserved;
} onb_agent;
typedef struct onb_fight_result {
    int64_t a_wins, b_wins, draws, plies_run;
    uint8_t* results;
    int64_t moves_chosen; /* (game, ply) pairs an agent had to choose a move for: each ply an agent searches ONLY the undecided games in
                             which it is to move (evaluator.rs:379), never the opponent's */
} onb_fight_result;
ONB_API int32_t onb_fight(onb_ctx* ctx, const onb_agent* a, const onb_agent* b, const uint8_t* a_is_red_host, uint32_t max_plies,
                          onb_fight_result* out, uint8_t* results_host);
/* FightStatistics of the last onb_fight (evaluator.rs:38-110), folded ON THE DEVICE over the per-game results in game order:
 * W/L/D of agent A in total and per colour it played, win rates, and the sequential Elo updates of EloRating::elo_change
 * (elo_rating.rs:53-70, K = 32) starting from (rating_a, rating_b). history_host (optional): [n][4] doubles = before_a, after_a,
 * before_b, after_b per game (RatingChange). color index 0 = games A played as Red, 1 = as Blue. */
typedef struct onb_fight_statistics {
    int64_t n_games, wins, loses, draws;
    int64_t color_wins[2], color_loses[2], color_draws[2];
    double winrate, color_winrate[2];
    double rating_a, rating_b;
} onb_fight_statistics;
ONB_API int32_t onb_fight_stats(onb_ctx* ctx, double rating_a, double rating_b, onb_fight_statistics* out, double* history_host);

/* ---- the one collective of the path: replay samples to the trainer GPU (SURVEY 8e; replaces the join + extend over the worker
 * threads of train.rs:241-245) ------------------------------------------------------------------------------------------------
 * Games shard over GPUs with no data-path collective; at the end of a self-play iteration every rank ships its samples (planes
 * [m][21][5][5], pi [m][2][25], z [m], all f32: 2 304 B per sample) to the trainer rank over NVLink / NVSwitch. NCCL is bound at
 * run time (dlopen of the libnccl.so.2 already mapped in the process, else the system one): without NCCL these calls return
 * ONB_E_STATE and everything else keeps working.
 *   onb_comm_unique_id(id)                      rank 0 makes an id and hands it to the other ranks (any host channel)
 *   onb_comm_create(ctx, n_ranks, rank, id, existing, &comm)
 *                                               one communicator per context (ncclCommInitRank on the context's device); or pass
 *                                               existing = an ncclComm_t the host already owns (id may then be NULL)
 *   onb_selfplay_pack(ctx, &result, &planes, &pi, &z, &m)
 *                                               the valid samples of an onb_self_play result as contiguous device arrays
 *   onb_gather_counts(ctx, comm, m_local, counts_host, &total)
 *                                               collective: every rank learns every rank's sample count (to size the buffers)
 *   onb_gather_samples(ctx, comm, dst_rank, planes, pi, z, m_local, out_planes, out_pi, out_z, out_cap, counts_host, &total)
 *                                               collective over all ranks of comm, on the context's stream: counts and the
 *                                               destination's capacity are exchanged (one 16-byte all-gather + host read), then
 *                                               rank dst_rank receives every rank's samples concatenated in rank order into its
 *                                               out_* DEVICE buffers (capacity out_cap samples; ignored on other ranks);
 *                                               counts_host [n_ranks] and total are filled on every rank. If the total exceeds
 *                                               the destination's capacity EVERY rank returns ONB_E_OVERFLOW and nothing is sent.
 *                                               The data transfer itself is asynchronous on the stream. */
typedef struct onb_comm onb_comm;
ONB_API int32_t onb_comm_unique_id(uint8_t id_out[128]);
ONB_API int32_t onb_comm_create(onb_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t id[128], void* existing_nccl_comm, onb_comm** out);
ONB_API int32_t onb_comm_destroy(onb_comm* comm);
ONB_API int32_t onb_selfplay_pack(onb_ctx* ctx, const onb_selfplay_result* res, float** planes, float** pi, float** z, int64_t* m_out);
ONB_API int32_t onb_gather_counts(onb_ctx* ctx, onb_comm* comm, int64_t m_local, int64_t* counts_host, int64_t* total);
ONB_API int32_t onb_gather_samples(onb_ctx* ctx, onb_comm* comm, int32_t dst_rank, const float* planes, const float* pi, const float* z,
                                   int64_t m_local, float* out_planes, float* out_pi, float* out_z, int64_t out_cap, int64_t* counts_host,
                                   int64_t* total);

/* ---- the trainer's replay buffer on the device (train.rs:213,241-245: `data_buffer = Vec::with_capacity(buffer_size)`, extended by
 * every iteration's self-play and never trimmed by the reference; minibatches by `data_buffer.iter().choose_multiple(&mut rng,
 * train_batch_size)`, train.rs:280-283) ----------------------------------------------------------------------------------
 * A fixed-capacity ring in HBM (2 304 B per sample: planes, pi, z). onb_replay_add appends DEVICE arrays (what onb_selfplay_pack
 * or onb_gather_samples produced; the newest samples overwrite the oldest). onb_replay_sample gathers min(batch, size) DISTINCT
 * samples, uniformly at random, into three contiguous device arrays owned by the ring (valid until the next sample / destroy) that
 * the trainer wraps as tensors: state [B,21,5,5], pi [B,2,25], z [B] (train.rs:285-310 stacks the same three batches). The choice
 * is a keyed pseudo-random permutation of [0, size) (the reference draws from thread_rng): (seed, size) -> the same minibatch;
 * onb_replay_indices returns the ring slots it selects (pure host helper). All device work is asynchronous on the context's stream. */
typedef struct onb_replay onb_replay;
ONB_API int32_t onb_replay_create(onb_ctx* ctx, int64_t capacity, onb_replay** out);
ONB_API int32_t onb_replay_destroy(onb_replay* rb);
ONB_API int32_t onb_replay_add(onb_replay* rb, const float* planes_dev, const float* pi_dev, const float* z_dev, int64_t m);
ONB_API int32_t onb_replay_size(onb_replay* rb, int64_t* size, int64_t* capacity);
ONB_API int32_t onb_replay_sample(onb_replay* rb, int64_t batch, uint64_t seed, float** planes, float** pi, float** z, int64_t* n_out);
ONB_API int32_t onb_replay_indices(int64_t size, int64_t batch, uint64_t seed, int64_t* out);

/* ---- plain UCT with random rollouts: the `Mcts` agent (onitama-game/src/ai/mcts/{mod.rs,mcts_arena.rs}) ---------------
 * The evaluation opponent of the reference's arena (evaluator.rs), one tree per game, rooted like the PUCT search:
 * onb_mcts_begin (its c_puct is ignored); onb_uct_run(ctx, exploration_c, min_node_visits, playouts);
 * onb_mcts_finish (best = the root child with most visits, last maximum wins = max_by_key of mcts_arena.rs:64-67; pi =
 * visit shares) / onb_mcts_play_best / onb_mcts_dump_tree (reward = the f32 reward sum, exactly). Defaults of the
 * reference: exploration_c = sqrt(2), min_node_visits = 5, 5000 playouts (mod.rs:21-30; its 1 s wall-clock limit is
 * not reproduced). The rollouts draw from the counter RNG keyed by (seed, global game id, playout, ply). */
ONB_API int32_t onb_uct_run(onb_ctx* ctx, float exploration_c, uint32_t min_node_visits, uint32_t playouts);

/* ---- fixed-depth alpha-beta: the `AlphaBeta` agent (onitama-game/src/ai/alpha_beta/{mod.rs,evaluation.rs}) ----------------
 * One search per game of the context, rooted at its current state, one game per GPU thread. The search is this project's own
 * definition (DESIGN.md §5d); its play is NOT pinned to the reference, whose evaluation tables and wall-clock limit are not
 * reproduced: the reference deepens iteratively until a time limit, this search runs to a fixed depth in plies.
 *   negamax with alpha-beta, fail-hard, int32 scores from the side to move's view, root window (-WIN - 1, WIN + 1), WIN = 1 000 000;
 *   a node at ply p below the root with depth left >= 1 whose side to move has a move that wins at once (captures the enemy king or
 *     puts the own king on the enemy temple) scores WIN - (p + 1), its best move is the first such move, no child is entered;
 *   otherwise children in generation order (hand slot, from, to ascending), score = -search(child, -beta, -alpha, depth - 1, p + 1),
 *     a child replaces the best move only with a strictly greater score, cut-off at alpha >= beta; a node without a legal move has
 *     the two pass children ONB_ACTION_PASS(slot 0), then slot 1 (the reference panics there);
 *   a leaf (depth left 0) scores eval = V(mover) - V(opponent), V = sum over pawns (100 + 4 adv + 2 ctr) + 6 (6 - manhattan(king,
 *     enemy temple)), adv = rows advanced from the own home row, ctr = 2 - |col - 2|.
 * best_host [n] (first maximal move in generation order), score_host [n] (exact root score), nodes_host [n] (positions entered,
 * root and leaves included) may each be NULL; the chosen actions also stay in ONB_BUF_ACTIONS, where onb_env_step takes them.
 * A decided game (result != 0 or State::current_state is a win) gets ONB_ACTION_NONE, score 0, 0 nodes.
 * depth outside 1 .. ONB_ALPHABETA_MAX_DEPTH: ONB_E_INVALID. Works on a context created with mcts_max_sims = 0. */
#define ONB_ALPHABETA_MAX_DEPTH 8
ONB_API int32_t onb_alphabeta_run(onb_ctx* ctx, int32_t depth, onb_action* best_host, int32_t* score_host, uint64_t* nodes_host);

/* ---- endgame tablebases (DESIGN.md §5g; the reference has none, so this definition is the project's own) ---------------------
 * Position: the four boards, the red hand and the blue hand as unordered pairs of cards, the neutral card and the side to move
 * (result, flags and the order within a hand are not part of it; that order only changes the generation order of the moves).
 * Game value, from the side to move's view, with unbounded play (no ply cap). The children of a position are its legal moves in
 * generation order (hand slot, from, to ascending); a position without a legal move has the two pass children ONB_ACTION_PASS of
 * its hand slot 0, then slot 1 (as in §5d). A move that captures the enemy king or puts the own king on the enemy temple wins at once.
 *   +n (n odd): win in n plies (the winning move is ply n; the winner minimises n, the loser maximises it; passes count as plies);
 *   -n (n even, >= 2): loss in n plies;  0: draw (neither side can force a win);  ONB_TB_NONE: not a position of the table.
 *   A position is +1 iff it has an immediately winning move; +n iff its smallest child loss is -(n-1); -n iff every child is a win
 *   and the largest is +(n-1); every other position is a draw. A value that does not fit in int16 makes the solve fail with
 *   ONB_E_OVERFLOW.
 * Index (public: part of the ABI). Card set: five distinct ids, s0 < ... < s4 sorted. Card configuration cfg = 6 j + r (0..29):
 * j = the neutral card's position in the sorted set, r = the colex rank of the red pair among the four remaining cards renumbered
 * 0..3; the blue hand is the other two. Class (p, q): p red and q blue pawns, p + q <= max_pawns <= ONB_TB_MAX_PAWNS, class id
 * 5 p + q, E(p, q) = 36 000 C(23, p) C(23 - p, q) entries. With squares n = 5 row + col (a5 = 0), entry
 *   ((cfg 2 + side) 600 + 24 kr + kb - [kb > kr]) C(23,p) C(23-p,q) + rank_r C(23-p,q) + rank_b,
 * rank_r = the colex rank of the red pawns' squares among the 23 squares without a king, rank_b = that of the blue pawns' squares
 * among the 23 - p squares left (a square's position among the free squares is s - popc(occupied below s)). Entries with the red
 * king on square 2 or the blue king on 22 (47 of the 600 king pairs) are decided positions and hold ONB_TB_NONE.
 *
 * onb_tb_solve: solves the classes with p + q <= max_pawns of the set cards5 (any order) on the device, replacing any table the
 *   context holds; out[5 p + q] receives the per-class counts (solved = 0 for the classes not in the table). Duplicate ids, ids
 *   above 15 or max_pawns outside 0..4: ONB_E_INVALID; a failed allocation: ONB_E_NOMEM (the message gives the bytes needed).
 *   Works on a context created with mcts_max_sims = 0. The table stays resident until onb_tb_free, the next solve or onb_destroy.
 * onb_tb_table: the device table of class (red_pawns, blue_pawns), borrowed, E(p, q) int16 entries.
 * onb_tb_probe: the value of every game of the context; ONB_TB_NONE for a decided game (result != 0 or State::current_state is a
 *   win), a game whose five card slots are another set, or whose class is not solved.
 * onb_tb_best: per game, in generation order of the game's actual slots (passes included), in a win in n the first move that wins
 *   at once (n = 1) or the first whose child holds -(n-1); in a loss in n the first whose child holds +(n-1); in a draw the first
 *   whose child holds 0. ONB_ACTION_NONE for a game outside the table. The moves also stay in ONB_BUF_ACTIONS.
 * Probe, best and the table pointer return ONB_E_STATE when no table is resident.
 * onb_tb_index (pure host): class and entry of each state; cls = idx = -1 for a state that is no position of the set's classes.
 * onb_tb_state (pure host): the states of entries of one class, each hand in ascending card order, then the neutral card,
 *   result = flags = 0; ONB_E_INVALID for an entry out of range.
 * ONB_AGENT_TABLEBASE in onb_fight plays onb_tb_best in the games in which it is to move (sims and c are ignored). onb_fight checks at
 * its start that every undecided game is in the table (ONB_E_INVALID otherwise; ONB_E_STATE without a table); a game cannot leave the
 * table by moving, because material only decreases. */
#define ONB_TB_MAX_PAWNS 4
#define ONB_TB_NONE ((int16_t)-32768)
#define ONB_AGENT_TABLEBASE 5
typedef struct onb_tb_class {
    int64_t entries, wins, losses, draws, invalid;
    int32_t max_win, max_loss;  /* longest win / loss in plies */
    int32_t iterations, solved; /* solved = 0: class not in the table */
    int64_t examined;           /* work-list entries examined over all iterations */
} onb_tb_class;
ONB_API int32_t onb_tb_solve(onb_ctx* ctx, const uint8_t cards5[5], int32_t max_pawns, onb_tb_class out[25]);
ONB_API int32_t onb_tb_free(onb_ctx* ctx);
ONB_API int32_t onb_tb_table(onb_ctx* ctx, int32_t red_pawns, int32_t blue_pawns, int16_t** dev_ptr, int64_t* entries);
ONB_API int32_t onb_tb_probe(onb_ctx* ctx, int16_t* values_host); /* [n] */
ONB_API int32_t onb_tb_best(onb_ctx* ctx, onb_action* best_host); /* [n], also left in ONB_BUF_ACTIONS */
ONB_API int32_t onb_tb_index(const uint8_t cards5[5], const onb_state* s, int64_t n, int32_t* cls, int64_t* idx);
ONB_API int32_t onb_tb_state(const uint8_t cards5[5], int32_t cls, const int64_t* idx, int64_t n, onb_state* out);
/* Tablebase leaves (DESIGN.md §5i): the PUCT search probes the resident table at its leaves. Off by default; enabled = 0 switches it
 * off, and every entry point then computes what it computes without this call. enabled != 0 switches it on for the searches begun
 * afterwards (ONB_E_STATE without a resident table); onb_tb_free and onb_tb_solve switch it off. A search begun with the switch on
 * (exact to the bit) takes, at the leaf L a descent reaches, v = the resident table's value of L's position by onb_tb_probe's rule
 * (ONB_TB_NONE for a decided position, another card set or a class the table does not hold):
 *   v = ONB_TB_NONE: as without the switch.
 *   v != ONB_TB_NONE, L not the root: L is NOT expanded (it stays an unexpanded node, n_child 0 and flags unchanged, on every later
 *     visit) and the evaluator's policy and value of L are ignored. The reward backed up is that of a decided leaf whose winner is the
 *     table's winner: reward colour = the colour of L's parent, so -1 if v > 0 (the side to move at L wins), +1 if v < 0, 0 if v = 0.
 *   v != ONB_TB_NONE, L the root (its first descent): the root is expanded with the evaluator's policy as without the switch (a search
 *     must have children) and backs up +1 / -1 / 0 by the sign of v, from the root mover's view.
 *   The backup is unchanged. Material never increases, so below a root inside the table every leaf is in the table or decided.
 * The rule holds in every search path: with virtual loss row j's leaf follows it (a table leaf is never expanded, so "an earlier
 * descent of the round expanded it" never applies to it); the Gumbel root and interior selection are unchanged above the leaf (r_x
 * is stored on expansion only); train-mode noise only touches the selection. onb_mcts_run with ONB_EVAL_UNIFORM / ONB_EVAL_HASH runs
 * the split phase's rounds (select, evaluation, expand/backup: three launches per simulation) instead of the fused kernel, so such a
 * search is launch-bound with few trees and slower than the fused one with many (DESIGN.md §5i has the measured cost); ONB_EVAL_NET
 * rounds are unchanged apart from the expand/backup. Refused with ONB_E_STATE: a begin with the switch on together with tree reuse; onb_uct_run after such a
 * begin; onb_self_play while the switch is on; onb_mcts_select / _run / _expand_backup of a search begun with the switch on after
 * onb_tb_free or onb_tb_solve (the search never reads a freed table). onb_fight probes the table only for ONB_AGENT_PUCT_TB agents,
 * whatever the switch says, and leaves the switch as it found it. */
ONB_API int32_t onb_mcts_set_tablebase(onb_ctx* ctx, int32_t enabled);
/* ONB_AGENT_PUCT_TB: as ONB_AGENT_PUCT (the same fields) with the table: in a game whose position is in the resident table it plays
 * onb_tb_best's move, in every other game it plays an eval-mode PUCT search with tablebase leaves (so games of another card set get
 * plain PUCT). It needs a resident table (ONB_E_STATE otherwise); unlike ONB_AGENT_TABLEBASE, games need not start in the table. */
#define ONB_AGENT_PUCT_TB 8

/* MCTS solver (DESIGN.md §5k; Winands, Bjornsson & Saito 2008): the PUCT search proves wins and losses and propagates the proofs to the
 * root. Off by default; enabled = 0 switches it off, and every entry point then computes what it computes without this call. enabled
 * != 0 switches it on for the searches begun afterwards and allocates ONB_BUF_ROOT_PROOF (reading that buffer before the first enabling
 * call gives ONB_E_STATE). A search begun with the switch on computes, exact to the bit:
 *   Flags (onb_tree_dump.flags): ONB_NODE_WIN = the side that moved into the node wins with best play, ONB_NODE_LOSS = it loses. A node
 *     never carries both; "proven" = either. The root follows the same convention: a root proven LOSS means its side to move wins.
 *   Sources of proof: (1) a child that a descent finds terminal gets TERMINAL | WIN (in Onitama a move only ends the game in the
 *     mover's favour); (2) at every successful expansion each child whose action captures on the enemy king's square, or moves the own
 *     king onto the enemy temple, is born TERMINAL | WIN; (3) with tablebase leaves (onb_mcts_set_tablebase) a table leaf below the
 *     root of value v gets LOSS if v > 0, WIN if v < 0, and no proof if v = 0 (draws are not proven).
 *   Propagation: after each descent's expansion and backup, from the deepest node that became proven up the descent's path: the parent
 *     of a node proven WIN becomes LOSS; the parent of a node proven LOSS becomes WIN if every child of it (pass pseudo-children
 *     included) is LOSS; it stops at the first level that does not change, or at the root.
 *   Selection: a descent stops at a proven node (the root included: once the root is proven every later descent ends there). At an
 *     unproven expanded node the PUCT argmax (last maximal child) skips children flagged LOSS; such a node has no WIN child and not
 *     every child is LOSS, so the choice is always defined.
 *   Reward: a descent that ends at a proven node, or whose expansion proves its leaf, backs up the reward of a decided leaf whose
 *     winner is the proven winner (the side that moved into the leaf for WIN, the side to move at it for LOSS) in place of the
 *     evaluator's value; N and W are otherwise backed up as without the switch.
 *   onb_mcts_finish / onb_mcts_play_best: best = the first terminal WIN root child in child order, else the WIN child with the most
 *     visits (last maximal); without WIN children the visit rule over the children without LOSS; if every child is LOSS, the visit
 *     rule over all. pi stays the visit distribution. ONB_BUF_ROOT_PROOF [game] = +1 (the side to move at the root wins: root LOSS),
 *     -1 (it loses: root WIN) or 0.
 * onb_mcts_run with ONB_EVAL_UNIFORM / ONB_EVAL_HASH runs a fused solver kernel (split rounds with tablebase leaves, as §5i), with
 * ONB_EVAL_NET the split phase's solver kernels. Refused with ONB_E_STATE: a begin with the switch on together with train-mode noise,
 * the Gumbel root search, virtual loss or tree reuse; onb_uct_run after such a begin; onb_self_play while the switch is on.
 * onb_fight searches with the solver only for ONB_AGENT_PUCT_SOLVER agents, whatever the switch says, and leaves it as it found it. */
#define ONB_NODE_WIN 8
#define ONB_NODE_LOSS 16
ONB_API int32_t onb_mcts_set_solver(onb_ctx* ctx, int32_t enabled);
/* ONB_AGENT_PUCT_SOLVER: as ONB_AGENT_PUCT (the same fields), searching with the solver and playing the solver's best move. */
#define ONB_AGENT_PUCT_SOLVER 9

/* ---- policy/value network on the device ---------------------------------------------------------------------
 * ConvResNet::forward (alphazero-training/src/net.rs:215-232) for every position of a plane buffer, as one fused
 * tensor-core kernel (BatchNorm in eval mode folded into the convolutions; f32 accumulation; heads in f32). Arithmetic of the
 * convolutions: ONB_NET_F32 reproduces the reference's f32 results (split operands, see below); ONB_NET_F16 (default, the fast
 * mode) and ONB_NET_TF32 round the operands to an 11-bit significand -- TF32 is what libtorch's cuDNN convolutions compute by
 * default on this GPU. f16-based modes reject a network whose folded weights exceed f16's range (ONB_E_INVALID: use TF32). This is the evaluator the search would otherwise get
 * from tch as a black box; with it a whole search needs no host round trip.
 * onb_net_precision selects the operand format used by the NEXT onb_net_load. Two networks can be resident (slots 0 and 1,
 * slot 0 initially): onb_net_select chooses the one that onb_net_load fills and onb_net_forward / ONB_EVAL_NET evaluate, so
 * an arena (evaluator.rs:355-399: the new model against the previous one) alternates between them without re-uploading.
 * onb_net_load takes the parameters under the reference's VarStore names (net.rs:118-213, `|` or `.` separators),
 * e.g. "conv_init_1|weight", "bn1|running_var", "resnet_0|resnet_small_block1|small_block_conv|weight",
 * "policy_conv|bias", "ph_linear2|weight", "vh_linear1|weight": host f32 arrays in libtorch layout (OIHW, [out][in]).
 * The number of residual blocks is taken from the names and hidden_channels from bn1|weight: 64 (ConvResNetConfig of train.rs)
 * or 128, with input_channels 21 -- any other width, or a tensor whose size does not match the width, is rejected with
 * ONB_E_INVALID. The two resident slots may hold networks of different widths.
 * onb_net_forward reads planes_buffer (ONB_BUF_LEAF_PLANES or ONB_BUF_PLANES, [n][21][5][5] f32) and writes
 * ONB_BUF_POLICY [n][2][25] (softmax over 50) and ONB_BUF_VALUE [n]. onb_mcts_eval / onb_mcts_run accept ONB_EVAL_NET. */
#define ONB_NET_F16 0  /* fast mode: operands rounded to f16 (11-bit significand), f32 accumulation */
#define ONB_NET_TF32 1 /* operands rounded to tf32 (11-bit significand, f32 exponent range) */
#define ONB_NET_F32 2  /* f32-faithful: every operand split as x = x1 + 2^-11 x2 (two f16 parts, >= 22 significand bits), three
                          tensor-core products per multiply-accumulate, f32 accumulation: max |dp|, |dv| <= 1e-5 against the f32
                          reference arithmetic of net.rs:215-232 (libtorch on Device::Cpu, train.rs:163-164); ~3x the time of F16 */
ONB_API int32_t onb_net_precision(onb_ctx* ctx, int32_t mode);
ONB_API int32_t onb_net_select(onb_ctx* ctx, int32_t slot);
ONB_API int32_t onb_net_load(onb_ctx* ctx, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel);
ONB_API int32_t onb_net_forward(onb_ctx* ctx, int32_t planes_buffer);

/* ---- device self-tests -------------------------------------------------------------------------------------- */
/* Arithmetic identities the kernels rely on, checked on the device itself. which = ONB_SELFTEST_DIV: the PUCT score
 * (mcts_arena.rs:204-207) divides by visit counts through a reciprocal table; this compares that division with the
 * correctly rounded IEEE quotient over every sqrt(N_parent) / (n + 1) with both below 4096 and over 2^25 pseudo-random
 * W / n. *mismatches receives the number of quotients whose bits differ (0 on a correct build). */
#define ONB_SELFTEST_DIV 0
ONB_API int32_t onb_selftest(onb_ctx* ctx, int32_t which, uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* ONB_H_ */
