// onitama_b200.hpp -- C++17 host-side mirror of the reference's Rust interface for the hot path, header-only, on top of
// the C ABI (onb.h / libonb.so). Same names, argument meaning and error behaviour as the reference so that tests read
// like the reference's own tests (tests/cpp/test_host_mirror.cpp). Every game/search operation executes on the GPU
// through libonb.so; there is no CPU implementation of the rules in this file.
//
//   reference (Rust)                                            here
//   onitama-game/src/game/{player_color,piece,move,done_move,move_result}.rs   PlayerColor, PieceKind, Move, DoneMove, MoveResult
//   onitama-game/src/game/card.rs (ORIGINAL_CARDS, CARD_NAMES)  Card, TIGER..COBRA, CARD_NAMES
//   onitama-game/src/game/deck.rs                               Deck
//   onitama-game/src/game/state.rs                              State
//   onitama-game/src/game/game_state.rs                         GameState
//   onitama-game/src/ai/agent.rs, ai/random.rs                  Agent, Random
//   alphazero-training/src/alphazero_mcts/mod.rs                AlphaZeroMctsConfig, TrainingAlphaZeroMcts, AlphaZeroMcts, reward
//   alphazero-training/src/train.rs:27-98                       SelfPlayData, TrainConfig (self-play fields), self_play
//   alphazero-training/src/evaluator.rs:355-399                 EvaluatorConfig, FightStatistics, fight
//
// Differences that are deliberate: rand::thread_rng is replaced by the counter RNG of onb.h (seeded, reproducible);
// search_time is ignored (no wall-clock cut-off); train-mode root noise is drawn from the counter RNG (statistical parity);
// where the reference panics (expect/unwrap), this header throws onitama::Error.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "onb.h"

namespace onitama {

struct Error : std::runtime_error {
    int32_t code;
    Error(int32_t c, const std::string& m) : std::runtime_error(m), code(c) {}
};

// ---------------------------------------------------------------------------------------------- small value types
enum class PlayerColor : int { Red = 0, Blue = 1 };  // player_color.rs:6-9
inline PlayerColor enemy(PlayerColor c) { return c == PlayerColor::Red ? PlayerColor::Blue : PlayerColor::Red; }
inline void switch_color(PlayerColor& c) { c = enemy(c); }  // PlayerColor::switch

enum class PieceKind : int { Pawn = 0, King = 1 };  // piece.rs:6-9
enum class MoveResult { Capture, RedWin, BlueWin, InProgress };  // move_result.rs:4-9
inline bool is_win(MoveResult r) { return r == MoveResult::RedWin || r == MoveResult::BlueWin; }

struct Move {  // move.rs:21-25 (derived Ord: from, to, piece)
    uint32_t from, to;
    PieceKind piece;
    bool operator==(const Move& o) const { return from == o.from && to == o.to && piece == o.piece; }
    bool operator<(const Move& o) const {
        return std::tie(from, to, piece) < std::tie(o.from, o.to, o.piece);
    }
    static Move from_2d(std::array<std::array<uint32_t, 2>, 2> rc, PieceKind piece) {  // impl From<([(u32,u32);2], PieceKind)>
        return Move{rc[0][0] * 5 + rc[0][1], rc[1][0] * 5 + rc[1][1], piece};
    }
    static std::string convert_idx_to_notation(uint32_t idx) {  // move.rs:35-47
        return std::string(1, "abcde"[idx % 5]) + std::to_string(5 - idx / 5);
    }
};
struct DoneMove {  // done_move.rs:4-7
    Move mov;
    size_t used_card_idx;
    bool operator==(const DoneMove& o) const { return mov == o.mov && used_card_idx == o.used_card_idx; }
};
inline onb_action to_action(const DoneMove& d) {
    return ONB_ACTION((uint32_t)d.used_card_idx, d.mov.from, d.mov.to, (uint32_t)d.mov.piece);
}
inline DoneMove from_action(onb_action a) {
    return DoneMove{Move{(uint32_t)((a >> 5) & 31), (uint32_t)(a & 31), ((a >> 12) & 1) ? PieceKind::King : PieceKind::Pawn}, (size_t)((a >> 10) & 3)};
}

// ---------------------------------------------------------------------------------------------- cards and deck
static const char* const CARD_NAMES[16] = {"Tiger", "Dragon", "Frog", "Rabbit", "Crab", "Elephant", "Goose", "Rooster",
                                           "Monkey", "Mantis", "Crane", "Horse", "Ox", "Boar", "Eel", "Cobra"};  // card.rs:471-474
struct Card {  // card.rs:7-16; the move patterns live in the library's __constant__ table, addressed by `index`
    size_t index;
    PlayerColor player_color() const { return ((0x5551u >> index) & 1u) ? PlayerColor::Blue : PlayerColor::Red; }
    const char* name() const { return CARD_NAMES[index]; }
    bool operator==(const Card& o) const { return index == o.index; }
};
static const Card TIGER{0}, DRAGON{1}, FROG{2}, RABBIT{3}, CRAB{4}, ELEPHANT{5}, GOOSE{6}, ROOSTER{7}, MONKEY{8}, MANTIS{9}, CRANE{10},
    HORSE{11}, OX{12}, BOAR{13}, EEL{14}, COBRA{15};

constexpr size_t RED_CARD1 = 0, RED_CARD2 = 1, BLUE_CARD1 = 2, BLUE_CARD2 = 3, NEUTRAL = 4;  // deck.rs:14-18
struct Deck {
    std::array<Card, 5> cards;
    Deck() : cards{TIGER, DRAGON, FROG, RABBIT, CRAB} {}
    explicit Deck(std::array<Card, 5> c) : cards(c) {}
    std::array<const Card*, 2> get_player_cards(PlayerColor c) const {
        return c == PlayerColor::Red ? std::array<const Card*, 2>{&cards[0], &cards[1]} : std::array<const Card*, 2>{&cards[2], &cards[3]};
    }
    std::array<size_t, 2> get_player_cards_idx(PlayerColor c) const { return c == PlayerColor::Red ? std::array<size_t, 2>{0, 1} : std::array<size_t, 2>{2, 3}; }
    const Card& neutral_card() const { return cards[NEUTRAL]; }
    const Card& get_card(size_t i) const {
        if (i >= 5) throw Error(ONB_E_INVALID, "card_idx < 5");
        return cards[i];
    }
    void rotate(size_t idx) {  // deck.rs:87-90
        if (idx >= 4) throw Error(ONB_E_INVALID, "idx < 4");
        std::swap(cards[idx], cards[NEUTRAL]);
    }
    /// Deck::default (deck.rs:139-151) with the counter RNG instead of thread_rng
    static Deck random(uint64_t seed, uint64_t game, uint32_t epoch = 0) {
        uint8_t d[5];
        onb_deal(seed, game, epoch, d);
        return Deck({Card{d[0]}, Card{d[1]}, Card{d[2]}, Card{d[3]}, Card{d[4]}});
    }
};

// ---------------------------------------------------------------------------------------------- engine (RAII over onb_ctx)
class Engine {
public:
    explicit Engine(int64_t n_games, uint32_t max_sims = 0, uint64_t seed = 0, int device = 0, bool planes = true, uint64_t game_id_base = 0) : n_(n_games) {
        onb_config cfg{};
        cfg.device = device; cfg.n_games = n_games; cfg.seed = seed; cfg.game_id_base = game_id_base;
        cfg.mcts_max_sims = max_sims; cfg.alloc_planes = planes ? 1 : 0;
        int32_t rc = onb_create(&cfg, &ctx_);
        if (rc != ONB_OK) throw Error(rc, onb_last_error(nullptr));
    }
    ~Engine() { if (ctx_) onb_destroy(ctx_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    onb_ctx* ctx() const { return ctx_; }
    int64_t n() const { return n_; }
    /// Hands the network to the library (the VarStore of train.rs as (name, values) pairs, names as in net.rs:118-213 with '|'
    /// or '.' separators); agents with device_evaluator = ONB_EVAL_NET then search without a host evaluator in the loop.
    /// precision: ONB_NET_F32 = the reference's f32 arithmetic (split operands), ONB_NET_F16 = fast mode, ONB_NET_TF32
    void load_network(const std::vector<std::pair<std::string, std::vector<float>>>& var_store, int precision = ONB_NET_F32) {
        std::vector<const char*> names;
        std::vector<const float*> data;
        std::vector<int64_t> numel;
        for (const auto& kv : var_store) {
            names.push_back(kv.first.c_str());
            data.push_back(kv.second.data());
            numel.push_back((int64_t)kv.second.size());
        }
        check(onb_net_precision(ctx_, precision));
        check(onb_net_load(ctx_, (int32_t)names.size(), names.data(), data.data(), numel.data()));
    }
    void check(int32_t rc) const { if (rc != ONB_OK) throw Error(rc, onb_last_error(ctx_)); }
    std::vector<uint8_t> last_fight_results;  ///< per-game MoveResult codes of the last fight_device (0 undecided, 1 RedWin, 2 BlueWin)
    onb_gumbel_config gumbel_applied{};       ///< the Gumbel setting last passed to onb_mcts_set_gumbel (enabled = 0: off)
    std::pair<uint32_t, double> vl_applied{1, 1.0};  ///< (leaves, virtual_loss) last passed to onb_mcts_set_virtual_loss (leaves 1: off)
    bool tb_applied = false;                  ///< the tablebase-leaf switch last passed to onb_mcts_set_tablebase
    bool solver_applied = false;              ///< the MCTS-solver switch last passed to onb_mcts_set_solver
    int32_t tb_max_pawns = -1;                ///< the table resident on this engine (solve_tablebase): max_pawns, -1 none
    std::array<uint8_t, 5> tb_cards{};        ///< ... and its card set as given
    /// onb_tb_solve on this engine's context: the table of one five-card set with at most max_pawns pawns, which tablebase leaves
    /// (AlphaZeroMctsConfig::tablebase_leaves) and ONB_AGENT_PUCT_TB agents in fight_device read. A solve switches tablebase leaves off.
    void solve_tablebase(const std::array<uint8_t, 5>& cards, int32_t max_pawns) {
        tb_max_pawns = -1;
        tb_applied = false;
        check(onb_tb_solve(ctx_, cards.data(), max_pawns, nullptr));
        tb_cards = cards;
        tb_max_pawns = max_pawns;
    }
    /// one-game engine shared by the single-state methods of State / the agents (thread local: a context is single threaded)
    static Engine& single(uint32_t min_sims = 0) {
        thread_local std::unique_ptr<Engine> e;
        thread_local uint32_t sims = 0;
        if (!e || sims < min_sims) { e.reset(); sims = std::max<uint32_t>(min_sims, 64); e = std::make_unique<Engine>(1, sims); }
        return *e;
    }
private:
    onb_ctx* ctx_ = nullptr;
    int64_t n_;
};

// ---------------------------------------------------------------------------------------------- State (state.rs)
constexpr uint32_t RED_KING_SP = 0x00000200u, BLUE_KING_SP = 0x20000000u, BLUE_PAWNS_SP = 0xD8000000u, RED_PAWNS_SP = 0x00000D80u;  // state.rs:24-45
constexpr size_t BLUE_TEMPLE = 2, RED_TEMPLE = 22;                                                                                  // state.rs:48-49
inline uint32_t get_bit(uint32_t x, size_t n) { return (x >> (31 - n)) & 1u; }  // common/mod.rs:2-4
inline uint32_t from_2d_to_bitboard(uint32_t row, uint32_t col) { return 0x80000000u >> (row * 5 + col); }  // common/mod.rs:10-16

struct State {
    Deck deck;
    uint32_t kings[2];
    uint32_t pawns[2];

    static State with_deck(const Deck& deck) {  // state.rs:67-73
        State s;
        s.deck = deck;
        s.kings[0] = RED_KING_SP; s.kings[1] = BLUE_KING_SP;
        s.pawns[0] = RED_PAWNS_SP; s.pawns[1] = BLUE_PAWNS_SP;
        return s;
    }
    onb_state to_onb(PlayerColor side) const {
        onb_state o{};
        o.pawns[0] = pawns[0]; o.pawns[1] = pawns[1]; o.kings[0] = kings[0]; o.kings[1] = kings[1];
        for (int i = 0; i < 5; ++i) o.cards[i] = (uint8_t)deck.cards[i].index;
        o.side = (uint8_t)side;
        return o;
    }
    void from_onb(const onb_state& o) {
        pawns[0] = o.pawns[0]; pawns[1] = o.pawns[1]; kings[0] = o.kings[0]; kings[1] = o.kings[1];
        for (int i = 0; i < 5; ++i) deck.cards[i] = Card{o.cards[i]};
    }
    /// state.rs:75-108: the board as text, row 5 (Blue's home row) first
    std::string display() const {
        const std::string border = "---+---+---+---+---+---+\n";
        std::string r = border;
        for (size_t i = 0; i < 25; ++i) {
            if (i % 5 == 0) r += " " + std::to_string(5 - i / 5) + " ";
            if (get_bit(pawns[0], i)) r += "| r ";
            else if (get_bit(pawns[1], i)) r += "| b ";
            else if (get_bit(kings[0], i)) r += "| R ";
            else if (get_bit(kings[1], i)) r += "| B ";
            else r += "| . ";
            if ((i + 1) % 5 == 0) { r += "|\n"; r += border; }
        }
        return r + "   | a | b | c | d | e |";
    }
    bool is_terminal() const {  // state.rs:111-117
        return kings[0] == 0 || kings[1] == 0 || kings[0] == BLUE_KING_SP || kings[1] == RED_KING_SP;
    }
    MoveResult current_state() const {  // state.rs:120-134
        if (kings[0] == 0 || kings[1] == RED_KING_SP) return MoveResult::BlueWin;
        if (kings[1] == 0 || kings[0] == BLUE_KING_SP) return MoveResult::RedWin;
        return MoveResult::InProgress;
    }
    /// state.rs:301-310, executed by k_legal_moves on the GPU; order = slot, from, to as in the reference
    std::vector<std::pair<size_t, Move>> generate_all_legal_moves(PlayerColor player_color) const {
        Engine& e = Engine::single();
        onb_state o = to_onb(player_color);
        e.check(onb_env_set_states(e.ctx(), &o, 0, 1));
        onb_action moves[40];
        uint8_t count = 0;
        e.check(onb_env_legal_moves(e.ctx(), moves, &count));
        std::vector<std::pair<size_t, Move>> out;
        for (int i = 0; i < count; ++i) { DoneMove d = from_action(moves[i]); out.emplace_back(d.used_card_idx, d.mov); }
        return out;
    }
    /// state.rs:323-378: moves of one card for `player_color` (the card does not have to be in that player's hand)
    std::vector<Move> generate_legal_moves(PlayerColor player_color, const Card& card) const {
        State tmp = *this;
        const size_t slot = player_color == PlayerColor::Red ? RED_CARD1 : BLUE_CARD1;
        tmp.deck.cards[slot] = card;
        std::vector<Move> out;
        for (auto& cm : tmp.generate_all_legal_moves(player_color))
            if (cm.first == slot) out.push_back(cm.second);
        return out;
    }
    std::vector<Move> generate_legal_moves_card_idx(PlayerColor player_color, size_t card_idx) const {
        return generate_legal_moves(player_color, deck.get_card(card_idx));
    }
    /// state.rs:145-202 (no legality check), executed by k_env_step on the GPU
    MoveResult make_move(const Move& mov, PlayerColor player_color, size_t used_card_idx) {
        Engine& e = Engine::single();
        onb_state o = to_onb(player_color);
        const uint32_t enemy_pawns_before = pawns[(int)enemy(player_color)];
        e.check(onb_env_set_states(e.ctx(), &o, 0, 1));
        onb_action a = to_action(DoneMove{mov, used_card_idx});
        e.check(onb_env_step(e.ctx(), &a, 0, 0, 0));
        e.check(onb_env_get_states(e.ctx(), &o, 0, 1));
        from_onb(o);
        if (o.result == ONB_RESULT_RED_WIN) return MoveResult::RedWin;
        if (o.result == ONB_RESULT_BLUE_WIN) return MoveResult::BlueWin;
        return pawns[(int)enemy(player_color)] != enemy_pawns_before ? MoveResult::Capture : MoveResult::InProgress;
    }
    MoveResult pass(size_t card_idx) {  // state.rs:139-142
        deck.rotate(card_idx);
        return MoveResult::InProgress;
    }
};

// ---------------------------------------------------------------------------------------------- GameState (game_state.rs)
struct GameState {
    State state;
    std::vector<State> history;
    size_t curr_agent_idx;
    PlayerColor curr_player_color;

    static GameState with_deck(const Deck& deck) {  // game_state.rs:34-49: first mover = the neutral card's stamp
        GameState g;
        g.state = State::with_deck(deck);
        g.curr_player_color = g.state.deck.neutral_card().player_color();
        g.curr_agent_idx = g.curr_player_color == PlayerColor::Red ? 0 : 1;
        return g;
    }
    MoveResult progress(const DoneMove& done_move) {  // game_state.rs:65-80
        history.push_back(state);
        MoveResult r = state.make_move(done_move.mov, curr_player_color, done_move.used_card_idx);
        curr_agent_idx = (curr_agent_idx + 1) % 2;
        switch_color(curr_player_color);
        return r;
    }
    void undo() {  // game_state.rs:82-89
        if (!history.empty()) { state = history.back(); history.pop_back(); }
        curr_agent_idx = (curr_agent_idx + 1) % 2;
        switch_color(curr_player_color);
    }
};

// ---------------------------------------------------------------------------------------------- agents
struct Agent {  // ai/agent.rs:7-17
    virtual ~Agent() = default;
    virtual std::pair<DoneMove, double> generate_move(const GameState& game_state) = 0;
    virtual const char* name() const = 0;
    virtual std::unique_ptr<Agent> clone_dyn() const = 0;
    virtual uint64_t id() const = 0;
};

/// ai/random.rs:12-43 including its quirks (fabricated a5->a4 pawn move when the drawn card has no move; used_card_idx is
/// the 0/1 slot number even for Blue). Draws come from the counter RNG keyed by (seed, game = 0, step = call number).
struct Random : Agent {
    uint64_t seed;
    uint32_t calls = 0;
    explicit Random(uint64_t seed_ = 0) : seed(seed_) {}
    std::pair<DoneMove, double> generate_move(const GameState& gs) override {
        thread_local std::unique_ptr<Engine> e;
        thread_local uint64_t e_seed = ~0ull;
        if (!e || e_seed != seed) { e = std::make_unique<Engine>(1, 0, seed); e_seed = seed; }
        onb_state o = gs.state.to_onb(gs.curr_player_color);
        e->check(onb_env_set_states(e->ctx(), &o, 0, 1));
        e->check(onb_env_choose_random(e->ctx(), calls++, ONB_POLICY_AGENT));
        onb_action a = 0;
        e->check(onb_read_buffer(e->ctx(), ONB_BUF_ACTIONS, &a, sizeof(a)));
        return {from_action(a), 0.};
    }
    const char* name() const override { return "Random AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<Random>(*this); }
    uint64_t id() const override { return seed; }
};

/// ai/mcts/mod.rs:13-68: plain UCT with random rollouts (mcts_arena.rs). The 1 s wall-clock limit of the reference is not
/// reproduced: a search always runs max_playouts playouts. Rollout draws come from the counter RNG keyed by (seed, game = 0).
struct Mcts : Agent {
    double search_time_ms = 1000.;  // ignored
    uint32_t min_node_visits = 5;
    float exploration_c = 1.41421356f;
    uint32_t max_playouts = 5000;
    uint64_t seed = 0;
    std::pair<DoneMove, double> generate_move(const GameState& gs) override {
        thread_local std::unique_ptr<Engine> e;
        thread_local uint64_t e_seed = ~0ull;
        thread_local uint32_t e_sims = 0;
        if (!e || e_seed != seed || e_sims < max_playouts) { e.reset(); e = std::make_unique<Engine>(1, max_playouts, seed, 0, false); e_seed = seed; e_sims = max_playouts; }
        onb_state o = gs.state.to_onb(gs.curr_player_color);
        e->check(onb_env_set_states(e->ctx(), &o, 0, 1));
        e->check(onb_mcts_begin(e->ctx(), 0., max_playouts));
        e->check(onb_uct_run(e->ctx(), exploration_c, min_node_visits, max_playouts));
        onb_action best = 0;
        uint32_t visits[40], root_visits = 0;
        e->check(onb_mcts_finish(e->ctx(), &best, nullptr, &root_visits, nullptr, visits));
        if (best == ONB_ACTION_NONE) throw Error(ONB_E_STATE, "Must find the best child");  // mcts_arena.rs:67
        // the reference returns the winrate of the chosen child (mcts_arena.rs:78-83)
        const size_t cap = 1 + 40 * (size_t)max_playouts + 2;
        std::vector<uint32_t> v(cap), fc(cap), nc(cap);
        std::vector<double> rew(cap);
        std::vector<uint16_t> act(cap);
        onb_tree_dump d{v.data(), rew.data(), nullptr, act.data(), nullptr, fc.data(), nc.data(), nullptr};
        int64_t n_nodes = 0;
        e->check(onb_mcts_dump_tree(e->ctx(), 0, (int64_t)cap, &d, &n_nodes));
        double winrate = 0.;
        for (uint32_t k = 0; k < nc[0]; ++k)
            if (act[fc[0] + k] == best && v[fc[0] + k]) winrate = (double)((float)rew[fc[0] + k] / (float)v[fc[0] + k]);
        return {from_action(best), winrate};
    }
    const char* name() const override { return "MCTS AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<Mcts>(*this); }
    uint64_t id() const override { return (uint64_t)search_time_ms * 1000000ull + (uint64_t)exploration_c + max_playouts + min_node_visits; }
};

/// ai/alpha_beta/mod.rs: the `AlphaBeta` agent as this project defines it (onb_alphabeta_run, DESIGN.md §5d): a negamax with
/// alpha-beta pruning to a fixed depth in plies, on the GPU. The reference deepens iteratively until a wall-clock limit and scores
/// leaves with its own tables; neither is reproduced, so this agent's play is not pinned to the reference. generate_move returns
/// the chosen move and the root's score (side to move's view; a win in k own moves scores 1 000 000 - (2k - 1)). Like the
/// reference (alpha_beta/mod.rs:165-167) it refuses a position without a legal move, where the search's answer is a pass.
struct AlphaBeta : Agent {
    int32_t depth = 4;
    explicit AlphaBeta(int32_t depth_ = 4) : depth(depth_) {}
    std::pair<DoneMove, double> generate_move(const GameState& gs) override {
        Engine& e = Engine::single();
        onb_state o = gs.state.to_onb(gs.curr_player_color);
        e.check(onb_env_set_states(e.ctx(), &o, 0, 1));
        onb_action best = 0;
        int32_t score = 0;
        e.check(onb_alphabeta_run(e.ctx(), depth, &best, &score, nullptr));
        if (best == ONB_ACTION_NONE) throw Error(ONB_E_STATE, "AlphaBeta: the game is already decided");
        if (best & (1u << 13)) throw Error(ONB_E_STATE, "AlphaBeta: no legal move (the search would pass)");
        return {from_action(best), (double)score};
    }
    const char* name() const override { return "AlphaBeta AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<AlphaBeta>(*this); }
    uint64_t id() const override { return (uint64_t)depth; }
};

/// The perfect endgame agent (onb_tb_solve / onb_tb_best, DESIGN.md §5g): plays the tablebase's move for one five-card set with at
/// most max_pawns pawns. The table is solved on first use on a one-game context of the agent's own (copies share it). generate_move
/// returns the move and the position's value (+n: win in n plies, -n: loss in n plies, 0: draw); it refuses a decided position and
/// one outside the table. A position without a legal move is answered with a pass, which DoneMove cannot carry: refused as well.
struct Tablebase : Agent {
    std::array<uint8_t, 5> cards;
    int32_t max_pawns = 3;
    explicit Tablebase(std::array<uint8_t, 5> cards_, int32_t max_pawns_ = 3) : cards(cards_), max_pawns(max_pawns_) {}
    std::pair<DoneMove, double> generate_move(const GameState& gs) override {
        if (!engine) {
            auto e = std::make_shared<Engine>(1, 0, 0, 0, false);
            e->check(onb_tb_solve(e->ctx(), cards.data(), max_pawns, nullptr));
            engine = e;
        }
        onb_state o = gs.state.to_onb(gs.curr_player_color);
        engine->check(onb_env_set_states(engine->ctx(), &o, 0, 1));
        int16_t value = 0;
        onb_action best = 0;
        engine->check(onb_tb_probe(engine->ctx(), &value));
        engine->check(onb_tb_best(engine->ctx(), &best));
        if (best == ONB_ACTION_NONE) throw Error(ONB_E_STATE, "Tablebase: the game is decided or not a position of the table");
        if (best & (1u << 13)) throw Error(ONB_E_STATE, "Tablebase: no legal move (the table's answer is a pass)");
        return {from_action(best), (double)value};
    }
    const char* name() const override { return "Tablebase AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<Tablebase>(*this); }
    uint64_t id() const override { return (uint64_t)max_pawns; }
private:
    std::shared_ptr<Engine> engine;
};

struct AlphaZeroMctsConfig {  // alphazero_mcts/mod.rs:26-43
    double search_time_ms = 400.;  // ignored: the search always runs max_playouts simulations
    double exploration_c = 1.4142135623730951;
    uint32_t max_playouts = 5000;
    bool train = false;  // root exploration noise, epsilon 0.25 / Dirichlet alpha 0.03 (mcts_arena.rs:186-202)
    uint64_t noise_seed = 0;
    // keep the played child's subtree between moves (onb_mcts_set_reuse): max_playouts then counts root visits, kept ones
    // included. Device evaluators only; false forgets the remembered trees.
    bool reuse = false;
    // the Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f): enabled = 1 makes every search select at the root by sequential
    // halving and report the improved policy as the move's tensor. The setting is applied when it changes (which sets the step to
    // step0); every search takes the next step. Does not combine with train or reuse (ONB_E_STATE). interior = 1: Gumbel MuZero's
    // interior selection below the root instead of PUCT.
    onb_gumbel_config gumbel{};
    // leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h): leaves_per_round >= 2 runs every search in rounds
    // of that many descents (round 0: one), each pending descent counting as a lost visit of virtual_loss; a HostEvaluator then
    // evaluates n * leaves_per_round rows per round. Applied when it changes. Does not combine with train, reuse or gumbel (ONB_E_STATE).
    uint32_t leaves_per_round = 1;
    double virtual_loss = 1.0;
    // tablebase leaves (onb_mcts_set_tablebase, DESIGN.md §5i): the search's engine holds the table of tablebase_cards with at most
    // tablebase_max_pawns pawns (solved on first use and whenever these change) and every search probes it at its leaves: a leaf below
    // the root that the table holds is not expanded and backs up the table's exact value. Does not combine with reuse (ONB_E_STATE).
    // With a device evaluator the search runs one select, evaluation and expand/backup launch per simulation instead of the fused
    // kernel (DESIGN.md §5i gives the cost).
    bool tablebase_leaves = false;
    std::array<uint8_t, 5> tablebase_cards{};
    int32_t tablebase_max_pawns = 3;
    // the MCTS solver (onb_mcts_set_solver, DESIGN.md §5k): every search proves wins and losses, propagates them to the root and
    // plays a proven win (the first terminal winning child, else the most visited proven win, else the visit rule over the children
    // not proven lost). Applied when it changes. Does not combine with train, reuse, gumbel or leaves_per_round >= 2 (ONB_E_STATE).
    bool solver = false;
};
inline double reward(MoveResult r, PlayerColor c) {  // alphazero_mcts/mod.rs:45-53
    if (c == PlayerColor::Red) return r == MoveResult::RedWin ? 1. : r == MoveResult::BlueWin ? -1. : 0.;
    return r == MoveResult::RedWin ? -1. : r == MoveResult::BlueWin ? 1. : 0.;
}

/// The policy/value network as a black box on host memory: planes [n][21][5][5] -> policy [n][2][25], value [n]
/// (ConvResNet::forward, net.rs:215-232). nullptr selects a device evaluator (ONB_EVAL_*).
using HostEvaluator = std::function<void(const float* planes, int64_t n, float* policy, float* value)>;

namespace detail {
inline void run_search(Engine& e, const AlphaZeroMctsConfig& cfg, int32_t device_eval, const HostEvaluator& net) {
    e.check(onb_mcts_set_noise(e.ctx(), cfg.train ? 1 : 0, 0.25, 0.03, cfg.noise_seed));
    if (cfg.reuse && net) throw Error(ONB_E_INVALID, "AlphaZeroMctsConfig::reuse needs a device evaluator");
    e.check(onb_mcts_set_reuse(e.ctx(), cfg.reuse ? 1 : 0));
    const onb_gumbel_config& g = cfg.gumbel;
    const onb_gumbel_config& a = e.gumbel_applied;
    if (g.enabled != a.enabled || (g.enabled && (g.max_considered != a.max_considered || g.c_visit != a.c_visit || g.c_scale != a.c_scale ||
                                                 g.gumbel_scale != a.gumbel_scale || g.seed != a.seed || g.step0 != a.step0 ||
                                                 g.interior != a.interior))) {
        e.check(onb_mcts_set_gumbel(e.ctx(), &g));
        e.gumbel_applied = g;
    }
    const uint32_t k = cfg.leaves_per_round > 1 ? cfg.leaves_per_round : 1u;
    const std::pair<uint32_t, double> vl{k, k > 1 ? cfg.virtual_loss : 1.0};
    if (vl != e.vl_applied) {
        e.check(onb_mcts_set_virtual_loss(e.ctx(), vl.first, vl.second));
        e.vl_applied = vl;
    }
    if (cfg.tablebase_leaves && (e.tb_max_pawns != cfg.tablebase_max_pawns || e.tb_cards != cfg.tablebase_cards))
        e.solve_tablebase(cfg.tablebase_cards, cfg.tablebase_max_pawns);
    if (cfg.tablebase_leaves != e.tb_applied) {
        e.check(onb_mcts_set_tablebase(e.ctx(), cfg.tablebase_leaves ? 1 : 0));
        e.tb_applied = cfg.tablebase_leaves;
    }
    if (cfg.solver != e.solver_applied) {
        e.check(onb_mcts_set_solver(e.ctx(), cfg.solver ? 1 : 0));
        e.solver_applied = cfg.solver;
    }
    e.check(onb_mcts_begin(e.ctx(), cfg.exploration_c, cfg.max_playouts));
    if (!net) {
        e.check(onb_mcts_run(e.ctx(), device_eval, cfg.max_playouts));
    } else {
        // rounds of one select / evaluation / expand-backup: sims of them, or 1 + ceil((sims - 1) / K) over n K rows with virtual loss
        const int64_t rows = e.n() * k;
        const uint32_t s = cfg.max_playouts, rounds = k > 1 && s ? 1u + (s - 1u + k - 1u) / k : s;
        std::vector<float> planes((size_t)rows * 525), pol((size_t)rows * 50), val((size_t)rows);
        for (uint32_t r = 0; r < rounds; ++r) {
            e.check(onb_mcts_select(e.ctx()));
            e.check(onb_read_buffer(e.ctx(), k > 1 ? ONB_BUF_VL_PLANES : ONB_BUF_LEAF_PLANES, planes.data(), rows * 2100));
            net(planes.data(), rows, pol.data(), val.data());
            e.check(onb_write_buffer(e.ctx(), k > 1 ? ONB_BUF_VL_POLICY : ONB_BUF_POLICY, pol.data(), rows * 200));
            e.check(onb_write_buffer(e.ctx(), k > 1 ? ONB_BUF_VL_VALUE : ONB_BUF_VALUE, val.data(), rows * 4));
            e.check(onb_mcts_expand_backup(e.ctx()));
        }
    }
}
}  // namespace detail

struct TrainingAlphaZeroMcts {  // alphazero_mcts/mod.rs:55-79
    AlphaZeroMctsConfig config;
    int32_t device_evaluator = ONB_EVAL_UNIFORM;
    HostEvaluator model;  // optional host network
    /// generate_move_tensor(&State, PlayerColor) -> (DoneMove, Tensor[2,25])
    std::pair<DoneMove, std::array<float, 50>> generate_move_tensor(const State& state, PlayerColor curr_player_color) const {
        Engine& e = Engine::single(config.max_playouts);
        onb_state o = state.to_onb(curr_player_color);
        e.check(onb_env_set_states(e.ctx(), &o, 0, 1));
        detail::run_search(e, config, device_evaluator, model);
        onb_action best = 0;
        std::array<float, 50> pi{};
        e.check(onb_mcts_finish(e.ctx(), &best, pi.data(), nullptr, nullptr, nullptr));
        if (best == ONB_ACTION_NONE) throw Error(ONB_E_STATE, "Must find the best child");  // mcts_arena.rs:94
        return {from_action(best), pi};
    }
};

struct AlphaZeroMcts : Agent {  // alphazero_mcts/mod.rs:81-161
    AlphaZeroMctsConfig config;
    int32_t device_evaluator = ONB_EVAL_UNIFORM;
    HostEvaluator model;
    std::pair<DoneMove, double> generate_move(const GameState& gs) override {
        TrainingAlphaZeroMcts t{config, device_evaluator, model};
        auto r = t.generate_move_tensor(gs.state, gs.curr_player_color);
        // the reference reports the network's value of the root position (mod.rs:136-142): one extra evaluation of the root (with
        // virtual loss on, round 0's single descent: row 0 of the VL rows)
        Engine& e = Engine::single(config.max_playouts);
        const bool vl = config.leaves_per_round > 1;
        double value = 0.;
        e.check(onb_mcts_begin(e.ctx(), config.exploration_c, config.max_playouts));
        e.check(onb_mcts_select(e.ctx()));
        float v = 0.f;
        if (model) {
            std::vector<float> planes(525), pol(50);
            e.check(onb_read_buffer(e.ctx(), vl ? ONB_BUF_VL_PLANES : ONB_BUF_LEAF_PLANES, planes.data(), 2100));
            model(planes.data(), 1, pol.data(), &v);
        } else {
            e.check(onb_mcts_eval(e.ctx(), device_evaluator));
            e.check(onb_read_buffer(e.ctx(), vl ? ONB_BUF_VL_VALUE : ONB_BUF_VALUE, &v, 4));
        }
        value = (double)v;
        return {r.first, value};
    }
    const char* name() const override { return "AlphaZero MCTS AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<AlphaZeroMcts>(*this); }
    uint64_t id() const override { return (uint64_t)config.exploration_c + config.max_playouts + (uint64_t)config.train; }
};

/// Gumbel MuZero (onb_gumbel_config.interior = 1, DESIGN.md §5f): AlphaZeroMcts with the Gumbel root search over m considered actions
/// and interior selection below the root (c_visit 50, gumbel_scale 1). The project's own agent; the reference has none.
struct GumbelMuZero : AlphaZeroMcts {
    explicit GumbelMuZero(uint32_t m = 16, double c_scale = 0.1, uint64_t seed = 0) {
        config.gumbel.enabled = 1;
        config.gumbel.max_considered = m;
        config.gumbel.c_visit = 50.0;
        config.gumbel.c_scale = c_scale;
        config.gumbel.gumbel_scale = 1.0;
        config.gumbel.seed = seed;
        config.gumbel.interior = 1;
    }
    const char* name() const override { return "Gumbel MuZero AI"; }
    std::unique_ptr<Agent> clone_dyn() const override { return std::make_unique<GumbelMuZero>(*this); }
};

// ---------------------------------------------------------------------------------------------- self_play (train.rs:27-98)
struct SelfPlayData {
    std::array<float, 50> pi;      // [2,25]
    float z;
    std::array<float, 525> state;  // [21,5,5]
    PlayerColor player_color;
};
struct TrainConfig {  // the self-play fields of train.rs:100-154
    AlphaZeroMctsConfig mcts_config;
    size_t self_play_game_amnt = 100;
    long max_plies = 150;
    std::optional<Deck> deck;
    uint64_t seed = 0;
    // AlphaZero's self-play move protocol (onb_self_play_set_protocol, DESIGN.md §5j; self_play_continuous only, the project's own
    // setting: the reference plays the best move and never resigns). The first temp_plies plies of a game sample their move in
    // proportion to N^(1/temperature); with resign_below set, the side to move resigns when max(v_root, q_best) < *resign_below,
    // except in a resign_holdout fraction of games. Draws are keyed by `seed`.
    uint32_t temp_plies = 0;
    double temperature = 1.0;
    std::optional<double> resign_below;
    double resign_holdout = 0.1;
};
/// All `self_play_game_amnt` games are played in lockstep on one engine (the reference plays them one after another on one
/// thread); samples are returned game-major, ply-minor like the reference's play_buffer.
inline std::vector<SelfPlayData> self_play(const TrainingAlphaZeroMcts& mcts, const TrainConfig& config) {
    const int64_t n = (int64_t)config.self_play_game_amnt;
    Engine e(n, mcts.config.max_playouts, config.seed);
    if (config.deck) {
        uint8_t d[5];
        for (int i = 0; i < 5; ++i) d[i] = (uint8_t)config.deck->cards[i].index;
        e.check(onb_env_reset(e.ctx(), d, 1, 0));
    } else {
        e.check(onb_env_reset(e.ctx(), nullptr, 0, 0));  // State::new(): random deal
    }
    std::vector<std::vector<SelfPlayData>> per_game((size_t)n);
    std::vector<onb_state> st((size_t)n);
    std::vector<float> planes((size_t)n * 525), pi((size_t)n * 50);
    long max_plies = config.max_plies;
    for (;;) {
        e.check(onb_env_get_states(e.ctx(), st.data(), 0, n));
        bool any = false;
        for (auto& s : st) any |= s.result == 0;
        if (!any) break;
        e.check(onb_env_encode(e.ctx(), planes.data()));
        detail::run_search(e, mcts.config, mcts.device_evaluator, mcts.model);
        e.check(onb_mcts_finish(e.ctx(), nullptr, pi.data(), nullptr, nullptr, nullptr));
        for (int64_t g = 0; g < n; ++g) {
            if (st[(size_t)g].result != 0) continue;
            SelfPlayData d;
            std::memcpy(d.pi.data(), &pi[(size_t)g * 50], 200);
            std::memcpy(d.state.data(), &planes[(size_t)g * 525], 2100);
            d.z = 0.f;
            d.player_color = (PlayerColor)st[(size_t)g].side;
            per_game[(size_t)g].push_back(d);
        }
        e.check(onb_mcts_play_best(e.ctx(), 0));
        if (max_plies < 0) break;  // train.rs:74-79 (check, then decrement: max_plies + 2 plies in total)
        max_plies -= 1;
    }
    e.check(onb_env_get_states(e.ctx(), st.data(), 0, n));
    std::vector<SelfPlayData> out;
    for (int64_t g = 0; g < n; ++g) {
        const uint8_t r = st[(size_t)g].result;
        const MoveResult progress = r == 1 ? MoveResult::RedWin : r == 2 ? MoveResult::BlueWin : MoveResult::InProgress;
        for (auto& d : per_game[(size_t)g]) { d.z = (float)reward(progress, d.player_color); out.push_back(d); }  // train.rs:83-85
    }
    return out;
}

/// self_play for a training run: `slots` games in flight on one engine; a slot starts its next game the moment one is over while
/// games remain to be started, and EVERY started game is played to its end: exactly max(config.self_play_game_amnt, slots) complete
/// games come back (onb_self_play: the loop runs inside the library, the samples are copied to the host once at the end). Needs a
/// device evaluator: mcts.device_evaluator = ONB_EVAL_NET after Engine::load_network, or ONB_EVAL_UNIFORM / ONB_EVAL_HASH. Samples
/// come ply-major. The move protocol of config (temp_plies, temperature, resign_below, resign_holdout; all default: off) becomes the
/// engine's setting: it replaces whatever protocol the caller set on e through onb_self_play_set_protocol and stays in force for
/// later onb_self_play calls on e (the C ABI has no getter to restore an earlier setting from; TrainConfig is the source of truth).
inline std::vector<SelfPlayData> self_play_continuous(Engine& e, const TrainingAlphaZeroMcts& mcts, const TrainConfig& config) {
    if (mcts.model) throw Error(ONB_E_INVALID, "self_play_continuous: a host evaluator cannot run inside the library; load the network instead");
    onb_selfplay_protocol proto{};
    proto.temp_plies = config.temp_plies;
    proto.temperature = config.temperature;
    proto.resign = config.resign_below ? 1u : 0u;
    proto.resign_below = config.resign_below.value_or(0.0);
    proto.resign_holdout = config.resign_holdout;
    proto.seed = config.seed;
    e.check(onb_self_play_set_protocol(e.ctx(), &proto));
    onb_selfplay_config cfg{};
    cfg.c_puct = mcts.config.exploration_c; cfg.sims = mcts.config.max_playouts; cfg.evaluator = mcts.device_evaluator;
    cfg.n_games = (int64_t)config.self_play_game_amnt; cfg.max_plies = (uint32_t)config.max_plies; cfg.train = mcts.config.train ? 1 : 0;
    cfg.noise_seed = mcts.config.noise_seed;
    const int64_t generations = 2 + 2 * ((int64_t)config.self_play_game_amnt + e.n() - 1) / e.n();
    cfg.sample_cap = e.n() * (config.max_plies + 2) * generations;
    onb_selfplay_result r{};
    e.check(onb_self_play(e.ctx(), &cfg, &r));
    std::vector<int64_t> idx((size_t)r.n_valid);
    std::vector<float> planes((size_t)r.n_samples * 525), pi((size_t)r.n_samples * 50), z((size_t)r.n_samples);
    std::vector<uint8_t> color((size_t)r.n_samples);
    e.check(onb_sync(e.ctx()));
    if (r.n_samples) {
        if (!idx.empty()) e.check(onb_copy_to_host(e.ctx(), idx.data(), r.valid_idx, (int64_t)idx.size() * 8));
        e.check(onb_copy_to_host(e.ctx(), planes.data(), r.planes, (int64_t)planes.size() * 4));
        e.check(onb_copy_to_host(e.ctx(), pi.data(), r.pi, (int64_t)pi.size() * 4));
        e.check(onb_copy_to_host(e.ctx(), z.data(), r.z, (int64_t)z.size() * 4));
        e.check(onb_copy_to_host(e.ctx(), color.data(), r.color, (int64_t)color.size()));
    }
    std::vector<SelfPlayData> out;
    out.reserve(idx.size());
    for (int64_t i : idx) {
        SelfPlayData d;
        std::memcpy(d.pi.data(), &pi[(size_t)i * 50], 200);
        std::memcpy(d.state.data(), &planes[(size_t)i * 525], 2100);
        d.z = z[(size_t)i];
        d.player_color = (PlayerColor)color[(size_t)i];
        out.push_back(d);
    }
    return out;
}

// ---------------------------------------------------------------------------------------------- fight (evaluator.rs:355-399)
struct EvaluatorConfig {
    size_t game_amnt = 20;
    long max_plies = 150;
    std::optional<Deck> deck;
    uint64_t seed = 0;
};
/// EloRating::elo_change (elo_rating.rs:53-70): K = 32, scale 1/400
struct EloRating {
    static std::pair<double, double> elo_change(double ra, double rb, bool is_a_win) {
        const double ea = 1. / (1. + std::pow(10.0, 2.5e-3 * (rb - ra))), eb = 1. / (1. + std::pow(10.0, 2.5e-3 * (ra - rb)));
        const double sa = is_a_win ? 1. : 0., sb = 1. - sa;
        return {ra + 32. * (sa - ea), rb + 32. * (sb - eb)};
    }
};
struct RatingChange {
    double before_a, after_a, before_b, after_b;
};
struct FightStatistics {  // evaluator.rs:38-110: W/L/D in total and per colour of the agent, win rates, sequential Elo updates
    size_t wins = 0, losses = 0, draws = 0, wins_red = 0, wins_blue = 0, games_red = 0, games_blue = 0;
    double winrate = 0., color_winrate[2] = {0., 0.};
    double rating_a = 800., rating_b = 800.;  // Rating::default (elo_rating.rs:17-21)
    std::vector<RatingChange> rating_change_history;
    FightStatistics() = default;
    FightStatistics(double ra, double rb) : rating_a(ra), rating_b(rb) {}
    void update(MoveResult progress, PlayerColor agent_color) {
        (agent_color == PlayerColor::Red ? games_red : games_blue) += 1;
        const double ba = rating_a, bb = rating_b;
        if (!is_win(progress)) {
            draws += 1;
        } else {
            const bool agent_won = (progress == MoveResult::RedWin) == (agent_color == PlayerColor::Red);
            std::tie(rating_a, rating_b) = EloRating::elo_change(rating_a, rating_b, agent_won);
            if (agent_won) { wins += 1; (agent_color == PlayerColor::Red ? wins_red : wins_blue) += 1; }
            else losses += 1;
        }
        rating_change_history.push_back({ba, rating_a, bb, rating_b});
        winrate = (double)wins / (double)(wins + losses + draws);
        color_winrate[0] = (double)wins_red / (double)games_red;
        color_winrate[1] = (double)wins_blue / (double)games_blue;
    }
};
inline FightStatistics fight(const EvaluatorConfig& config, std::unique_ptr<Agent> agent, std::unique_ptr<Agent> opponent) {
    std::array<std::unique_ptr<Agent>, 2> agents{std::move(agent), std::move(opponent)};
    PlayerColor agent_color = PlayerColor::Red;
    FightStatistics statistics;
    for (size_t game = 0; game < config.game_amnt; ++game) {
        Deck deck = config.deck ? *config.deck : Deck::random(config.seed, game);
        GameState state = GameState::with_deck(deck);
        MoveResult progress = MoveResult::InProgress;
        long max_plies = config.max_plies;
        while (!is_win(progress)) {
            auto mv = agents[state.curr_agent_idx]->generate_move(state);
            progress = state.progress(mv.first);
            if (max_plies < 0) break;
            max_plies -= 1;
        }
        statistics.update(progress, agent_color);
        switch_color(agent_color);
        std::swap(agents[0], agents[1]);
    }
    return statistics;
}

/// fight() for config.game_amnt games at once on one engine (onb_fight: the arena loop runs inside the library; each ply an agent
/// searches only the games in which it is to move). Agent A plays Red in games 0, 2, 4, ... like the colour swap of
/// evaluator.rs:393-397; the statistics incl. the Elo updates are folded in game order ON THE DEVICE (onb_fight_stats).
/// Agents are described by onb_agent (ONB_AGENT_RANDOM / ONB_AGENT_PUCT / ONB_AGENT_UCT / ONB_AGENT_ALPHABETA with the depth in
/// sims); the engine must have been created with n_games == config.game_amnt and enough mcts_max_sims for the searching agents.
/// ONB_AGENT_PUCT_TB (PUCT with tablebase leaves that plays the table's move in the games of the table, DESIGN.md §5i) and
/// ONB_AGENT_TABLEBASE read the table solved on the engine (Engine::solve_tablebase); without one onb_fight refuses them (ONB_E_STATE).
/// puct_tablebase_agent builds the former.
inline onb_agent puct_tablebase_agent(uint32_t sims, double c_puct = 2.0, int32_t evaluator = ONB_EVAL_UNIFORM, int32_t net_slot = 0) {
    onb_agent a{};
    a.kind = ONB_AGENT_PUCT_TB;
    a.evaluator = evaluator;
    a.net_slot = net_slot;
    a.sims = sims;
    a.c = c_puct;
    return a;
}
/// ONB_AGENT_PUCT_SOLVER: PUCT with the MCTS solver (DESIGN.md §5k), playing the solver's best move. onb_fight searches with the
/// solver for this agent only and leaves the engine's switch (AlphaZeroMctsConfig::solver) as it found it.
inline onb_agent puct_solver_agent(uint32_t sims, double c_puct = 2.0, int32_t evaluator = ONB_EVAL_UNIFORM, int32_t net_slot = 0) {
    onb_agent a{};
    a.kind = ONB_AGENT_PUCT_SOLVER;
    a.evaluator = evaluator;
    a.net_slot = net_slot;
    a.sims = sims;
    a.c = c_puct;
    return a;
}
inline FightStatistics fight_device(Engine& e, const EvaluatorConfig& config, const onb_agent& agent, const onb_agent& opponent, double rating_a = 800.,
                                    double rating_b = 800.) {
    if ((size_t)e.n() != config.game_amnt) throw Error(ONB_E_INVALID, "fight_device: the engine must hold game_amnt games");
    if (config.deck) {
        uint8_t d[5];
        for (int i = 0; i < 5; ++i) d[i] = (uint8_t)config.deck->cards[i].index;
        e.check(onb_env_reset(e.ctx(), d, 1, 0));
    } else {
        e.check(onb_env_reset(e.ctx(), nullptr, 0, 0));
    }
    std::vector<uint8_t> a_is_red(config.game_amnt), results(config.game_amnt);
    for (size_t g = 0; g < config.game_amnt; ++g) a_is_red[g] = g % 2 == 0;
    onb_fight_result r{};
    e.check(onb_fight(e.ctx(), &agent, &opponent, a_is_red.data(), (uint32_t)config.max_plies, &r, results.data()));
    onb_fight_statistics st{};
    std::vector<double> history(config.game_amnt * 4);
    e.check(onb_fight_stats(e.ctx(), rating_a, rating_b, &st, history.data()));
    FightStatistics statistics(rating_a, rating_b);
    statistics.wins = (size_t)st.wins; statistics.losses = (size_t)st.loses; statistics.draws = (size_t)st.draws;
    statistics.wins_red = (size_t)st.color_wins[0]; statistics.wins_blue = (size_t)st.color_wins[1];
    statistics.games_red = (size_t)(st.color_wins[0] + st.color_loses[0] + st.color_draws[0]);
    statistics.games_blue = (size_t)(st.color_wins[1] + st.color_loses[1] + st.color_draws[1]);
    statistics.winrate = st.winrate; statistics.color_winrate[0] = st.color_winrate[0]; statistics.color_winrate[1] = st.color_winrate[1];
    statistics.rating_a = st.rating_a; statistics.rating_b = st.rating_b;
    for (size_t g = 0; g < config.game_amnt; ++g)
        statistics.rating_change_history.push_back({history[4 * g], history[4 * g + 1], history[4 * g + 2], history[4 * g + 3]});
    e.last_fight_results = results;
    return statistics;
}

}  // namespace onitama
