/* sb_b200.h -- C ABI of libsb_b200.so, the B200 (sm_100a) batched Stormbound simulator.
 *
 * The reference has no FFI: its boundary is three Python class contracts (SURVEY.md 8b).  Every entry
 * point below names the reference interface it replaces; the Python shims in monsoon_b200/ (Game,
 * StormboundAdapter, HeuristicAgent, FitnessEvaluator) bind these with ctypes and keep the reference's
 * signatures.  INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions: plain C types only; every `*_d` pointer is a DEVICE pointer owned by the caller (e.g.
 * torch tensor .data_ptr()); `stream` is a cudaStream_t passed as void* (NULL = default stream); calls
 * are asynchronous on that stream unless named *_host; return 0 on success, a negative CUDA error
 * code otherwise (sb_last_error gives the text); no hidden allocation after sb_create except the
 * *_host helpers' staging buffers; one handle per device, not thread-safe.
 * There is NO CPU fallback: without a CUDA device sb_create fails.
 */
#ifndef SB_B200_H
#define SB_B200_H
#include <stddef.h>
#include <stdint.h>
#include "sb_state.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct SbHandle SbHandle;

/* library / layout introspection (no GPU needed) */
int sb_abi_version(void);
int sb_state_bytes(void);                 /* == SB_STATE_BYTES */
int sb_card_count(void);                  /* rows of the card table (130) */
int sb_card_info(int card, int32_t out[12]); /* kind,faction,cost,strength,movement,trigger,fixed,has_ability,first_type,types,obs_id,has_target */

/* One handle per device and per stream of use: the handle owns small device scratch (refill counter, staged archetypes,
 * host-variant staging buffer), so two calls through the SAME handle must not run concurrently on different streams. */
int sb_create(int device, SbHandle **out);
int sb_destroy(SbHandle *h);
const char *sb_last_error(SbHandle *h);
int sb_device(SbHandle *h);
int sb_sm_count(SbHandle *h);
/* tuning knobs for the rollout kernels (all default to "auto by batch size"): "games_per_warp" = 0 (auto) or
 * 1..32 consecutive lanes of every warp that carry a game; "turn_sync" 0/1; "block_sync" = -1 auto, 0, or the
 * CTA size (128..1024) whose warps change phase together; "refill" = -1 auto, 0/1: finished lanes of the random
 * rollout take the next game from a counter ("refill_ctas" persistent CTAs per SM, "refill_grid" CTAs in total,
 * 0 = auto); "dense" = -1 auto, 0/1: the 32-register builds with 2,048 resident lanes per SM (random rollout, k_step);
 * "heur_wpc" = -1 / 4: independent warps (default), 8 / 16 / 32: warps per CTA deciding in step; "heur_refill" = -1 auto
 * (batches beyond one wave of resident warps), 0/1: a warp of the heuristic rollout whose game ended takes the next game
 * from a counter; "heur_iw" = -1 auto, 4 / 8 / 16 independent warps per CTA; "heur_grid" = persistent CTAs of that shape
 * (0 = one wave; tests use tiny grids); "lanes_per_game" is accepted and ignored (retired shape).
 * Round 2: "engine" = -1 auto (measured per-kernel policy), 0 thread-per-game kernels, 1 warp-per-game kernels; "w_shape" /
 * "w_hshape" / "w_grid" = CTA shape and persistent grid of the warp-per-game rollouts (-1 / 0 = auto); "heur_pack" = -1 auto
 * (= 1), 0 the round-1 heuristic rollout, 1 one game per warp in the owner / holder structure, 2 / 3 / 4 / 8 several games per
 * warp (candidates of K games dealt to the 32 lanes), 5 / 6 / 7 other CTA shapes of K = 1.  Every setting gives identical results. */
int sb_set_option(SbHandle *h, const char *key, int value);
/* kernels launched through this handle so far (bench.py's gpu_launches) */
uint64_t sb_launch_count(SbHandle *h);

/* Stormbound.__init__ + Player.__init__ + Board.__init__ (games/stormbound.py:293-304, player.py:13-37,
 * board.py:16-28): shuffle both 12-card decks, weights, draw 4, base 20, mana 3/4.
 * decks_d: u8[n,2,n_deck] card indices, or u8[2,n_deck] when decks_shared; factions_d: u8[n,2] or u8[2]. */
int sb_reset(SbHandle *h, int n, const uint64_t *seeds_d, const uint8_t *decks_d, int n_deck, int decks_shared,
             const uint8_t *factions_d, uint8_t *states_d, void *stream);

/* Stormbound.legal_actions (games/stormbound.py:528-557) -> 156-bit mask per game, u32[n,5] */
int sb_legal_mask(SbHandle *h, int n, const uint8_t *states_d, uint32_t *masks_d, void *stream);

/* Stormbound.step (games/stormbound.py:318-373): apply actions_d[n]; reward {0,1} (Game.step multiplies
 * by 10, :140), done, err (non-zero = the reference raises here); next_masks_d (nullable) = legal set
 * of the resulting state, fused into the same pass. */
int sb_step(SbHandle *h, int n, uint8_t *states_d, const uint8_t *actions_d, int8_t *reward_d, uint8_t *done_d,
            uint8_t *err_d, uint32_t *next_masks_d, void *stream);

/* Stormbound.get_observation (games/stormbound.py:400-526): i32[n,27,5,4] */
int sb_observe(SbHandle *h, int n, const uint8_t *states_d, int32_t *obs_d, uint8_t *err_d, void *stream);

/* StateFeatures(obs).get_feature_vector() (evo/features.py:12-342): f64[n,10] */
int sb_features(SbHandle *h, int n, const uint8_t *states_d, double *feat_d, uint8_t *err_d, void *stream);

/* HeuristicAgent.select_action / score_action (evo/heuristic_agent.py:23-80) on StormboundAdapter forks
 * (evo/game_adapter.py:280-324): weights_d f64[n,10]; actions_d u8[n]; scores_d (nullable) f64[n,156],
 * NaN for illegal actions.  One warp per game, one lane per candidate action. */
int sb_select_action(SbHandle *h, int n, const uint8_t *states_d, const double *weights_d, uint8_t *actions_d,
                     double *scores_d, void *stream);

/* DeckEvolutionConfig.get_deck_configuration / generate_random_deck (utils.py:26-119,121-241) for n games: game g
 * draws from philox(counter=(draw, generation, 0xDEC4, 0), key=seeds_d[g]) with CPython's random.sample call
 * shape.  mode 0 exploit (archetypes verbatim), 1 explore (n_preserve = min(int(12*preserve_ratio), 12) cards
 * sampled from the archetype, the rest from own faction + NEUTRAL), 2 balance (random() < q keeps the archetype,
 * drawn for both seats first), 3 fully random decks for per-game factions_d u8[n,2] (BASELINE config 5).
 * archetypes u8[2][12] card ids and arch_factions u8[2] are HOST pointers (the config object's fields);
 * factions_d nullable (= arch_factions for every game); decks_d u8[n,2,12]; factions_out_d nullable u8[n,2].
 * The outputs feed sb_reset(decks_d, 12, 0, factions). */
int sb_generate_decks(SbHandle *h, int n, const uint64_t *seeds_d, uint32_t generation, int mode, int n_preserve, double q,
                      const uint8_t *archetypes, const uint8_t *arch_factions, const uint8_t *factions_d, uint8_t *decks_d,
                      uint8_t *factions_out_d, void *stream);

/* ---- (mu + lambda) evolution-strategy operators on a device-resident population (SURVEY 8f, row f1).
 * weights / sigmas: f64 [rows][n_features] row-major, n_features <= 64, mu <= 4096.  Row r draws from
 * philox(counter=(draw, r, tag, generation), key=seed) with the reference's call shapes; exp/log use correctly
 * rounded basic operations only, so results are bit-identical to oracle/sb_oracle_es.c.
 *
 * sb_es_offspring: Population.generate_offspring (evo/population.py:75-90) + WeightVector.mutate
 * (evo/weights.py:20-40): child c = mutate(copy(parent randint(0, mu))) written to row mu + c; parents_d nullable i32[lambda].
 * sb_es_select: the top-mu part of Population.select_from_combined (evo/population.py:99-107): fitness descending,
 * ties in input order; order_d nullable i32[mu] = source row of each survivor.
 * sb_es_reset_sigmas: evo/population.py:128-139.  sb_es_inject_diversity: evo/population.py:146-170; chosen_d
 * nullable i32[max(1, mu/2)].  The caller evaluates the two trigger conditions from the survivors' statistics. */
int sb_es_offspring(SbHandle *h, uint64_t seed, uint32_t generation, int mu, int lambda, int n_features, double tau, double tau_prime,
                    double min_sigma, double *w_d, double *s_d, int32_t *parents_d, void *stream);
int sb_es_select(SbHandle *h, int total, int mu, int n_features, const double *fitness_d, const double *w_d, const double *s_d,
                 double *w_out_d, double *s_out_d, double *fit_out_d, int32_t *order_d, void *stream);
int sb_es_reset_sigmas(SbHandle *h, uint64_t seed, uint32_t generation, int mu, int n_features, double initial_sigma, double *s_d, void *stream);
int sb_es_inject_diversity(SbHandle *h, uint64_t seed, uint32_t generation, int mu, int n_features, double tau, double tau_prime,
                           double min_sigma, double initial_sigma, double *w_d, double *s_d, int32_t *chosen_d, void *stream);

/* Stormbound.expert_action (games/stormbound.py:563-637) for n games: the scripted opponent behind
 * Game.expert_agent (games/stormbound.py:201-209).  It draws its choices from the GAME's stream, so each
 * state's draw counter (and err byte, for the reference's choice([]) / max([]) exceptions) is updated in
 * place; actions_d u8[n]. */
int sb_expert_action(SbHandle *h, int n, uint8_t *states_d, uint8_t *actions_d, void *stream);

/* Uniform-random legal agent until done/err or max_steps more steps (SURVEY 8d config 2; the agent
 * stream is philox(counter=(step,0,0xA6E7,0), key=seed)).  steps_d i32[n] = steps taken by this call;
 * chain_d (nullable) u64[n] = running hash of the per-step state digests (parity evidence). */
int sb_rollout_random(SbHandle *h, int n, uint8_t *states_d, int max_steps, int32_t *steps_d, uint64_t *chain_d,
                      void *stream);

/* FitnessEvaluator._play_game (evo/fitness.py:178-228) with the intended loop (until have_winner or
 * max_steps env steps): FIRST plays w_first_d[idx_first_d[g]], SECOND w_second_d[idx_second_d[g]]
 * (idx arrays nullable = row g... row 0 when the weight table has one row is expressed by idx).
 * A NULL weight table hands that seat to Stormbound.expert_action (games/stormbound.py:563-637): the agent-vs-expert
 * match of play_vs_expert.py:65-94, batched.
 * result_d i8[n]: 0 FIRST won, 1 SECOND won, -1 draw/timeout, -2 aborted by an engine exception. */
int sb_rollout_heuristic(SbHandle *h, int n, uint8_t *states_d, const double *w_first_d, const double *w_second_d,
                         const int32_t *idx_first_d, const int32_t *idx_second_d, int max_steps, int8_t *result_d,
                         int32_t *steps_d, void *stream);

/* Batched auto-resetting environment: Game.reset / Game.step (games/stormbound.py:121-250) driven by an outside policy, and
 * the agent-vs-expert loop of play_vs_expert.py:65-94, one env per 512-byte record of states_d u8[n,512].
 * opponent: 0 none (self-play: the caller acts for both seats), 1 uniform-random legal agent (the stream of
 * sb_rollout_random), 2 Stormbound.expert_action (the game's own stream, as sb_expert_action), 3 heuristic agent
 * (sb_select_action) with weights w_opp_d f64[P,10], row idx_opp_d[g] (nullable = row g).  seat_d u8[n] (nullable = 0):
 * the learner's seat, 0 FIRST / non-zero SECOND; ignored for opponent 0.
 * sb_env_reset: sb_reset for seeds_d (byte-identical), then the opponent plays until the learner is to move.
 * sb_env_step: (1) actions_d[g] outside the legal mask leaves env g untouched, result -4; (2) apply it; (3) the opponent plays
 * until the learner is to move or the episode is over; (4) at the end of an episode the finished record goes to
 * final_states_d and the env deals its next game in place from next_seed(Philox key of the finished record), with the same
 * decks / factions (u8[2,n_deck] + u8[2] when decks_shared, else u8[n,2,n_deck] + u8[n,2]), and the opponent opens it when it
 * is FIRST; (5) observation obs_d i32[n,27,5,4] with obs_err_d (observe()'s code: non-zero only for UP01-03) and legal mask
 * masks_d u32[n,5] of the returned record.  An episode is over when a base is below 0, state.err is set, or the record's
 * steps (both seats, since the deal) reach max_steps.  result_d i8[n]: 0 FIRST won, 1 SECOND won, -1 draw / timeout,
 * -2 aborted by an engine status (as sb_rollout_heuristic), -3 the episode continues, -4 action rejected; length_d i32[n] =
 * env steps of the episode that ended in this call, else 0.  Between calls every record is what chaining sb_step (plus
 * sb_expert_action / sb_select_action for the opponent) gives.  next_seed(s): z = s + 0x9E3779B97F4A7C15,
 * z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9, z = (z ^ z >> 27) * 0x94D049BB133111EB, z ^= z >> 31, z & 0x7FFFFFFFFFFFFFFF.
 * obs_d, masks_d, obs_err_d, final_states_d are nullable.  A bad opponent kind, kind 3 without a table, n_deck outside 1..16
 * or max_steps outside 1..65535 returns -1 (sb_last_error) and launches nothing; n = 0 is a no-op.  One call = one kernel
 * launch without handle scratch, atomics or host synchronisation: calls on different streams through one handle do not race,
 * and a call can be captured in a CUDA graph.  The kernel is fixed by the opponent kind ("engine" of sb_set_option does not
 * apply): one env per thread for 0-2, one env per warp for 3. */
int sb_env_reset(SbHandle *h, int n, const uint64_t *seeds_d, const uint8_t *decks_d, int n_deck, int decks_shared,
                 const uint8_t *factions_d, int opponent, const uint8_t *seat_d, const double *w_opp_d,
                 const int32_t *idx_opp_d, int max_steps, uint8_t *states_d, int32_t *obs_d, uint32_t *masks_d,
                 uint8_t *obs_err_d, void *stream);
int sb_env_step(SbHandle *h, int n, uint8_t *states_d, const uint8_t *actions_d, const uint8_t *decks_d, int n_deck,
                int decks_shared, const uint8_t *factions_d, int opponent, const uint8_t *seat_d, const double *w_opp_d,
                const int32_t *idx_opp_d, int max_steps, int8_t *result_d, int32_t *length_d, uint8_t *final_states_d,
                int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d, void *stream);

/* Batched Monte-Carlo tree search (PUCT) with a caller-supplied evaluator: n independent trees, tree g rooted at record
 * roots_d[g] (u8[n,512]), at most max_nodes nodes each, node 0 the root.  The evaluator (prior f32[n,156] over action ids,
 * value f32[n] from the point of view of the seat to move at the leaf) stays with the caller; the loop is
 *   sb_search_begin -> evaluate -> (sb_search_simulate -> evaluate) x S -> sb_search_end.
 * Transitions: the child of (s, a) is the record sb_step(s, a) produces (game_step + end_of_step on the parent record, draws
 * from the game's own stream), so the tree sees both hands and the future draws (perfect-information search).
 * Terminal (as sb_env_step): a base below 0, err set, or steps >= max_steps; value +1 FIRST won, -1 SECOND won, 0 draw,
 * timeout or engine status.  Selection at a non-terminal node s: the legal a maximising q + u, q = sgn(s) W(child) / n_a
 * (fpu when n_a = 0), u = ((c_puct P(s,a)) sqrt(N(s))) / (1 + n_a), sgn = +1 when FIRST is to move; correctly rounded
 * FP64 in this order, ties to the lowest action id; descent continues through existing non-terminal children.  A missing
 * child is expanded into the next free node; a terminal node ends the walk without a new node.  Backup: N += 1 and W += v
 * (FIRST's view: the caller's value times sgn(leaf), or the game value at a terminal leaf) from the leaf to the root.
 * Leaf outputs (all nullable): leaf_states_d u8[n,512] the leaf record, obs_d i32[n,27,5,4] / obs_err_d u8[n] (sb_observe),
 * masks_d u32[n,5] (sb_legal_mask), to_move_d u8[n] (0 FIRST, 1 SECOND), leaf_kind_d u8[n]: 0 evaluate the leaf, 1 terminal
 * (the game value is used, the caller's prior / value are ignored), 2 the tree is full and nothing is pending (the root is
 * emitted).  A tree that has used all max_nodes nodes stops: that call backs up and reports 2, later calls leave it alone.
 * sb_search_begin: root -> node 0, emitted as the first pending leaf.  sb_search_simulate: store prior_d / value_d for the
 * pending leaf and back it up, then select, expand and emit the next leaf.  sb_search_end: back up the last pending leaf,
 * then visits_d i32[n,156] (N of the root's children, 0 where none), q_d f64[n,156] (sgn(root) W / N of the root's
 * children, NaN where unvisited), root_value_d f64[n] (sgn(root) W / N of the root).
 * The workspace ws_d is caller-owned and opaque, 16-byte aligned, at least sb_search_workspace_bytes(n, max_nodes) bytes
 * (host only, no GPU; 0 for n < 0 or max_nodes outside 1..2^24); every call of one search passes the same n, max_nodes and
 * workspace.  Bad arguments return -1 (sb_last_error) and launch nothing: n < 0, max_nodes outside 1..2^24, a NULL,
 * misaligned or too small workspace, max_steps outside 1..65535, c_puct negative or not finite, fpu not finite, NULL
 * roots / prior / value / visits / q / root_value where they are used; n = 0 is a no-op.  One call = one kernel launch, one
 * tree per thread, without handle scratch, atomics or host synchronisation: searches on different streams through one handle
 * do not race, and a whole search with a capture-safe evaluator can be captured in a CUDA graph. */
size_t sb_search_workspace_bytes(int n, int max_nodes);
int sb_search_begin(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const uint8_t *roots_d, int max_steps,
                    uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d,
                    uint8_t *leaf_kind_d, void *stream);
int sb_search_simulate(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d,
                       const float *value_d, double c_puct, double fpu, uint8_t *leaf_states_d, int32_t *obs_d,
                       uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_search_end(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d, const float *value_d,
                  int32_t *visits_d, double *q_d, double *root_value_d, void *stream);

/* Information-set Monte-Carlo tree search (single-observer ISMCTS) with a caller-supplied evaluator: n trees, tree g built
 * over the information set of the player to move at its root, at most max_nodes nodes, node 0 the root.  The loop is
 *   sb_ismcts_begin(world 0) -> evaluate -> (sb_ismcts_simulate(world k) -> evaluate) x S -> sb_ismcts_end.
 * Worlds come from the caller: det_d u8[n,512] is this call's world of each root, normally sb_determinize(roots, keys_k)
 * with fresh keys_k per call (simulation k walks world k; world 0 is the one passed to begin).  The kernels do not
 * determinize; the caller promises that every world of tree g is a determinization of the same root for that root's own
 * local_order, so the root's legal set is the same in every world.
 * Nodes carry no record: parent, first child, next sibling, the move code of the edge into the node, the seat to move,
 * N, W (FIRST's view) and the f32[156] prior the caller gave when the node was evaluated (zero for a node created terminal).
 * Move codes (u32, kind << 24 | card << 16 | x) key an edge by what the move is, from the mover's hand in the current
 * world, ci the hand slot: PLACE a < 64 -> (0, hand[ci].card, a & 15); SPELL 64..147 -> (1, card, (a - 64) % 21);
 * CYCLE 148..151 -> (2, card, 0); 152..154 -> (3, hand[ci].card, hand[0].card); PASS -> 4 << 24.  When two legal ids
 * give one code (copies of a card), the lowest id represents it and the others are never chosen.
 * Walk (sb_ismcts_simulate, after the backup): unpack the world's record at the root; at each node (1) if the world's
 * state is over (as sb_env_step: a base below 0, err set, or steps >= max_steps) the walk ends: a terminal leaf, kind 1,
 * with this world's game value (a node can be terminal in one world and not in another); (2) else select among the
 * world's legal representative ids with sb_search_simulate's PUCT formula, FP64 order and ties (n_a, W of the child with
 * that id's code, P the node's stored prior at the world's action id); (3) step as sb_step does (game_step + end_of_step +
 * pack + unpack) and descend into the child with the code, or expand a new node for it, emitted with kind 0, or 1 when
 * its state is over.  Leaf outputs (all nullable) as sb_search_*: the WORLD's record at the leaf (so the evaluator never
 * sees the true root's hidden cards or key), observation, legal mask, seat to move, kind.  Backup as sb_search_*: N += 1,
 * W += v from the leaf to the root.  A tree that has used all max_nodes nodes stops: kind 2, the world's root record is
 * emitted, later calls leave it alone.  sb_ismcts_end: back up the last pending leaf, then visits_d i32[n,156], q_d
 * f64[n,156] and root_value_d f64[n] as sb_search_end, by the root's action ids through the codes stored at begin; an id
 * that does not represent its code (or is illegal) reads 0 / NaN.
 * Workspace: caller-owned, opaque, 16-byte aligned, at least sb_ismcts_workspace_bytes(n, max_nodes) = n * 656 * (1 +
 * max_nodes) bytes (host only; 0 for n < 0 or max_nodes outside 1..2^24); every call of one search passes the same n,
 * max_nodes and workspace.  Node indices read from the workspace are bounds-checked, so a workspace not written by
 * sb_ismcts_begin cannot send a thread outside its own tree.  Bad arguments return -1 (sb_last_error) and launch nothing,
 * as sb_search_*, plus a NULL det_d; n = 0 is a no-op.  One call = one kernel launch, one tree per thread, without handle
 * scratch, atomics or host synchronisation (capturable in a CUDA graph with a capture-safe evaluator). */
size_t sb_ismcts_workspace_bytes(int n, int max_nodes);
int sb_ismcts_begin(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const uint8_t *det_d, int max_steps,
                    uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d,
                    uint8_t *leaf_kind_d, void *stream);
int sb_ismcts_simulate(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const uint8_t *det_d,
                       const float *prior_d, const float *value_d, double c_puct, double fpu, uint8_t *leaf_states_d,
                       int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d,
                       void *stream);
int sb_ismcts_end(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d, const float *value_d,
                  int32_t *visits_d, double *q_d, double *root_value_d, void *stream);

/* Gumbel search (Gumbel MuZero, Danihelka et al. 2022; mctx's gumbel_muzero_policy) for both tree searches, ABI 5's additive
 * entry points.  A search is the PUCT begin, then S calls of the Gumbel simulate with sim = 1..S, then the Gumbel end:
 *   sb_search_begin -> evaluate -> (sb_search_simulate_gumbel(sim = k) -> evaluate) x S -> sb_search_end_gumbel
 *   sb_ismcts_begin(world 0) -> evaluate -> (sb_ismcts_simulate_gumbel(world k, sim = k) -> evaluate) x S -> sb_ismcts_end_gumbel
 * Workspaces, backup, expansion, terminal rule, leaf outputs and full trees are those of sb_search_* / sb_ismcts_*; mixing
 * PUCT and Gumbel calls in one search is unsupported.  gumbel_d f32[n,156] is the caller's Gumbel noise (normally
 * -log(-log u)), the same for every call of one search; only entries at legal ids are read.  Selection (correctly rounded
 * FP64, log / exp the library's own, DESIGN.md 8.9), at a non-terminal node s with legal set A (8.6: its legal ids; 8.8: the
 * world's legal representatives, children by move code), n_a / W_a of a's child, q_a = sgn(s) W_a / n_a:
 *   vhat = sgn (W(s) - sum_children W) / (N(s) - sum_children N) (0 if that denominator is < 1);
 *   vmix = (vhat + sumN * (sum_{n_a>0} p~_a q_a / sum_{n_a>0} p~_a)) / (1 + sumN), p~ = max(prior, 2^-126), sumN = sum_A n_a;
 *   completed q = q_a (n_a > 0) else vmix, rescaled to [0, 1] over A (range floor 1e-8);
 *   sigma_a = (c_visit + max_A n) * c_scale * rescaled q_a;  logit_a = log(prior_a) (-1e9 where prior_a <= 0);
 *   interior nodes: argmax_A of softmax_A(logit + sigma)_a - n_a / (1 + sumN);
 *   the root at call sim = k: argmax of max(-1e9, g_a + logit_a + sigma_a) over the ids whose n_a equals seq(m, S)[k-1]
 *   (all of A when none does), m = min(max_considered, |A|), seq mctx's sequential-halving visit schedule.
 * Ties go to the lowest id and a NaN never wins, so a non-empty A always gives a legal id.  The end backs up the last pending
 * leaf and writes visits_d, q_d and root_value_d exactly as sb_search_end / sb_ismcts_end, plus action_d i32[n] (argmax of
 * g + logit + sigma over the ids with the most root visits; 255 when no root id has a visit, e.g. a terminal root) and
 * policy_d f32[n,156] (the softmax of logit + sigma over A with the final counts, 0 outside A; 8.8's A at the end is the ids
 * with a root code, so an id that repeats a lower id's card reads 0).  Bad arguments return -1 and launch nothing: those of
 * the PUCT sibling, sim outside 1..num_simulations, num_simulations outside 1..2^24, max_considered outside 1..156, c_visit
 * or c_scale negative or not finite, a NULL gumbel (and, at the end, action or policy) with n > 0; n = 0 is a no-op.  One
 * call = one kernel launch, without handle scratch, atomics or host synchronisation (capturable in a CUDA graph). */
int sb_search_simulate_gumbel(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d,
                              const float *value_d, const float *gumbel_d, int sim, int num_simulations, int max_considered,
                              double c_visit, double c_scale, uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d,
                              uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_search_end_gumbel(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d,
                         const float *value_d, const float *gumbel_d, double c_visit, double c_scale, int32_t *action_d,
                         float *policy_d, int32_t *visits_d, double *q_d, double *root_value_d, void *stream);
int sb_ismcts_simulate_gumbel(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const uint8_t *det_d,
                              const float *prior_d, const float *value_d, const float *gumbel_d, int sim, int num_simulations,
                              int max_considered, double c_visit, double c_scale, uint8_t *leaf_states_d, int32_t *obs_d,
                              uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_ismcts_end_gumbel(SbHandle *h, int n, int max_nodes, void *ws_d, size_t ws_bytes, const float *prior_d,
                         const float *value_d, const float *gumbel_d, double c_visit, double c_scale, int32_t *action_d,
                         float *policy_d, int32_t *visits_d, double *q_d, double *root_value_d, void *stream);

/* Tree reuse between moves for both PUCT searches, ABI 5's additive entry points (DESIGN.md 8.10).  An advance is the
 * matching begin (sb_search_begin on roots_d / sb_ismcts_begin on world 0 det_d, same leaf outputs and kinds), except that
 * it may carry each tree's subtree below the new root over from a finished search:
 *   sb_search_advance(ws_src -> ws_dst, roots) -> evaluate -> (sb_search_simulate -> evaluate) x S -> sb_search_end
 *   sb_ismcts_advance(ws_src -> ws_dst, world 0, played) -> evaluate -> (sb_ismcts_simulate(world k) -> evaluate) x S -> ...
 * ws_src and ws_dst are two non-overlapping workspaces of this n and max_nodes (ws_bytes is checked for both); ws_src is
 * consumed: its contents afterwards are unspecified, except that each of its trees then holds no node, so advancing from
 * it again (e.g. replaying a captured advance) starts every tree fresh.  ws_dst receives, for each tree g, either exactly what the begin
 * writes for this call's root (kept_d[g] = 0) or the kept subtree of ws_src's tree g (kept_d[g] = its node count >= 1):
 * the matched node j and its descendants in creation order (increasing node index), the first `keep` of them, j as node 0
 * with parent -1.  Kept nodes keep N, W, prior, mask, record or code, seat and terminal data; a child link to a node not
 * kept becomes none (8.6: 0 in child[], 8.8: left out of the sibling list, whose order is otherwise kept).  The new root is
 * the pending leaf (kind 0, or 1 when terminal); the next simulate or end backs it up as usual, so the caller's prior
 * replaces the stored one and N / W gain that evaluation.  The ancestors' N / W still count the visits of dropped nodes.
 * A tree is reused only when ws_src's header says finished (by _end, or stopped full: nothing pending) with this call's
 * max_steps, and the rule finds j:
 *   sb_search_advance: j = the lowest-index node whose 512-byte record equals roots_d[g] byte for byte;
 *   sb_ismcts_advance: j = the child of the source root with the code ws_src's header stores for root action id played_d[g]
 *     (0..155, not ISM_NONE), when det_d[g] is not over and its seat to move is both j's and the source root's (one
 *     observer: a PASS or a turn handed over starts fresh).  The caller promises that the new root
 *     is the record sb_step(old root, played) gives; -1 (or any id outside 0..155) starts the tree fresh.
 * Otherwise the tree starts fresh.  Gumbel simulate / end calls on an advanced workspace are unsupported.  Bad arguments
 * return -1 (sb_last_error) and launch nothing: those of the begin, keep outside 1..max_nodes, a NULL or misaligned ws_src,
 * ws_src == ws_dst or overlapping, a NULL played_d (sb_ismcts_advance); kept_d and the leaf outputs are nullable; n = 0 is a
 * no-op.  One call = one kernel launch (one warp per tree for the copy), without handle scratch, atomics or host
 * synchronisation (capturable in a CUDA graph).  Node indices read from ws_src are bounds-checked against its node count. */
int sb_search_advance(SbHandle *h, int n, int max_nodes, void *ws_src_d, void *ws_dst_d, size_t ws_bytes,
                      const uint8_t *roots_d, int max_steps, int keep, int32_t *kept_d, uint8_t *leaf_states_d, int32_t *obs_d,
                      uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_ismcts_advance(SbHandle *h, int n, int max_nodes, void *ws_src_d, void *ws_dst_d, size_t ws_bytes,
                      const uint8_t *det_d, const int32_t *played_d, int max_steps, int keep, int32_t *kept_d,
                      uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d, uint8_t *to_move_d,
                      uint8_t *leaf_kind_d, void *stream);

/* Several leaves per tree per call for the perfect-information search, under virtual loss, ABI 5's additive entry points
 * (DESIGN.md 8.11):
 *   sb_search_begin or sb_search_advance -> evaluate (n rows) -> (sb_search_simulate_batch -> evaluate (n * L rows)) x C
 *   -> sb_search_end_batch
 * The workspace is sb_search_batch_workspace_bytes(n, max_nodes, L) bytes: 8.6's workspace of sb_search_workspace_bytes(n,
 * max_nodes) bytes, unchanged (so begin and advance write it, and advance reads a finished batched tree, as for 8.6), then
 * per tree a tail holding the call's L pending slots and one int of virtual visits per node.  0 for bad arguments (n < 0,
 * max_nodes outside 1..2^24, leaves outside 1..256, an overflow).  Every call of one search uses the same n, max_nodes and L.
 * Slot l of tree g is row g * L + l of prior_d f32[n * L,156], value_d f32[n * L] and of every leaf output (sb_search_begin's
 * outputs with n * L rows).  On a tree that begin, advance or a plain simulate left (one pending leaf), a batch call or
 * the batch end backs up that leaf from row g * L (slot 0); afterwards the L slots are pending.  Mixing plain and batch
 * calls within one search is otherwise unsupported (it computes wrong numbers, never outside the tree).  One batch call:
 *   1. backs up the L pending slots in ascending slot order: EVAL stores the prior and adds sgn(leaf) * value along the path,
 *      N += 1; TERMINAL adds the node's game value; FULL and COLLISION add nothing;
 *   2. selects L leaves one after another: V(x) = the number of earlier slots of this call whose path (root to stop node
 *      inclusive) contains x; at a non-terminal node s, for each legal a with child c (n_a = 0 without one) and sgn the sign
 *      of s's seat: n_a = N(c) + V(c), q = ((sgn * W(c)) - (vl * V(c))) / n_a (fpu when n_a = 0),
 *      u = ((c_puct * P(s,a)) * sqrt(N(s) + V(s))) / (1 + n_a), score = q + u, the highest wins, ties to the lowest id;
 *      correctly rounded FP64 in this order (with V = 0 exactly sb_search_simulate's scores).  A walk stops at a new edge
 *      (it takes the next free node at once: the slot is EVAL, or TERMINAL when the new record is over), at an existing
 *      terminal node (TERMINAL, backed up again), at a node allocated earlier in the same call (COLLISION = 3: the root is
 *      emitted, nothing is backed up) or, when no free node is left, with this and every later slot FULL (the root is
 *      emitted; later calls stop the tree, as sb_search_simulate does);
 *   3. expands the new nodes (the records sb_step(parent, a) gives) and emits every slot's leaf outputs, in parallel over
 *      the n * L slots.  Virtual visits are zero again when the call returns.
 * sb_search_end_batch backs up what is pending and writes sb_search_end's read-out (visits, q NaN where unvisited, root
 * value); root visits then add up to the slots that were neither COLLISION nor FULL (plus the root's own evaluation).
 * Bad arguments return -1 (sb_last_error) and launch nothing: those sb_search_simulate / sb_search_end reject (ws_bytes
 * against the batch size), leaves outside 1..256, a negative or non-finite virtual_loss, n * leaves >= 2^31; n = 0 is a
 * no-op.  sb_search_simulate_batch is two kernel launches (selection, one thread per tree; expansion, one thread per slot),
 * sb_search_end_batch one, without handle scratch, atomics or host synchronisation (capturable in a CUDA graph).  Every
 * index read from the workspace is checked; a bad one stops the tree (FULL) and is never dereferenced. */
size_t sb_search_batch_workspace_bytes(int n, int max_nodes, int leaves);
int sb_search_simulate_batch(SbHandle *h, int n, int max_nodes, int leaves, void *ws_d, size_t ws_bytes,
                             const float *prior_d, const float *value_d, double c_puct, double fpu, double virtual_loss,
                             uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d, uint8_t *obs_err_d,
                             uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_search_end_batch(SbHandle *h, int n, int max_nodes, int leaves, void *ws_d, size_t ws_bytes, const float *prior_d,
                        const float *value_d, int32_t *visits_d, double *q_d, double *root_value_d, void *stream);

/* Several leaves per tree per call for the information-set search, under virtual loss, ABI 5's additive entry points
 * (DESIGN.md 8.12): sb_search_simulate_batch's contract over sb_ismcts_*'s tree, with one world per slot.
 *   sb_ismcts_begin (world 0) or sb_ismcts_advance -> evaluate (n rows) -> (sb_ismcts_simulate_batch (the worlds of call c)
 *   -> evaluate (n * L rows)) x C -> sb_ismcts_end_batch
 * The workspace is sb_ismcts_batch_workspace_bytes(n, max_nodes, L) bytes: sb_ismcts_workspace_bytes(n, max_nodes) bytes of
 * 8.8's layout, unchanged (so begin and advance write it, and advance reads a finished batched tree), then per tree a tail
 * of the L pending slots (node, kind and the game value a TERMINAL slot was reached with in its world) and one int of
 * virtual visits per node.  0 for bad arguments, as sb_search_batch_workspace_bytes.  det_d u8[n * L,512]: row g * L + l is
 * the world of slot l of tree g, a determinization of root g for root g's own local_order.  prior_d, value_d and every leaf
 * output have n * L rows in the same layout.  A tree that begin, advance or a plain simulate left is backed up from row
 * g * L (slot 0).  One batch call is what running these steps slot by slot gives:
 *   1. back up the pending slots in ascending slot order: EVAL stores the prior and adds sgn(leaf) * value along the path,
 *      N += 1; TERMINAL adds the slot's stored game value; FULL and COLLISION add nothing;
 *   2. for l = 0 .. L-1, walk from the root through world l as sb_ismcts_simulate does: where world l is over (env_over)
 *      the walk ends as TERMINAL with world l's value; else select among world l's legal representatives with
 *      sb_search_simulate_batch's score (children matched by move code; V(x) = the earlier slots of this call whose path
 *      contains x; with V = 0 exactly sb_ismcts_simulate's scores), ties to the lowest id, and step the world.  Then descend
 *      into an existing child; stop at a node created earlier in this call (COLLISION = 3: world l's root is emitted,
 *      nothing is backed up); or, for a code without a child, take the next free node at once (inserted at the head of the
 *      sibling list; the slot is EVAL, or TERMINAL with a zero prior when world l is over there).  When no node is free,
 *      this and every later slot are FULL (world l's root emitted).  V is zero again when the call returns;
 *   3. every slot emits world l's record at its leaf (leaf record, observation, obs_err, mask, seat to move, kind).
 * sb_ismcts_end_batch backs up what is pending and writes sb_ismcts_end's read-out by the root codes stored at begin.
 * Bad arguments return -1 (sb_last_error) and launch nothing: those sb_ismcts_simulate / sb_ismcts_end reject (ws_bytes
 * against the batch size), leaves outside 1..256, a negative or non-finite virtual_loss, n * leaves >= 2^31; n = 0 is a
 * no-op.  Each call is one kernel launch, without handle scratch, atomics or host synchronisation (capturable in a CUDA
 * graph).  Mixing plain and batch calls within one search is unsupported (wrong numbers, never outside the tree).  Every
 * index read from the workspace is checked; a bad one stops the tree (FULL) and is never dereferenced. */
size_t sb_ismcts_batch_workspace_bytes(int n, int max_nodes, int leaves);
int sb_ismcts_simulate_batch(SbHandle *h, int n, int max_nodes, int leaves, void *ws_d, size_t ws_bytes,
                             const uint8_t *det_d, const float *prior_d, const float *value_d, double c_puct, double fpu,
                             double virtual_loss, uint8_t *leaf_states_d, int32_t *obs_d, uint32_t *masks_d,
                             uint8_t *obs_err_d, uint8_t *to_move_d, uint8_t *leaf_kind_d, void *stream);
int sb_ismcts_end_batch(SbHandle *h, int n, int max_nodes, int leaves, void *ws_d, size_t ws_bytes, const float *prior_d,
                        const float *value_d, int32_t *visits_d, double *q_d, double *root_value_d, void *stream);

/* Determinization for sampled (PIMC) search:out_d[g] = states_d[g] with everything observer o cannot see resampled and
 * everything o sees kept byte for byte (sb_observe / sb_legal_mask / sb_features of o's view are unchanged).
 * observer_d u8[n] is nullable: NULL = each record's own local_order (the seat sb_observe and sb_legal_mask show); a
 * non-zero byte means SECOND.  keys_d u64[n] is the new Philox key of each record.  With r = 1 - o:
 *   movable slots of pl[r]: hand 0..n_hand-1, then deck 0..n_deck-1 (clamped to 4 / 16), skipping every record whose
 *   flags carry SB_CF_OBJ (ext[91..107] addresses those by slot); Fisher-Yates from the end over the (card, cost, flags)
 *   triples at those slots, for i = m-1 .. 1: j = umulhi(w0, i + 1), w0 = word 0 of
 *   philox(counter=(t, 0, 0xDE7E, 0), key=(keys_d[g] low, high)), t = 0, 1, .. the swap index; deck_wn stays with its
 *   slot; seed_lo / seed_hi <- keys_d[g].  Every other byte is unchanged (turn, draw, steps, err, done included).
 * The opponent's card multiset (hand + deck) is taken as known: both decks are fixed per game.  out_d may equal
 * states_d (in place); partial overlap is undefined.  Bad arguments return -1 (sb_last_error) and launch nothing: n < 0,
 * NULL states / keys / out with n > 0; n = 0 is a no-op.  One call = one kernel launch (one record per warp), without
 * handle scratch, atomics or host synchronisation, so it can be captured in a CUDA graph. */
int sb_determinize(SbHandle *h, int n, const uint8_t *states_d, const uint8_t *observer_d, const uint64_t *keys_d,
                   uint8_t *out_d, void *stream);

/* FitnessEvaluator.evaluate_population inner reduction (evo/fitness.py:95,160-166): counts_d i32[P,3]
 * += {wins, draws, losses} of individual idx_first_d[g] over the n finished games. */
int sb_accumulate_fitness(SbHandle *h, int n, const int8_t *result_d, const int32_t *idx_first_d, int32_t *counts_d,
                          void *stream);

/* The evaluation schedule on the device (evo/fitness.py:52-59 pairings, :100-121 games per pairing): game index
 * game_lo + t -> idx_first_d[t], idx_second_d[t] (rows of the weight table) and seeds_d[t] for t < n.  A pairing plays
 * games_per_pair consecutive games.  mode 0 = the reference's round robin: ordered pairs (i, j), i < n_ind, j < n_total,
 * j != i (rows n_ind.. are the hall of fame); mode 1 = every individual as FIRST against each of the n_total - n_ind fixed
 * opponents; mode 2 = (i, i), for a SECOND seat played by expert_action.  seeds are the partition-invariant hash of
 * (base_seed, generation, i, j, replicate) (the reference seeds every game from OS entropy, SURVEY Q16).  A bad schedule
 * returns -1 (sb_last_error) and launches nothing: mode outside 0..2, n_ind < 1, games_per_pair < 1, n_total < n_ind, a round
 * robin of fewer than 2 rows, or versus without an opponent row (n_total == n_ind).  n <= 0 is a no-op. */
int sb_eval_schedule(SbHandle *h, int mode, int n_ind, int n_total, int games_per_pair, uint64_t base_seed, uint32_t generation,
                     int64_t game_lo, int n, int32_t *idx_first_d, int32_t *idx_second_d, uint64_t *seeds_d, void *stream);

/* FitnessEvaluator.evaluate_population (evo/fitness.py:32-121) for the games [game_lo, game_hi) of a schedule (a rank's shard),
 * entirely on the device: sb_eval_schedule -> sb_reset (decks_d u8[2,n_deck] shared by all games, factions_d u8[2]) ->
 * sb_rollout_heuristic over weights_d f64[n_total,10] -> sb_accumulate_fitness into counts_d i32[n_ind,3] (+=) and
 * sb_count_aborted into aborted_d i32[2] (+=, nullable), chunk_games at a time (<= 0: 262,144) in a workspace owned by the
 * handle.  Asynchronous on `stream`; nothing is copied to the host.  A bad schedule returns -1 as sb_eval_schedule does,
 * before the first launch. */
int sb_eval_population(SbHandle *h, int mode, int n_ind, int n_total, int games_per_pair, uint64_t base_seed, uint32_t generation,
                       int64_t game_lo, int64_t game_hi, const double *weights_d, const uint8_t *decks_d, int n_deck,
                       const uint8_t *factions_d, int max_steps, int chunk_games, int32_t *counts_d, int32_t *aborted_d, void *stream);

/* Games a rollout aborted (result -2), split by cause: out_d i32[2] += {games stopped by an exception the reference raises
 * too (state.err 1..4; evo/fitness.py:208-210 scores them as a draw as well), games stopped by a limit of this engine
 * (state.err 5..7: SB_ERR_UNSUPPORTED / OVERFLOW / DEPTH -- the reference would have kept playing)}.  The evaluator
 * reports both and warns when the second exceeds 1 % of the games. */
int sb_count_aborted(SbHandle *h, int n, const uint8_t *states_d, const int8_t *result_d, int32_t *out_d, void *stream);

/* Host-buffer variants (pinned or pageable host memory; H2D + kernel + D2H + sync inside): the e2e path. */
int sb_step_host(SbHandle *h, int n, uint8_t *states, const uint8_t *actions, int8_t *reward, uint8_t *done,
                 uint8_t *err, uint32_t *next_masks);
int sb_rollout_random_host(SbHandle *h, int n, const uint64_t *seeds, const uint8_t *decks, int n_deck,
                           const uint8_t *factions, int max_steps, uint8_t *states_out, int32_t *steps_out,
                           uint64_t *chain_out);

#ifdef __cplusplus
}
#endif
#endif
