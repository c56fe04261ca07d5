// sb_kernels.cu -- sm_100a kernels and the C ABI of libsb_b200.so (include/sb_b200.h).
//
// Kernels
//   k_reset            one game per thread: shuffle, weights, opening hands (games/stormbound.py:293-304)
//   k_generate_decks   one game per thread: both decks of DeckEvolutionConfig.get_deck_configuration (utils.py:26-241)
//   k_legal_mask       one game per thread -> 156-bit mask (games/stormbound.py:528-557)
//   k_expert_action    one game per thread: the scripted opponent (games/stormbound.py:563-637)
//   k_step             one game per thread: unpack, Stormbound.step, pack, fused next legal mask
//   k_observe/k_features  one game per thread
//   k_rollout_random   one game per thread, whole rollout in one launch (state never leaves the SM); turn-synchronous
//                      phases, persistent grid with lane refill and a 32-register dense build for large batches
//   k_select_action    one WARP per game, one lane per candidate action (fork, step, features, score,
//                      warp arg-max by shuffles) -- evo/heuristic_agent.py:53-80
//   k_rollout_heuristic  one warp per game, whole game in one launch, working-set image of the game in shared memory;
//                      a seat without weights is played by the scripted opponent
//   k_env_step         one env per thread: learner action, random / expert / no opponent, auto-reset, observation + mask
//   k_env_step_heur    one env per warp: the same with a heuristic-agent opponent (decide(), as in k_rollout_heuristic)
//   k_search_*         batched PUCT tree search, one tree per thread, one launch per simulation (sb_search.cuh)
//   k_ismcts_*         information-set tree search over caller-supplied worlds, one tree per thread (sb_ismcts.cuh)
//   k_*_gumbel         Gumbel selection and read-out for both tree searches (sb_gumbel.cuh)
//   k_determinize      one record per warp: resample what the observer cannot see (sb_determinize.cuh)
//   k_accumulate_fitness win/draw/loss counts per individual (evo/fitness.py:95,160-166)
//   k_es_*             evolution-strategy operators on the resident population (sb_es.cuh; evo/weights.py, evo/population.py)
// State is AoS [n][512 B]; every thread (or warp) moves its record with 128-bit loads/stores; the card
// table (130 x 24 B) is staged in shared memory once per CTA.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include "../../include/sb_b200.h"
#include "sb_effects.cuh"
#include "sb_state_io.cuh"
#include "sb_es.cuh"
#include "sbw_launch.h"

#define SB_ABI_VERSION 5
#define TPB_GAME 64      // threads per CTA for thread-per-game kernels
#define WARPS_PER_CTA 4  // games per CTA for warp-per-game kernels
#ifndef HEUR_MIN_CTAS
#define HEUR_MIN_CTAS 16  // 4-warp CTAs per SM the heuristic rollout is compiled for (12 -> 42 registers, 1,536 threads/SM)
#endif

// ---------------------------------------------------------------- helpers
SBD_FI void stage_cards(DCard* s_cards, const DCard* cards) {
  const u32* src = reinterpret_cast<const u32*>(cards);
  u32* dst = reinterpret_cast<u32*>(s_cards);
  for (int i = threadIdx.x; i < (int)(SBC_COUNT * sizeof(DCard) / 4); i += blockDim.x) dst[i] = __ldg(src + i);
  __syncthreads();
}
SBD_FI void init_g(G& g, const DCard* s_cards, const double* wt) { g.cards = s_cards; g.wt = wt; }

// ---------------------------------------------------------------- thread-per-game kernels
// Stormbound.__init__ for one game: the working set of an all-zero record, dealt from `seed` with decks dk u8[2,n_deck]
// and factions fc u8[2] (k_reset and the environment kernels)
SBD_FI void new_game(G& g, unsigned long long seed, const u8* dk, int n_deck, const u8* fc) {
  __align__(16) SbState s;  // 128-bit moves
  uint4* z = reinterpret_cast<uint4*>(&s);
  for (int k = 0; k < SB_STATE_BYTES / 16; k++) z[k] = make_uint4(0, 0, 0, 0);
  unpack(g, s);
  g.seed_lo = (u32)seed; g.seed_hi = (u32)(seed >> 32);
  g.local_order = 0; g.current_order = 0; g.player_sign = 1; g.phase = PH_PLAY;
  for (int o = 0; o < 2; o++) {
    Ply& p = g.pl[o];
    p.max_mana = o == 0 ? 3 : 4; p.mana = p.max_mana; p.base = 20; p.front_line = o == 0 ? 4 : 0;
    p.replacable = 1; p.leftmost = 1; p.faction = fc[o]; p.n_hand = 0;
    i8 order[SB_DECK_MAX];
    int nd = n_deck < SB_DECK_MAX ? n_deck : SB_DECK_MAX;
    for (int k = 0; k < nd; k++) {  // a card id outside the table would index shared memory out of bounds: flag the game instead
      const int cid = dk[o * n_deck + k];
      if (cid <= 0 || cid >= SBC_COUNT) { GERR(g, SB_ERR_INDEX); order[k] = (i8)SBC_TOKEN_UNIT0; } else order[k] = (i8)cid;
    }
    shuffle(g, order, nd);  // player.py:28
    p.n_deck = (u8)nd;
    for (int k = 0; k < nd; k++) {  // player.py:30-32
      CardRec& c = p.deck[k];
      c.card = (u8)order[k]; c.cost = CARD(g, c.card).cost; c.flags = (CARD(g, c.card).flags & DCF_FIXED) ? SB_CF_FIXED : 0;
      c.link = -1; c.wn = (u16)k; c.xstr = 0;
    }
    player_fill_hand(g, o);  // player.py:35
  }
}
__global__ void __launch_bounds__(TPB_GAME) k_reset(int n, const unsigned long long* seeds, const u8* decks, int n_deck,
                                                    int decks_shared, const u8* factions, u8* states, const DCard* cards,
                                                    const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  new_game(g, seeds[i], decks + (decks_shared ? 0 : (size_t)i * 2 * n_deck), n_deck, factions + (decks_shared ? 0 : (size_t)i * 2));
  __align__(16) SbState s;  // 128-bit moves
  pack(g, s);
  store_state(states + (size_t)i * SB_STATE_BYTES, s);
}

// ---------------------------------------------------------------- deck generation (utils.py:26-241)
// One game per thread draws both decks from its own stream: philox(counter=(draw, generation, 0xDEC4, 0), key=seed).
// random.sample call shape of CPython 3.12: pool method while n <= setsize, else the rejection-set method.
struct DeckRng { u32 lo, hi, gen, draw; };
SBD_FI int deck_below(DeckRng& r, int n) {
  u32 w0, w1;
  philox(r.draw++, r.gen, 0xDEC4u, 0u, r.lo, r.hi, w0, w1);
  return (int)__umulhi(w0, (u32)n);
}
SBD_FI double deck_random(DeckRng& r) {
  u32 w0, w1;
  philox(r.draw++, r.gen, 0xDEC4u, 0u, r.lo, r.hi, w0, w1);
  return ((double)(w0 >> 5) * 67108864.0 + (double)(w1 >> 6)) / 9007199254740992.0;
}
#define POOL_W 80  // own faction + NEUTRAL: 70..74 of the 112 cards
SBD void py_sample(DeckRng& r, const u8* pop, int n, int k, u8* out) {
  int setsize = 21;
  if (k > 5) { int p = 1; while (p < 3 * k) p *= 4; setsize += p; }
  if (n <= setsize) {
    u8 pool[POOL_W];
    for (int i = 0; i < n; i++) pool[i] = pop[i];
    for (int i = 0; i < k; i++) { const int j = deck_below(r, n - i); out[i] = pool[j]; pool[j] = pool[n - i - 1]; }
  } else {
    u32 taken[(POOL_W + 31) / 32] = {0, 0, 0};
    for (int i = 0; i < k; i++) {
      int j = deck_below(r, n);
      while (taken[j >> 5] >> (j & 31) & 1u) j = deck_below(r, n);
      taken[j >> 5] |= 1u << (j & 31);
      out[i] = pop[j];
    }
  }
}
SBD void random_deck(DeckRng& r, const u8* pool, int n_pool, const u8* original, int n_preserve, u8* deck) {
  if (n_preserve >= 12) { for (int i = 0; i < 12; i++) deck[i] = original[i]; return; }
  if (n_preserve > 0) py_sample(r, original, 12, n_preserve, deck); else n_preserve = 0;
  py_sample(r, pool, n_pool, 12 - n_preserve, deck + n_preserve);
}
// pools: [5][POOL_W] card ids per faction (row 0 = NEUTRAL only), pool_n[5]; factions: per game [n][2] or one shared pair
struct ArchParams { u8 arch[24]; u8 fac[2]; };  // the two archetype decks and their factions travel as kernel arguments
__global__ void __launch_bounds__(128) k_generate_decks(int n, const unsigned long long* seeds, u32 generation, int mode, int n_preserve,
                                                       double q, const ArchParams ap, const u8* factions_d, int factions_shared,
                                                       const u8* pools, const int* pool_n, u8* decks, u8* factions_out) {
  const u8* archetypes = ap.arch;
  const u8* factions = factions_shared ? ap.fac : factions_d;
  __shared__ u8 s_pool[5 * POOL_W];
  __shared__ int s_pn[5];
  __shared__ u8 s_arch[24];
  for (int i = threadIdx.x; i < 5 * POOL_W; i += blockDim.x) s_pool[i] = pools[i];
  if (threadIdx.x < 5) s_pn[threadIdx.x] = pool_n[threadIdx.x];
  if (threadIdx.x < 24) s_arch[threadIdx.x] = archetypes[threadIdx.x];
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long seed = seeds[i];
  DeckRng r = {(u32)seed, (u32)(seed >> 32), generation, 0u};
  const u8* fc = factions + (factions_shared ? 0 : (size_t)i * 2);
  u8 d[24];
  bool keep[2] = {false, false};
  if (mode == 2) { keep[0] = deck_random(r) < q; keep[1] = deck_random(r) < q; }  // both drawn before any deck (utils.py:207-208)
  for (int o = 0; o < 2; o++) {
    const int f = fc[o] <= 4 ? fc[o] : 0;
    if (mode == 0 || (mode == 2 && keep[o])) { for (int k = 0; k < 12; k++) d[12 * o + k] = s_arch[12 * o + k]; }
    else random_deck(r, s_pool + f * POOL_W, s_pn[f], s_arch + 12 * o, mode == 1 ? n_preserve : 0, d + 12 * o);
  }
  for (int k = 0; k < 24; k++) decks[(size_t)i * 24 + k] = d[k];
  if (factions_out) { factions_out[(size_t)i * 2] = fc[0]; factions_out[(size_t)i * 2 + 1] = fc[1]; }
}

__global__ void __launch_bounds__(TPB_GAME) k_legal_mask(int n, const u8* states, u32* masks, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  load_state(s, states + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  u32 m[SB_MASK_WORDS];
  legal_mask(g, m);
  for (int k = 0; k < SB_MASK_WORDS; k++) masks[(size_t)i * SB_MASK_WORDS + k] = m[k];
}

// Stormbound.expert_action: only the stream position (and a possible error code) change in the record.
__global__ void __launch_bounds__(TPB_GAME) k_expert_action(int n, u8* states, u8* actions, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  load_state(s, states + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  actions[i] = (u8)expert_action(g);
  SbState* out = reinterpret_cast<SbState*>(states + (size_t)i * SB_STATE_BYTES);
  out->draw = g.draw;
  out->err = g.err;
}

template <bool DENSE>  // DENSE: compiled for 32 CTAs per SM (32 registers, 2,048 resident threads) for batches that fill the chip
__global__ void __launch_bounds__(TPB_GAME, DENSE ? 32 : 1) k_step(int n, u8* states, const u8* actions, i8* reward, u8* done, u8* err,
                                                   u32* next_masks, const DCard* cards, const double* wt, int gpw) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  // gpw games per warp on consecutive lanes, like the rollout kernel: small batches spread over more warps / SMs
  const int lane = threadIdx.x & 31;
  const int i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * gpw + lane;
  if (lane >= gpw || i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  load_state(s, states + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  game_step(g, actions[i]);
  pack(g, s);
  store_state(states + (size_t)i * SB_STATE_BYTES, s);
  if (reward) reward[i] = (g.done & SB_REWARD) ? 1 : 0;
  if (done) done[i] = (g.done & SB_DONE) ? 1 : 0;
  if (err) err[i] = s.err;
  if (next_masks) {
    u32 m[SB_MASK_WORDS];
    legal_mask(g, m);
    for (int k = 0; k < SB_MASK_WORDS; k++) next_masks[(size_t)i * SB_MASK_WORDS + k] = m[k];
  }
}

__global__ void __launch_bounds__(TPB_GAME) k_observe(int n, const u8* states, int* obs, u8* err, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  load_state(s, states + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  int e = observe(g, obs + (size_t)i * SB_OBS_INTS);
  if (err) err[i] = (u8)e;
}

__global__ void __launch_bounds__(TPB_GAME) k_features(int n, const u8* states, double* feat, u8* err, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  load_state(s, states + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  scan_badobs(g);
  double f[SB_N_FEATURES];
  int e = features(g, f);
  for (int k = 0; k < SB_N_FEATURES; k++) feat[(size_t)i * SB_N_FEATURES + k] = f[k];
  if (err) err[i] = (u8)e;
}

// whole uniform-random rollout in one launch; HBM is touched once on the way in and once on the way out.
//
// Turn-synchronous warp schedule.  A game alternates "a few non-PASS actions, then PASS"; the PASS step
// (flip, refill with FP64 draws, front lines, turn-start structures, every unit's move) carries most of the
// instructions.  Lanes therefore do NOT step in lock-step by step index: phase A lets every lane play its
// non-PASS actions (lanes already at their PASS wait), phase B executes the PASS of all 32 lanes together.
// Games are independent, so the order is free; what changes is that the long PASS pipeline is entered
// converged (one instruction stream per warp instead of one per lane group), which is what the ncu profile
// of the lock-step version asked for: 2.6-3.0 of 32 lanes active, 73 % of stall samples = instruction fetch.
SBD_FI int pick_action(const G& g) {
  u32 m[SB_MASK_WORDS];
  int nl = legal_mask(g, m);
  int pick = (int)agent_pick(g.seed_lo, g.seed_hi, g.steps, (u32)nl);
#pragma unroll 1
  for (int w = 0; w < SB_MASK_WORDS; w++) {  // pick-th set bit
    int c = __popc(m[w]);
    if (pick < c) { u32 v = m[w]; for (int q = 0; q < pick; q++) v &= v - 1; return w * 32 + __ffs(v) - 1; }
    pick -= c;
  }
  return SB_ACTION_PASS;
}
// TPB / BSYNC: with BSYNC the two phases are separated by CTA-wide votes (__syncthreads_or) instead of
// warp votes, so all TPB/32 warps of a CTA walk the PASS pipeline at the same time and share the
// instruction-cache lines they fetch (the saturated kernel is instruction-fetch bound).
template <bool DIGEST, int TPB, bool BSYNC, int MINB = 1>
__global__ void __launch_bounds__(TPB, MINB) k_rollout_random(int n, u8* states, int max_steps, int* steps_out,
                                                        unsigned long long* chain, const DCard* cards, const double* wt,
                                                        int gpw, int turn_sync, int* queue) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  // gpw games per warp on CONSECUTIVE lanes (32 = plain thread per game).  Fewer games per warp = fewer
  // divergent paths serialised on one scheduler slot when the batch is small; consecutive lanes keep the
  // 32-byte local-memory sectors of the thread-private working set dense.  All 32 lanes stay in the kernel
  // (full-mask votes below); lanes without a game just never become `alive`.
  // queue != nullptr (batches larger than the resident lanes): a lane whose game ended takes the next game
  // index from a global counter instead of idling until the longest game of its CTA is over.
  const unsigned FULL = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  int i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * gpw + lane;
  bool has_game = !queue && lane < gpw && i < n;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  unsigned long long ch = 0ull;
  int k = 0;
  bool alive = false;
  if (has_game) {
    load_state(s, states + (size_t)i * SB_STATE_BYTES);
    unpack(g, s);
    if (DIGEST) ch = chain[i];
    alive = !(g.done & SB_DONE) && !g.err && max_steps > 0;
  }
  if (!turn_sync) {  // lock-step by step index (kept for A/B measurements)
    while (alive) {
      game_step(g, pick_action(g));
      end_of_step(g);
      if (DIGEST) { pack(g, s); ch = (ch ^ digest_state(s)) * 0x100000001B3ull; }
      k++;
      alive = !(g.done & SB_DONE) && !g.err && k < max_steps;
    }
  } else {
    bool at_pass = false;
    bool dry = queue == nullptr;  // no more games to take
    for (;;) {
      if (!dry) {  // warp-converged here (after the vote at the bottom of the previous round)
        const unsigned want = __ballot_sync(FULL, !alive);
        if (want) {
          int base = 0;
          if (lane == 0) base = atomicAdd(queue, __popc(want));
          base = __shfl_sync(FULL, base, 0);
          if (!alive) {
            if (has_game) {  // retire the finished game
              pack(g, s);
              store_state(states + (size_t)i * SB_STATE_BYTES, s);
              if (steps_out) steps_out[i] = k;
              if (DIGEST) chain[i] = ch;
              has_game = false;
            }
            i = base + __popc(want & ((1u << lane) - 1u));
            if (i < n) {
              has_game = true;
              load_state(s, states + (size_t)i * SB_STATE_BYTES);
              unpack(g, s);
              ch = DIGEST ? chain[i] : 0ull;
              k = 0;
              at_pass = false;
              alive = !(g.done & SB_DONE) && !g.err && max_steps > 0;
            }
          }
          dry = base + __popc(want) >= n;  // warp-uniform
        }
      }
      if (!(BSYNC ? __syncthreads_or(alive) : __any_sync(FULL, alive))) break;
      for (;;) {  // phase A: non-PASS actions
        int a = -1;
        if (alive && !at_pass) {
          a = pick_action(g);
          if (a == SB_ACTION_PASS) { at_pass = true; a = -1; }
        }
        // CTA-wide vote per round in CTA-synchronous mode: measured against warp votes + one barrier per turn
        // (tools/sweep_phase.py, removed): the shared instruction stream is worth more than the barrier waits (343 vs 300 M)
        if (!(BSYNC ? __syncthreads_or(a >= 0) : __any_sync(FULL, a >= 0))) break;
        if (a >= 0) {
          game_step(g, a);
          end_of_step(g);
          if (DIGEST) { pack(g, s); ch = (ch ^ digest_state(s)) * 0x100000001B3ull; }
          k++;
          alive = !(g.done & SB_DONE) && !g.err && k < max_steps;
        }
      }
      if (alive && at_pass) {  // phase B: everybody's PASS, converged
        game_step(g, SB_ACTION_PASS);
        end_of_step(g);
        if (DIGEST) { pack(g, s); ch = (ch ^ digest_state(s)) * 0x100000001B3ull; }
        k++;
        at_pass = false;
        alive = !(g.done & SB_DONE) && !g.err && k < max_steps;
      }
    }
  }
  if (has_game) {
    pack(g, s);
    store_state(states + (size_t)i * SB_STATE_BYTES, s);
    if (steps_out) steps_out[i] = k;
    if (DIGEST) chain[i] = ch;
  }
}

// ---------------------------------------------------------------- warp-per-game kernels (heuristic agent)
struct Best { double score; int action; };
SBD_FI Best warp_argmax(Best b) {  // np.argmax: first maximum = lowest action id among equal scores
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    double os = __shfl_xor_sync(0xFFFFFFFFu, b.score, off);
    int oa = __shfl_xor_sync(0xFFFFFFFFu, b.action, off);
    bool take = oa >= 0 && (b.action < 0 || os > b.score || (os == b.score && oa < b.action));
    if (take) { b.score = os; b.action = oa; }
  }
  return b;
}
SBD_FI double score_delta(const double* w, const double* fc, const double* fn) {  // evo/heuristic_agent.py:23-51,82-122
  double d = 0.0;
#pragma unroll
  // np.dot at n = 10 is OpenBLAS's scalar tail loop with FMA contraction: sequential fused multiply-add
  for (int i = 0; i < SB_N_FEATURES; i++) d = __fma_rn(w[i], __dsub_rn(fn[i], fc[i]), d);
  double eff = __dsub_rn(fn[0], fc[0]);
  double rp = eff < -0.3 ? __dmul_rn(fabs(eff), 0.2) : 0.0;
  return __dsub_rn(__dsub_rn(-d, d), rp);
}
// The base state of a decision is either the packed 512-byte record (k_select_action: states come from the caller
// one decision at a time) or a raw image of the working set G kept in shared memory for the whole game
// (k_rollout_heuristic).  The image avoids the pack / unpack of every decision: ncu on the packed version showed
// unpack 18 % and pack 14 % (one lane) of all warp instructions.  copy_g moves the live parts 64 bits at a time:
// the entity pool up to n_ent, the block [board .. strc] and the Temple-of-Time memories up to n_mem; the trigger
// stack is empty between steps and the table pointers belong to each copy.
SBD_NI void copy_g(G& dst, const G& src) {
  typedef unsigned long long u64;
  static_assert(offsetof(G, board) % 8 == 0 && offsetof(G, trig) % 8 == 0 && sizeof(Ent) % 8 == 0 && sizeof(Mem) % 8 == 0, "copy_g layout");
  static_assert(offsetof(G, pl) % 8 == 0 && sizeof(Ply) % 8 == 0 && offsetof(Ply, deck) % 8 == 0 && sizeof(CardRec) == 8, "copy_g layout");
  const u64* s8 = reinterpret_cast<const u64*>(&src);
  u64* d8 = reinterpret_cast<u64*>(&dst);
  const int ne = src.n_ent * (int)(sizeof(Ent) / 8);
  #pragma unroll 4
  for (int i = 0; i < ne; i++) d8[i] = s8[i];
  // the block [board .. trig) without the unused tails of the two deck arrays (a deck holds 8-12 of its 20 slots; slots
  // beyond n_deck are never read before they are written): board + player 0 up to its last deck card, player 1 likewise,
  // then the scalars behind the players
  const int p0 = (int)(offsetof(G, pl) / 8), pw = (int)(sizeof(Ply) / 8), dk = (int)(offsetof(Ply, deck) / 8);
  const int e0 = p0 + dk + src.pl[0].n_deck, e1 = p0 + pw + dk + src.pl[1].n_deck;
  #pragma unroll 4
  for (int i = (int)(offsetof(G, board) / 8); i < e0; i++) d8[i] = s8[i];
  #pragma unroll 4
  for (int i = p0 + pw; i < e1; i++) d8[i] = s8[i];
  #pragma unroll
  for (int i = p0 + 2 * pw; i < (int)(offsetof(G, trig) / 8); i++) d8[i] = s8[i];
  const int m0 = (int)(offsetof(G, mem) / 8), nm = src.n_mem * (int)(sizeof(Mem) / 8);
  #pragma unroll 1
  for (int i = 0; i < nm; i++) d8[m0 + i] = s8[m0 + i];
}
SBD_FI void base_load(G& g, const SbState& b) { unpack(g, b); scan_badobs(g); }
SBD_FI void base_store(SbState& b, G& g) { pack(g, b); }
SBD_FI void base_load(G& g, const G& b) { copy_g(g, b); }
SBD_FI void base_store(G& b, G& g) { end_of_step(g); copy_g(b, g); }  // same lazy compaction / overflow rules as the random rollout

// One decision for the game whose base state sits in shared memory.  Every lane forks the base,
// applies its candidate(s), scores them; returns the warp-wide best action.  If `commit`, the lane that
// owns the winner leaves the post-action state packed in `base` (the fork becomes the game).
template <class Base>
SBD_NI int decide(G& g, Base* base, const double* w, double* scores_out, bool commit) {
  const int lane = threadIdx.x & 31;
  base_load(g, *base);
  u32 m[SB_MASK_WORDS];
  legal_mask(g, m);
  double fc[SB_N_FEATURES], fn[SB_N_FEATURES];
  Best best; best.score = 0.0; best.action = -1;
  int last = -1;
  bool dirty = false;
  int n_legal = 0;
#pragma unroll
  for (int i = 0; i < SB_MASK_WORDS; i++) n_legal += __popc(m[i]);
  const int cur_err = (n_legal > 1 || scores_out) ? features(g, fc) : 0;
  // Round r gives lane l the (32 r + l)-th legal action.  The trip count is uniform over the warp, so all
  // lanes enter game_step/features TOGETHER (the first version walked the 156 action ids per lane and
  // reached the fork at different iterations: ncu showed 1.00 thread per instruction in every step function).
#pragma unroll 1
  for (int r = 0; r * 32 < n_legal; r++) {
    int k = r * 32 + lane, a = -1;
    if (k < n_legal) {
#pragma unroll 1
      for (int wd = 0; wd < SB_MASK_WORDS; wd++) {
        int c = __popc(m[wd]);
        if (k < c) { u32 v = m[wd]; for (int q = 0; q < k; q++) v &= v - 1; a = wd * 32 + __ffs(v) - 1; break; }
        k -= c;
      }
    }
    if (a < 0) continue;
    if (n_legal == 1 && !scores_out) { best.score = 0.0; best.action = a; break; }  // forced move: argmax of one
    if (dirty) base_load(g, *base);
    game_step(g, a);
    end_of_step(g);  // a candidate that leaves more than the packed layout holds is an engine status, like for the state that gets committed
    dirty = true; last = a;
    double sc = 0.0;
    int nerr = g.err;
    if (!nerr) nerr = features(g, fn);
    if (!nerr && !cur_err) sc = score_delta(w, fc, fn);
    if (scores_out) scores_out[a] = sc;
    if (best.action < 0 || sc > best.score) { best.score = sc; best.action = a; }
  }
  Best win = warp_argmax(best);
  int action = win.action < 0 ? SB_ACTION_PASS : win.action;
  if (commit) {
    __syncwarp();  // everybody is done reading the base
    bool owner = (win.action >= 0) ? (best.action == win.action) : (lane == 0);
    if (owner) {
      if (last != action) { base_load(g, *base); game_step(g, action); }
      base_store(*base, g);
    }
    __syncwarp();
  }
  return action;
}

__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_select_action(int n, const u8* states, const double* weights, u8* actions,
                                                                      double* scores, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  __shared__ __align__(16) SbState s_base[WARPS_PER_CTA];
  stage_cards(s_cards, cards);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gi = blockIdx.x * WARPS_PER_CTA + warp;
  if (gi >= n) return;
  reinterpret_cast<uint4*>(&s_base[warp])[lane] = reinterpret_cast<const uint4*>(states + (size_t)gi * SB_STATE_BYTES)[lane];
  __syncwarp();
  if (scores) for (int a = lane; a < SB_N_ACTIONS; a += 32) scores[(size_t)gi * SB_N_ACTIONS + a] = __longlong_as_double(0x7FF8000000000000ll);
  __syncwarp();
  G g;
  init_g(g, s_cards, wt);
  double w[SB_N_FEATURES];
  for (int k = 0; k < SB_N_FEATURES; k++) w[k] = weights[(size_t)gi * SB_N_FEATURES + k];
  int a = decide(g, &s_base[warp], w, scores ? scores + (size_t)gi * SB_N_ACTIONS : nullptr, false);
  if (lane == 0) actions[gi] = (u8)a;
}

// WPC warps (games) per CTA.  BSYNC: all warps of the CTA take their decisions in step (CTA-wide vote per
// decision), so they walk fork/step/features at the same time and share instruction-cache lines.
// queue != nullptr (independent warps only): persistent grid; a warp whose game is over takes the next game index from
// a global counter, so a CTA slot never idles while its longest game finishes (games differ 3x in length; ncu showed
// 72 % active warps with one game per warp and CTA) and CTAs can be large enough to share one card table.
template <int WPC, bool BSYNC>
__global__ void __launch_bounds__(WPC * 32, BSYNC ? 1 : (HEUR_MIN_CTAS * 4) / WPC) k_rollout_heuristic(int n, u8* states, const double* w_first, const double* w_second,
                                                                const int* idx_first, const int* idx_second, int max_steps,
                                                                i8* result, int* steps_out, const DCard* cards, const double* wt, int* queue) {
  __shared__ DCard s_cards[SBC_COUNT];
  extern __shared__ __align__(16) unsigned char s_dyn[];  // WPC working-set images (sizeof(G) each)
  G* s_base = reinterpret_cast<G*>(s_dyn);
  stage_cards(s_cards, cards);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  G* base = &s_base[warp];
  G g;
  init_g(g, s_cards, wt);
  double wf[SB_N_FEATURES], ws[SB_N_FEATURES];
  int gi = blockIdx.x * WPC + warp;
  #pragma unroll 1
  for (;;) {
    if (!BSYNC && queue) {
      if (lane == 0) gi = atomicAdd(queue, 1);
      gi = __shfl_sync(0xFFFFFFFFu, gi, 0);
    }
    const bool has_game = gi < n;
    if (!BSYNC && !has_game) return;
    if (has_game) {
      if (lane == 0) {  // packed record -> working set -> shared image, once per game
        __align__(16) SbState s;
        load_state(s, states + (size_t)gi * SB_STATE_BYTES);
        unpack(g, s);
        scan_badobs(g);
        copy_g(*base, g);
      }
      // a seat without a weight table is played by the scripted opponent (Stormbound.expert_action)
      if (w_first) {
        const double* pf = w_first + (size_t)(idx_first ? idx_first[gi] : gi) * SB_N_FEATURES;
        for (int k = 0; k < SB_N_FEATURES; k++) wf[k] = pf[k];
      }
      if (w_second) {
        const double* ps = w_second + (size_t)(idx_second ? idx_second[gi] : gi) * SB_N_FEATURES;
        for (int k = 0; k < SB_N_FEATURES; k++) ws[k] = ps[k];
      }
    }
    __syncwarp();
    int k = 0, res = -1;
    bool alive = has_game;
    for (;;) {
      if (alive && (k >= max_steps || base->pl[0].base < 0 || base->pl[1].base < 0)) alive = false;
      if (BSYNC) { if (!__syncthreads_or(alive)) break; } else if (!alive) break;
      if (alive) {
        const bool first_to_move = base->player_sign == 1;
        if (first_to_move ? w_first != nullptr : w_second != nullptr) decide(g, base, first_to_move ? wf : ws, nullptr, true);
        else {  // expert_action draws from the game's own stream, then the action is stepped (games/stormbound.py:563-637)
          if (lane == 0) {
            copy_g(g, *base);
            const int a = expert_action(g);
            game_step(g, a);
            base_store(*base, g);
          }
          __syncwarp();
        }
        k++;
        if (base->err) { res = -2; alive = false; }
      }
    }
    if (has_game) {
      if (res != -2) {
        bool l0 = base->pl[0].base < 0, l1 = base->pl[1].base < 0;
        res = (l1 && !l0) ? 0 : (l0 && !l1) ? 1 : -1;
      }
      __syncwarp();
      if (lane == 0) {
        __align__(16) SbState s;
        copy_g(g, *base);
        pack(g, s);
        store_state(states + (size_t)gi * SB_STATE_BYTES, s);
        if (result) result[gi] = (i8)res;
        if (steps_out) steps_out[gi] = k;
      }
    }
    if (BSYNC || !queue) return;
    __syncwarp();  // the image is free for the next game
  }
}

// ---------------------------------------------------------------- heuristic rollout, K games per warp
// The kernel above gives a whole warp to one game: a decision offers 18.6 candidates on average (oracle statistics over
// default-deck games: median 16, 20 % of the decisions forced), so 40 % of the lanes have nothing to fork, every lane still
// copies the base and recomputes the legal mask and the base features, and 2,048 resident threads per SM at 32 registers
// spill into the same local memory the forks live in.  Here a warp owns K games.  Lane q < K is the OWNER of slot q: it
// loads / retires the game, computes its legal mask and base features once (shared memory), and applies the chosen action.
// The candidates of all K games are numbered consecutively and dealt to the 32 lanes round by round, so the lanes are
// busy whatever the games' candidate counts are; the arg-max is a segmented warp reduction (first maximum = lowest action
// id, like np.argmax).  The winner is re-applied to the base by the owner lane (one extra step per decision instead of
// keeping 32 forks alive).  A quarter of the threads for the same number of games in flight: 3-4x the registers per
// thread and a quarter of the call frames.  Same results as k_rollout_heuristic, game for game.
struct __align__(8) PSlot { double w[2][SB_N_FEATURES]; double fc[SB_N_FEATURES]; u32 mask[SB_MASK_WORDS]; int cerr, seat, fc_valid, n_legal; };  // n_legal >= 0: mask is this decision's legal set
// The base state of a slot between decisions, in shared memory: what copy_g moves, stored WITHOUT the unused pool slots (a
// base has at most 20 entities: end_of_step compacts beyond that, unpack creates at most that): 1.2 KB instead of the 1.9 KB of
// a whole G, so that twice the warps fit an SM.  The block [board .. trig) keeps G's layout: `view()` reads its scalars in place.
#define IMG_BLOCK ((int)(offsetof(G, trig) - offsetof(G, board)))
struct __align__(8) Img {
  unsigned char block[IMG_BLOCK];
  Ent e[SB_N_TILES];
  Mem mem[NMEM];
  SBD_FI const G& view() const { return *reinterpret_cast<const G*>(block - offsetof(G, board)); }  // fields of [board .. trig) only
};
#define PACK_BYTES(K) ((int)((K) * (sizeof(Img) + sizeof(PSlot))))
SBD_NI void img_store(Img& dst, const G& src) {  // src.n_ent <= 20 (after end_of_step / unpack)
  typedef unsigned long long u64;
  static_assert(IMG_BLOCK % 8 == 0 && offsetof(Img, e) % 8 == 0 && offsetof(Img, mem) % 8 == 0, "Img layout");
  const u64* s8 = reinterpret_cast<const u64*>(&src);
  u64* blk = reinterpret_cast<u64*>(dst.block) - offsetof(G, board) / 8;  // blk[i] is word i of a G
  const int p0 = (int)(offsetof(G, pl) / 8), pw = (int)(sizeof(Ply) / 8), dk = (int)(offsetof(Ply, deck) / 8);
  const int e0 = p0 + dk + src.pl[0].n_deck, e1 = p0 + pw + dk + src.pl[1].n_deck;
#pragma unroll 4
  for (int i = (int)(offsetof(G, board) / 8); i < e0; i++) blk[i] = s8[i];
#pragma unroll 4
  for (int i = p0 + pw; i < e1; i++) blk[i] = s8[i];
#pragma unroll
  for (int i = p0 + 2 * pw; i < (int)(offsetof(G, trig) / 8); i++) blk[i] = s8[i];
  u64* d8 = reinterpret_cast<u64*>(dst.e);
  const int ne = (src.n_ent < SB_N_TILES ? src.n_ent : SB_N_TILES) * (int)(sizeof(Ent) / 8);
#pragma unroll 4
  for (int i = 0; i < ne; i++) d8[i] = s8[i];
  u64* m8 = reinterpret_cast<u64*>(dst.mem);
  const int m0 = (int)(offsetof(G, mem) / 8), nm = src.n_mem * (int)(sizeof(Mem) / 8);
#pragma unroll 1
  for (int i = 0; i < nm; i++) m8[i] = s8[m0 + i];
}
SBD_NI void img_load(G& dst, const Img& src) {
  typedef unsigned long long u64;
  u64* d8 = reinterpret_cast<u64*>(&dst);
  const G& v = src.view();
  const u64* blk = reinterpret_cast<const u64*>(src.block) - offsetof(G, board) / 8;
  const int p0 = (int)(offsetof(G, pl) / 8), pw = (int)(sizeof(Ply) / 8), dk = (int)(offsetof(Ply, deck) / 8);
  const int e0 = p0 + dk + v.pl[0].n_deck, e1 = p0 + pw + dk + v.pl[1].n_deck;
#pragma unroll 4
  for (int i = (int)(offsetof(G, board) / 8); i < e0; i++) d8[i] = blk[i];
#pragma unroll 4
  for (int i = p0 + pw; i < e1; i++) d8[i] = blk[i];
#pragma unroll
  for (int i = p0 + 2 * pw; i < (int)(offsetof(G, trig) / 8); i++) d8[i] = blk[i];
  const u64* s8 = reinterpret_cast<const u64*>(src.e);
  const int ne = v.n_ent * (int)(sizeof(Ent) / 8);
#pragma unroll 4
  for (int i = 0; i < ne; i++) d8[i] = s8[i];
  const u64* m8 = reinterpret_cast<const u64*>(src.mem);
  const int m0 = (int)(offsetof(G, mem) / 8), nm = v.n_mem * (int)(sizeof(Mem) / 8);
#pragma unroll 1
  for (int i = 0; i < nm; i++) d8[m0 + i] = m8[i];
}
SBD_FI void img_commit(Img& b, G& g) { end_of_step(g); img_store(b, g); }  // same lazy compaction / overflow rules as the random rollout
SBD_FI int nth_action(const u32* m, int k) {
#pragma unroll 1
  for (int wd = 0; wd < SB_MASK_WORDS; wd++) {
    const int c = __popc(m[wd]);
    if (k < c) { u32 v = m[wd]; for (int q = 0; q < k; q++) v &= v - 1; return wd * 32 + __ffs(v) - 1; }
    k -= c;
  }
  return SB_ACTION_PASS;
}
// once per game, out of line: keeps the decision loop's instruction lines dense
SBD_NI void slot_retire(G& g, const Img& b, u8* record) {
  __align__(16) SbState s;
  img_load(g, b);
  pack(g, s);
  store_state(record, s);
}
SBD_NI void slot_load(G& g, Img& b, PSlot& me, const u8* record, const double* pf, const double* pw) {
  __align__(16) SbState s;
  load_state(s, record);
  unpack(g, s);
  scan_badobs(g);
  img_store(b, g);
  if (pf) for (int k = 0; k < SB_N_FEATURES; k++) me.w[0][k] = pf[k];
  if (pw) for (int k = 0; k < SB_N_FEATURES; k++) me.w[1][k] = pw[k];
}
template <int K, int WPC, int MINB>
__global__ void __launch_bounds__(WPC * 32, MINB) k_rollout_heuristic_packed(int n, u8* states, const double* w_first, const double* w_second,
                                                                             const int* idx_first, const int* idx_second, int max_steps, i8* result,
                                                                             int* steps_out, const DCard* cards, const double* wt, int* queue) {
  __shared__ DCard s_cards[SBC_COUNT];
  extern __shared__ __align__(16) unsigned char s_dyn[];
  stage_cards(s_cards, cards);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Img* base = reinterpret_cast<Img*>(s_dyn + (size_t)warp * PACK_BYTES(K));
  PSlot* ps = reinterpret_cast<PSlot*>(base + K);
  G g;
  init_g(g, s_cards, wt);
  const bool owner = lane < K;
  Img& b = base[owner ? lane : 0];
  const G& bv = b.view();
  PSlot& me = ps[owner ? lane : 0];
  int gi = -1, steps = 0;
  bool alive = false, aborted = false, exhausted = false;
#pragma unroll 1
  for (;;) {
    // ---- owner lanes: retire a finished game, take the next one from the queue
    if (owner) {
#pragma unroll 1
      for (;;) {
        if (alive) {
          const bool l0 = bv.pl[0].base < 0, l1 = bv.pl[1].base < 0;
          if (!(aborted || steps >= max_steps || l0 || l1)) break;
          slot_retire(g, b, states + (size_t)gi * SB_STATE_BYTES);
          if (result) result[gi] = (i8)(aborted ? -2 : (l1 && !l0) ? 0 : (l0 && !l1) ? 1 : -1);
          if (steps_out) steps_out[gi] = steps;
          alive = false;
        }
        if (exhausted) break;
        gi = atomicAdd(queue, 1);
        if (gi >= n) { exhausted = true; break; }
        slot_load(g, b, me, states + (size_t)gi * SB_STATE_BYTES, w_first ? w_first + (size_t)(idx_first ? idx_first[gi] : gi) * SB_N_FEATURES : nullptr,
                  w_second ? w_second + (size_t)(idx_second ? idx_second[gi] : gi) * SB_N_FEATURES : nullptr);
        me.fc_valid = 0; me.n_legal = -1;
        steps = 0; aborted = false; alive = true;
      }
    }
    if (!__ballot_sync(0xFFFFFFFFu, owner && alive)) break;
    // ---- phase 1, owner lanes: legal set and base features of the slot's decision
    int n_cand = 0, forced = -1;
    bool expert = false;
    if (owner && alive) {
      const bool first = bv.player_sign == 1;
      expert = first ? (w_first == nullptr) : (w_second == nullptr);
      if (!expert) {
        int n_legal = me.n_legal;  // >= 0: left, with the mask, by the lane that committed the last action
        const bool need_fc = !me.fc_valid;
        if (n_legal < 0 || need_fc) img_load(g, b);
        if (n_legal < 0) {
          u32 m[SB_MASK_WORDS];
          legal_mask(g, m);
          n_legal = 0;
#pragma unroll
          for (int i = 0; i < SB_MASK_WORDS; i++) { n_legal += __popc(m[i]); me.mask[i] = m[i]; }
        }
        me.seat = first ? 0 : 1;
        if (n_legal > 1) {
          if (need_fc) {  // else: the committed fork's features (same mover, same perspective)
            double fc[SB_N_FEATURES];
            me.cerr = features(g, fc);
#pragma unroll
            for (int i = 0; i < SB_N_FEATURES; i++) me.fc[i] = fc[i];
          }
          n_cand = n_legal;
        } else forced = n_legal == 1 ? nth_action(me.mask, 0) : SB_ACTION_PASS;  // forced move: argmax of one (none: PASS)
      }
    }
    __syncwarp();
    // ---- phase 2: the candidates of all slots, numbered consecutively, 32 per round
    int incl = n_cand;
#pragma unroll
    for (int off = 1; off < K; off <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, off); if (lane >= off) incl += t; }
    const int total = __shfl_sync(0xFFFFFFFFu, incl, K - 1);
    const int excl = incl - n_cand;
    Best mine; mine.score = 0.0; mine.action = -1;
    int held_k = -1, held_a = -1, held_err = 1;  // the fork this lane still holds after the rounds (its last candidate)
    double fn[SB_N_FEATURES];
#pragma unroll 1
    for (int r0 = 0; r0 < total; r0 += 32) {
      const int c = r0 + lane;
      int k = -1, j = 0;
#pragma unroll
      for (int q = 0; q < K; q++) {
        const int e = __shfl_sync(0xFFFFFFFFu, excl, q), nc = __shfl_sync(0xFFFFFFFFu, n_cand, q);
        if (c >= e && c < e + nc) { k = q; j = c - e; }
      }
      double sc = 0.0;
      int a = -1;
      if (k >= 0) {
        const PSlot& p = ps[k];
        a = nth_action(p.mask, j);
        img_load(g, base[k]);
        game_step(g, a);
        end_of_step(g);  // a candidate that leaves more than the packed layout holds is an engine status, like for the state that gets committed
        int nerr = g.err;
        if (!nerr) nerr = features(g, fn);
        if (!nerr && !p.cerr) sc = score_delta(p.w[p.seat], p.fc, fn);
        held_k = k; held_a = a; held_err = nerr;
      }
      // segmented arg-max: one warp reduction per slot present in this round; the owner keeps the first maximum
#pragma unroll
      for (int q = 0; q < K; q++) {
        const int e = __shfl_sync(0xFFFFFFFFu, excl, q), nc = __shfl_sync(0xFFFFFFFFu, n_cand, q);
        if (nc == 0 || e + nc <= r0 || e >= r0 + 32) continue;  // uniform
        Best t;
        t.score = k == q ? sc : 0.0;
        t.action = k == q ? a : -1;
        t = warp_argmax(t);
        if (lane == q && t.action >= 0 && (mine.action < 0 || t.score > mine.score)) mine = t;
      }
    }
    // ---- phase 3: ONE lane per slot ends up with the post-action state in its private working set -- the lane that still
    // holds the winner's fork, else the owner lane (forced and expert moves, winners of an earlier round) after applying the
    // action to a fresh copy of the base.  That lane commits the state and, while it has it at hand, prepares the slot's next
    // decision: legal set and base features (the fork's own features when the same seat moves again).
    int chosen = -1;
    if (owner && alive && !expert) chosen = forced >= 0 ? forced : (mine.action < 0 ? SB_ACTION_PASS : mine.action);
    const int want = __shfl_sync(0xFFFFFFFFu, chosen, held_k < 0 ? 0 : held_k);  // the action slot held_k plays
    const bool scored = __shfl_sync(0xFFFFFFFFu, (int)(n_cand > 0), held_k < 0 ? 0 : held_k) != 0;
    // a candidate appears once per decision: at most one lane per slot.  An owner lane may hold its own slot's winner only: it
    // may have to apply that slot's action itself below
    bool holder = held_k >= 0 && scored && held_a == want && (lane >= K || held_k == lane);
    u32 done_slots = 0;
#pragma unroll
    for (int q = 0; q < K; q++) if (__ballot_sync(0xFFFFFFFFu, holder && held_k == q)) done_slots |= 1u << q;
    bool have_fn = holder && !held_err;
    if (owner && alive && !((done_slots >> lane) & 1u)) {
      img_load(g, b);
      held_a = expert ? expert_action(g) : chosen;
      game_step(g, held_a);
      held_k = lane; holder = true; have_fn = false;
    }
    if (holder) {
      PSlot& p = ps[held_k];
      img_commit(base[held_k], g);
      p.n_legal = -1; p.fc_valid = 0;
      const bool next_first = g.player_sign == 1;
      if (!g.err && (next_first ? w_first != nullptr : w_second != nullptr)) {
        u32 m[SB_MASK_WORDS];
        legal_mask(g, m);
        int nl = 0;
#pragma unroll
        for (int i = 0; i < SB_MASK_WORDS; i++) { nl += __popc(m[i]); p.mask[i] = m[i]; }
        p.n_legal = nl;
        if (nl > 1) {
          if (!(have_fn && held_a != SB_ACTION_PASS)) p.cerr = features(g, fn); else p.cerr = 0;
#pragma unroll
          for (int i = 0; i < SB_N_FEATURES; i++) p.fc[i] = fn[i];
          p.fc_valid = 1;
        }
      }
    }
    __syncwarp();
    if (owner && alive) {
      steps++;
      if (bv.err) aborted = true;
    }
  }
}

// ---------------------------------------------------------------- batched environment (sb_env_reset / sb_env_step)
// One call moves every env from "the learner is to move" to "the learner is to move" again: check and apply the learner's
// action, let the opponent play, close a finished episode and deal the next one in place, then emit observation and legal
// mask.  Opponent kinds: 0 none (self-play), 1 uniform-random legal agent (the stream of k_rollout_random), 2 expert_action,
// 3 heuristic agent (k_env_step_heur).  Episode end and result codes are those of k_rollout_heuristic.
struct EnvArgs {
  int n;
  u8* states;
  const unsigned long long* seeds;  // non-null: sb_env_reset (deal from these seeds), null: sb_env_step (apply actions)
  const u8* actions;
  const u8* decks; int n_deck; int decks_shared; const u8* factions;
  int opponent; const u8* seat; const double* w_opp; const int* idx_opp; int max_steps;
  i8* result; int* length; u8* final_states; int* obs; u32* masks; u8* obs_err;
};
#define ENV_CONTINUES (-3)
#define ENV_REJECTED (-4)
// seed of an env's next episode from the Philox key of the finished one (splitmix64 finaliser, 63 bits)
SBD_FI unsigned long long env_next_seed(unsigned long long s) {
  unsigned long long z = s + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z & 0x7FFFFFFFFFFFFFFFull;
}
SBD_FI unsigned long long env_key(const G& g) { return ((unsigned long long)g.seed_hi << 32) | g.seed_lo; }
SBD_FI bool env_over(const G& g, int max_steps) { return g.pl[0].base < 0 || g.pl[1].base < 0 || g.err || (int)g.steps >= max_steps; }
SBD_FI int env_result(const G& g) {
  if (g.err) return -2;
  const bool l0 = g.pl[0].base < 0, l1 = g.pl[1].base < 0;
  return (l1 && !l0) ? 0 : (l0 && !l1) ? 1 : -1;
}
SBD_FI bool env_learner_moves(const G& g, const EnvArgs& a, int seat) { return a.opponent == 0 || (g.player_sign == 1 ? 0 : 1) == seat; }
SBD_FI const u8* env_deck(const EnvArgs& a, int i) { return a.decks + (a.decks_shared ? 0 : (size_t)i * 2 * a.n_deck); }
SBD_FI const u8* env_factions(const EnvArgs& a, int i) { return a.factions + (a.decks_shared ? 0 : (size_t)i * 2); }
// a fresh game as sb_reset writes it, and the working set as the next sb_* call would unpack it from that record
SBD_FI void env_deal(G& g, SbState& s, const EnvArgs& a, int i, unsigned long long seed) {
  new_game(g, seed, env_deck(a, i), a.n_deck, env_factions(a, i));
  pack(g, s);
  unpack(g, s);
}
SBD_FI bool env_legal(const u32* m, int action) { return action < SB_N_ACTIONS && (m[action >> 5] >> (action & 31) & 1u); }
SBD_FI void env_outputs(const G& g, const EnvArgs& a, int i, int res, int len, const u32* m) {
  if (a.result) a.result[i] = (i8)res;
  if (a.length) a.length[i] = len;
  if (a.masks) for (int k = 0; k < SB_MASK_WORDS; k++) a.masks[(size_t)i * SB_MASK_WORDS + k] = m[k];
  if (a.obs) {
    const int e = observe(g, a.obs + (size_t)i * SB_OBS_INTS);
    if (a.obs_err) a.obs_err[i] = (u8)e;
  } else if (a.obs_err) {
    int scratch[SB_OBS_INTS];
    a.obs_err[i] = (u8)observe(g, scratch);
  }
}

// opponents 0-2: one env per thread, the record in registers / local memory from load to store
SBD_FI void env_opponent_thread(G& g, const EnvArgs& a, int seat) {
  #pragma unroll 1
  while (!env_learner_moves(g, a, seat) && !env_over(g, a.max_steps)) {
    const int act = a.opponent == 1 ? pick_action(g) : expert_action(g);  // expert_action draws from the game's stream first
    game_step(g, act);
    end_of_step(g);
  }
}
__global__ void __launch_bounds__(TPB_GAME) k_env_step(const EnvArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;  // 128-bit moves
  const int seat = a.seat && a.seat[i] ? 1 : 0;  // any non-zero seat byte is SECOND
  int res = ENV_CONTINUES, len = 0;
  u32 m[SB_MASK_WORDS];
  if (a.seeds) {
    env_deal(g, s, a, i, a.seeds[i]);
    env_opponent_thread(g, a, seat);
  } else {
    load_state(s, a.states + (size_t)i * SB_STATE_BYTES);
    unpack(g, s);
    legal_mask(g, m);
    if (!env_legal(m, a.actions[i])) res = ENV_REJECTED;
    else {
      game_step(g, a.actions[i]);
      end_of_step(g);
      env_opponent_thread(g, a, seat);
      if (env_over(g, a.max_steps)) {
        res = env_result(g); len = g.steps;
        if (a.final_states) { pack(g, s); store_state(a.final_states + (size_t)i * SB_STATE_BYTES, s); }
        env_deal(g, s, a, i, env_next_seed(env_key(g)));
        env_opponent_thread(g, a, seat);
      }
    }
  }
  if (res != ENV_REJECTED) {
    pack(g, s);
    store_state(a.states + (size_t)i * SB_STATE_BYTES, s);
    legal_mask(g, m);
  }
  env_outputs(g, a, i, res, len, m);
}

// opponent 3: one env per warp, like k_rollout_heuristic: the working-set image of the game in shared memory, decide() for the
// opponent's decisions (a lane per candidate), lane 0 for the learner's action, the deal and the outputs
SBD_FI void env_opponent_warp(G& g, G* base, const EnvArgs& a, const double* w, int seat) {
  #pragma unroll 1
  while (!env_learner_moves(*base, a, seat) && !env_over(*base, a.max_steps)) decide(g, base, w, nullptr, true);
}
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_env_step_heur(const EnvArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  extern __shared__ __align__(16) unsigned char s_dyn[];  // WARPS_PER_CTA working-set images (sizeof(G) each)
  stage_cards(s_cards, cards);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS_PER_CTA + warp;
  if (i >= a.n) return;
  G* base = reinterpret_cast<G*>(s_dyn) + warp;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  double w[SB_N_FEATURES];
  const double* pw = a.w_opp + (size_t)(a.idx_opp ? a.idx_opp[i] : i) * SB_N_FEATURES;
  for (int k = 0; k < SB_N_FEATURES; k++) w[k] = pw[k];
  const int seat = a.seat && a.seat[i] ? 1 : 0;  // any non-zero seat byte is SECOND
  int res = ENV_CONTINUES, len = 0;
  u32 m[SB_MASK_WORDS];
  if (lane == 0) {
    if (a.seeds) env_deal(g, s, a, i, a.seeds[i]);
    else {
      load_state(s, a.states + (size_t)i * SB_STATE_BYTES);
      unpack(g, s);
      legal_mask(g, m);
      if (!env_legal(m, a.actions[i])) res = ENV_REJECTED;
      else { game_step(g, a.actions[i]); end_of_step(g); }
    }
    scan_badobs(g);
    copy_g(*base, g);
  }
  res = __shfl_sync(0xFFFFFFFFu, res, 0);
  __syncwarp();
  if (res != ENV_REJECTED) {
    env_opponent_warp(g, base, a, w, seat);
    if (!a.seeds && env_over(*base, a.max_steps)) {  // warp-uniform: every lane reads the same image
      __syncwarp();
      if (lane == 0) {
        copy_g(g, *base);
        res = env_result(g); len = g.steps;
        if (a.final_states) { pack(g, s); store_state(a.final_states + (size_t)i * SB_STATE_BYTES, s); }
        env_deal(g, s, a, i, env_next_seed(env_key(g)));
        scan_badobs(g);
        copy_g(*base, g);
      }
      __syncwarp();
      env_opponent_warp(g, base, a, w, seat);
    }
    __syncwarp();
    if (lane == 0) {
      copy_g(g, *base);
      pack(g, s);
      store_state(a.states + (size_t)i * SB_STATE_BYTES, s);
      legal_mask(g, m);
    }
  }
  if (lane == 0) env_outputs(g, a, i, res, len, m);
}

// ---------------------------------------------------------------- batched tree search (sb_search_*)
#include "sb_search.cuh"

// ---------------------------------------------------------------- information-set tree search (sb_ismcts_*)
#include "sb_ismcts.cuh"

// ---------------------------------------------------------------- Gumbel search for both trees (sb_*_gumbel)
#include "sb_gumbel.cuh"

// ---------------------------------------------------------------- determinization for sampled search (sb_determinize)
#include "sb_determinize.cuh"

__global__ void k_accumulate_fitness(int n, const i8* result, const int* idx_first, int* counts) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int ind = idx_first ? idx_first[i] : i;
  int r = result[i];
  atomicAdd(&counts[ind * 3 + (r == 0 ? 0 : r == 1 ? 2 : 1)], 1);
}

// games a rollout aborted (result -2), split by who would have raised: out[0] += codes the reference raises too
// (SB_ERR_NONE_TARGET .. SB_ERR_OBS_ID: its callers turn them into a draw as well), out[1] += limits of THIS engine
// (SB_ERR_UNSUPPORTED / OVERFLOW / DEPTH: the reference would have kept playing)
__global__ void k_count_aborted(int n, const u8* states, const i8* result, int* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || result[i] != -2) return;
  const int code = states[(size_t)i * SB_STATE_BYTES + 18];
  atomicAdd(&out[code >= SB_ERR_UNSUPPORTED ? 1 : 0], 1);
}

// The evaluation schedule on the device (evo/fitness.py:52-59,100-121): game index -> (FIRST individual, SECOND individual,
// seed).  A pairing plays games_per_pair consecutive games; pairings are enumerated
//   mode 0  round robin: (i, j) for i < n_ind, j < n_total, j != i, row-major (everyone against everyone and the hall of fame)
//   mode 1  versus: (i, n_ind + b) for i < n_ind, b < n_total - n_ind (every individual against fixed opponents)
//   mode 2  solo: (i, i) (the SECOND seat is the scripted opponent)
// seed = the partition-invariant hash of (base seed, generation, i, j, replicate) that evo.game_seed computes on the host.
__global__ void k_eval_schedule(int mode, int n_ind, int n_total, int gpp, unsigned long long base_seed, unsigned int generation,
                                long long g_lo, int n, int* idx_first, int* idx_second, unsigned long long* seeds) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long gi = g_lo + t;
  const long long p = gi / gpp;
  const unsigned long long k = (unsigned long long)(gi % gpp);
  long long i, j;
  if (mode == 0) { const long long per = n_total - 1; i = p / per; const long long r = p % per; j = r < i ? r : r + 1; }
  else if (mode == 1) { const long long per = n_total - n_ind; i = p / per; j = n_ind + p % per; }
  else { i = p; j = p; }
  const unsigned long long M = 0x7FFFFFFFFFFFFFFFull;
  unsigned long long x = (base_seed * 0x9E3779B97F4A7C15ull + (unsigned long long)generation * 0xBF58476D1CE4E5B9ull +
                          (unsigned long long)i * 0x94D049BB133111EBull + (unsigned long long)j * 0xD6E8FEB86659FD93ull + k) & M;
  x ^= x >> 31;
  x = (x * 0x2545F4914F6CDD1Dull) & M;
  idx_first[t] = (int)i;
  idx_second[t] = (int)j;
  seeds[t] = x;
}

// ================================================================ host side / C ABI
#include "sb_card_table_host.h"

struct SbHandle {
  int device;
  int sm_count;
  DCard* d_cards;
  double* d_wt;
  unsigned long long launches;
  char err[256];
  // staging for the *_host entry points
  u8* d_stage; size_t stage_bytes;
  u8* d_eval; size_t eval_bytes;  // workspace of sb_eval_population (states, schedule, results of one chunk)
  cudaStream_t stream;
  int gpw;  // games per warp for the thread-per-game shape (0 = choose by batch size)
  int turn_sync;   // 1: turn-synchronous warp schedule in the rollout kernel
  int block_sync;  // 0, or 128/256/512: CTA size whose warps change phase together (CTA-wide votes)
  int heur_wpc;    // heuristic rollout: 4 (independent warps) or 8/16/32 warps per CTA deciding in step
  int ctas_per_sm;
  int refill;      // -1 auto, 0 off, 1 on: finished lanes of the random rollout take the next game from a counter
  int refill_ctas; // persistent CTAs per SM in refill mode (0 = 1024 threads per SM)
  int dense;       // -1 auto, 0/1: the 32-register variant of the random rollout with two 1,024-thread CTAs per SM
  int refill_grid; // persistent CTAs in total (tests: a grid much smaller than the batch); 0 = sm_count x refill_ctas
  int heur_iw;     // heuristic rollout, independent warps: warps per CTA (4, 8, 16; -1 = auto)
  int heur_grid;   // persistent CTAs in refill mode (tests: a grid much smaller than the batch); 0 = one wave
  int heur_refill; // -1 auto, 0 off, 1 on: a warp whose game ended takes the next game from a counter
  int heur_pack;   // heuristic rollout with K games per warp (k_rollout_heuristic_packed): 0 off, 2 / 4 / 8; -1 auto
  int* d_queue;
  int engine;      // -1 auto, 0 thread-per-game kernels (sb_engine.cuh), 1 warp-per-game kernels (sbw_*.cuh)
  int w_shape;     // warp engine, random rollout: -1 auto, 0/1/2 = CTA shapes of sbw_rollout_random
  int w_grid;      // warp engine: persistent CTAs (tests: a grid much smaller than the batch); 0 = fill the chip
  int w_hshape;    // warp engine, heuristic rollout: -1 auto, 0/1
  SbwCtx wctx;
  u8* d_pools;    // deck generation: [5][POOL_W] card ids per faction
  int* d_pool_n;
  u8* d_arch;     // staged archetypes [24] + factions [2]
};

// Every entry point runs with the handle's device current and restores the caller's device afterwards: two handles in
// one process (or a caller whose current device is another GPU) launch on the right device without the library ever
// changing the caller's device for good.
struct DevGuard {
  int prev;
  bool switched;
  explicit DevGuard(int device) : prev(-1), switched(false) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
  }
  ~DevGuard() { if (switched) cudaSetDevice(prev); }
};
#define DEV_GUARD(h) DevGuard dev_guard_((h)->device)

static int fail(SbHandle* h, cudaError_t e, const char* what) {
  if (h) snprintf(h->err, sizeof h->err, "%s: %s", what, cudaGetErrorString(e));
  return -(int)e;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, e_, #call); } while (0)
#define LAUNCH_CHECK() do { h->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) return fail(h, e_, "kernel launch"); } while (0)

static inline int grid_for(int n, int per_cta) { return (n + per_cta - 1) / per_cta; }
// Which engine runs a call.  Both give identical results (tests/test_gpu_engines.py); the policy is MEASURED
// (profiles/r2_summary.md): one game per warp wins while the batch leaves the chip mostly empty -- its chain per env step is
// 2.5x shorter (6.8 us against 17 us) but every warp is its own instruction stream, so 28+ warps per SM thrash the
// instruction cache -- and for the record-streaming queries, whose pack / unpack it does one lane per tile; one game per
// thread wins once ~10 games share a warp's instruction stream.
enum { WK_ROLLOUT_RANDOM, WK_STEP, WK_LEGAL_MASK, WK_OBSERVE, WK_FEATURES, WK_EXPERT, WK_SELECT, WK_ROLLOUT_HEUR };
static inline bool use_warp_engine(const SbHandle* h, int kind, int n) {
  if (h->engine >= 0) return h->engine != 0;
  switch (kind) {
    case WK_ROLLOUT_RANDOM: return n <= h->sm_count * 32;   // one wave of 32-warp CTAs (4,096 games: 85 against 73 M env-steps/s)
    case WK_STEP: return n <= 8192;                          // 4,096 games: 0.077 against 0.143 ms; 65,536: 0.89 against 0.37 ms
    case WK_LEGAL_MASK: return true;                         // streaming kernel: 1,843 against 651 GB/s at 1 M records
    case WK_OBSERVE: return true;                            // streaming kernel: 1,626 against 382 GB/s at 65,536 records
    case WK_FEATURES: return n <= 65536;                     // 407 against 355 GB/s at 65,536 records; 512 against 650 at 1 M
    case WK_EXPERT: return n <= 16384;
    default: return false;                                   // heuristic agent: lane per candidate wins 3.5x
  }
}
static inline int games_per_warp(const SbHandle* h, int n) {
  if (h->gpw > 0 && h->gpw <= 32) return h->gpw;
  // auto (measured, tools/sweep_gpw.py): aim at ~3.5 warps per SM while the batch is small
  // (4096 games -> 8 per warp, 8192 -> 16, 16384 and up -> full warps)
  const int per_warp = (2 * n + h->sm_count * 7 - 1) / (h->sm_count * 7);
  return per_warp > 16 ? 32 : per_warp > 8 ? 16 : 8;
}
template <bool DIGEST>
static void launch_rollout_random(SbHandle* h, int n, uint8_t* states_d, int max_steps, int32_t* steps_d, uint64_t* chain_d,
                                  cudaStream_t st) {
  const int gpw = games_per_warp(h, n);
  unsigned long long* ch = (unsigned long long*)chain_d;
  int bs = h->block_sync;
  if (bs < 0) bs = n >= 90000 ? 1024 : n >= 57000 ? 512 : n >= 30000 ? 128 : 0;  // auto (tools/sweep_bsync.py): pays off once the chip is full
  // lane refill: persistent grid of resident CTAs, lanes take games from a counter (batches beyond the resident lanes)
  int* q = nullptr;
  const int resident = h->sm_count * 1024;  // 64 registers x 1024 threads fill one SM's register file
  int refill = h->refill;
  if (refill < 0) refill = n > resident;  // any batch that does not fit one wave (163,840 games: 258 -> 366 M env-steps/s)
  if (refill && bs >= 128 && h->turn_sync && gpw == 32) {
    q = h->d_queue;
    cudaMemsetAsync(q, 0, sizeof(int), st);
  }
  // resident CTAs per SM of the persistent grid (0 = fill the register file: 1024 threads per SM)
  const int tpb = bs >= 1024 ? 1024 : bs >= 512 ? 512 : bs >= 256 ? 256 : 128;
  const int per_sm = h->refill_ctas > 0 ? h->refill_ctas : 1024 / tpb;
  const int qgrid = h->refill_grid > 0 ? h->refill_grid : h->sm_count * per_sm;
  // dense variant: compiled for two 1,024-thread CTAs per SM (32 registers, 2,048 resident lanes per SM); more lanes in
  // flight hide more of the local-memory latency than the spills cost (tools/sweep_resident.py: 371 -> 400 M at 262 k games)
  int dense = h->dense;
  if (dense < 0) dense = n >= h->sm_count * 1536;
  if (bs >= 1024 && h->turn_sync && q && dense)
    k_rollout_random<DIGEST, 1024, true, 2><<<h->refill_grid > 0 ? h->refill_grid : 2 * h->sm_count, 1024, 0, st>>>(
        n, states_d, max_steps, steps_d, ch, h->d_cards, h->d_wt, gpw, 1, q);
  else if (bs >= 1024 && h->turn_sync)
    k_rollout_random<DIGEST, 1024, true><<<q ? qgrid : grid_for(n, gpw * 32), 1024, 0, st>>>(n, states_d, max_steps, steps_d, ch, h->d_cards, h->d_wt, gpw, 1, q);
  else if (bs >= 512 && h->turn_sync)
    k_rollout_random<DIGEST, 512, true><<<q ? qgrid : grid_for(n, gpw * 16), 512, 0, st>>>(n, states_d, max_steps, steps_d, ch, h->d_cards, h->d_wt, gpw, 1, q);
  else if (bs >= 256 && h->turn_sync)
    k_rollout_random<DIGEST, 256, true><<<q ? qgrid : grid_for(n, gpw * 8), 256, 0, st>>>(n, states_d, max_steps, steps_d, ch, h->d_cards, h->d_wt, gpw, 1, q);
  else if (bs >= 128 && h->turn_sync)
    k_rollout_random<DIGEST, 128, true><<<q ? qgrid : grid_for(n, gpw * 4), 128, 0, st>>>(n, states_d, max_steps, steps_d, ch, h->d_cards, h->d_wt, gpw, 1, q);
  else
    k_rollout_random<DIGEST, TPB_GAME, false><<<grid_for(n, gpw * (TPB_GAME / 32)), TPB_GAME, 0, st>>>(n, states_d, max_steps, steps_d, ch,
                                                                                                    h->d_cards, h->d_wt, gpw, h->turn_sync, nullptr);
}

extern "C" {

int sb_abi_version(void) { return SB_ABI_VERSION; }
int sb_state_bytes(void) { return (int)sizeof(SbState); }
int sb_card_count(void) { return SBC_COUNT; }
int sb_card_info(int card, int32_t out[12]) {
  if (card < 0 || card >= SBC_COUNT) return -1;
  const HostCard& c = HOST_CARDS[card];
  const int v[12] = {c.kind, c.faction, c.cost, c.strength, c.movement, c.trigger, c.fixed, c.has_ability, c.first_type, c.types, c.obs_id, c.has_target};
  for (int i = 0; i < 12; i++) out[i] = v[i];
  return 0;
}

int sb_create(int device, SbHandle** out) {
  *out = nullptr;
  SbHandle* h = (SbHandle*)calloc(1, sizeof(SbHandle));
  if (!h) return -2;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0 || device >= count) { free(h); return e != cudaSuccess ? -(int)e : -(int)cudaErrorNoDevice; }
  h->device = device;
  *out = h;
  DEV_GUARD(h);
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  h->sm_count = prop.multiProcessorCount;
  // the rules engine recurses (ability -> damage -> death trigger -> ability ...): size the per-thread stack
  CK(cudaDeviceSetLimit(cudaLimitStackSize, 48 * 1024));
  DCard tab[SBC_COUNT];
  sb_build_dcards(tab);
  CK(cudaMalloc(&h->d_cards, sizeof tab));
  CK(cudaMemcpy(h->d_cards, tab, sizeof tab, cudaMemcpyHostToDevice));
  static double wt[WT_N];
  sb_build_weights(wt);
  h->turn_sync = 1;
  h->block_sync = -1;
  h->heur_wpc = -1;
  {
    // shared-memory carveout: left to the driver by default.  Measured (tools/sweep_sync.py): forcing
    // MaxL1 halves the saturated throughput (the 3 KB card table per CTA no longer fits 16 CTAs/SM).
    const char* co = getenv("SB_CARVEOUT");
    const int carve = co ? atoi(co) : 25;  // 25 % = 57 KB shared: fits 16 CTAs x 3 KB, leaves ~170 KB of L1 (+2-4 % measured vs driver default)
    if (carve >= 0) {
      CK(cudaFuncSetAttribute(k_rollout_random<false, TPB_GAME, false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
      CK(cudaFuncSetAttribute(k_rollout_random<true, TPB_GAME, false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
      CK(cudaFuncSetAttribute(k_select_action, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
      CK(cudaFuncSetAttribute(k_step<false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
      CK(cudaFuncSetAttribute(k_step<true>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    }
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_rollout_random<false, TPB_GAME, false>, TPB_GAME, 0));
    h->ctas_per_sm = nb > 0 ? nb : 8;
  }
  CK(cudaMalloc(&h->d_wt, sizeof wt));
  CK(cudaMemcpy(h->d_wt, wt, sizeof wt, cudaMemcpyHostToDevice));
  // the heuristic rollout keeps one working-set image per warp in dynamic shared memory (up to 32 x sizeof(G) = 62 KB)
  CK(cudaFuncSetAttribute(k_rollout_heuristic<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(32 * sizeof(G))));
  CK(cudaFuncSetAttribute(k_rollout_heuristic<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(16 * sizeof(G))));
  CK(cudaFuncSetAttribute(k_rollout_heuristic<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(8 * sizeof(G))));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<8, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * PACK_BYTES(8)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<4, 4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * PACK_BYTES(4)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<2, 8, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * PACK_BYTES(2)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<2, 8, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * PACK_BYTES(2)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<1, 8, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * PACK_BYTES(1)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<1, 8, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * PACK_BYTES(1)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<1, 8, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * PACK_BYTES(1)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic_packed<1, 4, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * PACK_BYTES(1)));
  CK(cudaFuncSetAttribute(k_rollout_heuristic<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(4 * sizeof(G))));
  CK(cudaFuncSetAttribute(k_rollout_heuristic<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(8 * sizeof(G))));
  CK(cudaFuncSetAttribute(k_rollout_heuristic<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(16 * sizeof(G))));
  CK(cudaMalloc(&h->d_queue, 4 * sizeof(int)));  // [0] random rollout lanes, [1] heuristic rollout warps, [2..3] warp-engine grids
  CK(sbw_init());
  h->wctx.d_cards = h->d_cards; h->wctx.d_wt = h->d_wt; h->wctx.d_queue = h->d_queue + 2; h->wctx.sm_count = h->sm_count;
  h->engine = -1; h->w_shape = -1; h->w_hshape = -1;
  { const char* e = getenv("SB_ENGINE"); if (e) h->engine = atoi(e); }
  {  // deck pools: dir(cards) order == card index order; own faction + NEUTRAL (utils.py:74-84)
    static u8 pools[5 * POOL_W];
    int pn[5] = {0, 0, 0, 0, 0};
    memset(pools, 0, sizeof pools);
    for (int f = 0; f <= 4; f++)  // f = 0: an archetype led by a NEUTRAL card gives Faction.NEUTRAL (utils.py:152-153)
      for (int c = 1; c <= 112; c++)
        if ((HOST_CARDS[c].faction == f || HOST_CARDS[c].faction == 0) && pn[f] < POOL_W) pools[f * POOL_W + pn[f]++] = (u8)c;
    CK(cudaMalloc(&h->d_pools, sizeof pools));
    CK(cudaMemcpy(h->d_pools, pools, sizeof pools, cudaMemcpyHostToDevice));
    CK(cudaMalloc(&h->d_pool_n, sizeof pn));
    CK(cudaMemcpy(h->d_pool_n, pn, sizeof pn, cudaMemcpyHostToDevice));
    CK(cudaMalloc(&h->d_arch, 32));
  }
  h->refill = -1;
  h->dense = -1;
  h->heur_iw = -1; h->heur_pack = -1;
  h->heur_refill = -1;
  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  const char* env = getenv("SB_GPW");
  h->gpw = env ? atoi(env) : 0;
  return 0;
}
int sb_destroy(SbHandle* h) {
  if (!h) return 0;
  DEV_GUARD(h);
  if (h->d_cards) cudaFree(h->d_cards);
  if (h->d_wt) cudaFree(h->d_wt);
  if (h->d_queue) cudaFree(h->d_queue);
  if (h->d_pools) cudaFree(h->d_pools);
  if (h->d_pool_n) cudaFree(h->d_pool_n);
  if (h->d_arch) cudaFree(h->d_arch);
  if (h->d_stage) cudaFree(h->d_stage);
  if (h->d_eval) cudaFree(h->d_eval);
  if (h->stream) cudaStreamDestroy(h->stream);
  free(h);
  return 0;
}
const char* sb_last_error(SbHandle* h) { return h ? h->err : "null handle"; }
int sb_device(SbHandle* h) { return h->device; }
int sb_sm_count(SbHandle* h) { return h->sm_count; }
uint64_t sb_launch_count(SbHandle* h) { return h->launches; }


int sb_reset(SbHandle* h, int n, const uint64_t* seeds_d, const uint8_t* decks_d, int n_deck, int decks_shared,
             const uint8_t* factions_d, uint8_t* states_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  k_reset<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(n, (const unsigned long long*)seeds_d, decks_d, n_deck,
                                                                        decks_shared, factions_d, states_d, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_generate_decks(SbHandle* h, int n, const uint64_t* seeds_d, uint32_t generation, int mode, int n_preserve, double q,
                      const uint8_t* archetypes, const uint8_t* arch_factions, const uint8_t* factions_d, uint8_t* decks_d,
                      uint8_t* factions_out_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (mode < 0 || mode > 3 || (mode != 3 && (!archetypes || !arch_factions)) || (mode == 3 && !factions_d)) {
    snprintf(h->err, sizeof h->err, "sb_generate_decks: bad mode/arguments");
    return -1;
  }
  ArchParams ap;  // by value: no staging copy, no stream synchronisation inside the call
  memset(&ap, 0, sizeof ap);
  if (archetypes) memcpy(ap.arch, archetypes, 24);
  if (arch_factions) memcpy(ap.fac, arch_factions, 2);
  cudaStream_t st = (cudaStream_t)stream;
  const bool shared = factions_d == nullptr;
  k_generate_decks<<<grid_for(n, 128), 128, 0, st>>>(n, (const unsigned long long*)seeds_d, generation, mode, n_preserve, q, ap,
                                                   factions_d, shared ? 1 : 0, h->d_pools, h->d_pool_n, decks_d, factions_out_d);
  LAUNCH_CHECK();
  return 0;
}
static int es_args_ok(SbHandle* h, int mu, int nf, const char* what) {
  if (mu <= 0 || mu > ES_MAX_MU || nf <= 0 || nf > ES_MAX_FEATURES) {
    snprintf(h->err, sizeof h->err, "%s: mu must be 1..%d and n_features 1..%d", what, ES_MAX_MU, ES_MAX_FEATURES);
    return 0;
  }
  return 1;
}
int sb_es_offspring(SbHandle* h, uint64_t seed, uint32_t generation, int mu, int lambda, int n_features, double tau, double tau_prime,
                    double min_sigma, double* w_d, double* s_d, int32_t* parents_d, void* stream) {
  DEV_GUARD(h);
  if (!es_args_ok(h, mu, n_features, "sb_es_offspring")) return -1;
  if (lambda <= 0) return 0;
  k_es_offspring<<<grid_for(lambda, 128), 128, 0, (cudaStream_t)stream>>>(seed, generation, mu, lambda, n_features, tau, tau_prime, min_sigma,
                                                                         w_d, s_d, parents_d);
  LAUNCH_CHECK();
  return 0;
}
int sb_es_select(SbHandle* h, int total, int mu, int n_features, const double* fitness_d, const double* w_d, const double* s_d,
                 double* w_out_d, double* s_out_d, double* fit_out_d, int32_t* order_d, void* stream) {
  DEV_GUARD(h);
  if (!es_args_ok(h, mu, n_features, "sb_es_select")) return -1;
  if (total < mu) { snprintf(h->err, sizeof h->err, "sb_es_select: total < mu"); return -1; }
  k_es_select<<<grid_for(total, 128), 128, 0, (cudaStream_t)stream>>>(total, mu, n_features, fitness_d, w_d, s_d, w_out_d, s_out_d, fit_out_d, order_d);
  LAUNCH_CHECK();
  return 0;
}
int sb_es_reset_sigmas(SbHandle* h, uint64_t seed, uint32_t generation, int mu, int n_features, double initial_sigma, double* s_d, void* stream) {
  DEV_GUARD(h);
  if (!es_args_ok(h, mu, n_features, "sb_es_reset_sigmas")) return -1;
  k_es_reset_sigmas<<<grid_for(mu, 128), 128, 0, (cudaStream_t)stream>>>(seed, generation, mu, n_features, initial_sigma, s_d);
  LAUNCH_CHECK();
  return 0;
}
int sb_es_inject_diversity(SbHandle* h, uint64_t seed, uint32_t generation, int mu, int n_features, double tau, double tau_prime,
                           double min_sigma, double initial_sigma, double* w_d, double* s_d, int32_t* chosen_d, void* stream) {
  DEV_GUARD(h);
  if (!es_args_ok(h, mu, n_features, "sb_es_inject_diversity")) return -1;
  k_es_inject_diversity<<<1, 256, 0, (cudaStream_t)stream>>>(seed, generation, mu, n_features, tau, tau_prime, min_sigma, initial_sigma, w_d, s_d,
                                                             chosen_d);
  LAUNCH_CHECK();
  return 0;
}
int sb_legal_mask(SbHandle* h, int n, const uint8_t* states_d, uint32_t* masks_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_LEGAL_MASK, n)) { sbw_legal_mask(&h->wctx, n, states_d, masks_d, (cudaStream_t)stream); LAUNCH_CHECK(); return 0; }
  k_legal_mask<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, masks_d, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_expert_action(SbHandle* h, int n, uint8_t* states_d, uint8_t* actions_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_EXPERT, n)) { sbw_expert_action(&h->wctx, n, states_d, actions_d, (cudaStream_t)stream); LAUNCH_CHECK(); return 0; }
  k_expert_action<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, actions_d, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_step(SbHandle* h, int n, uint8_t* states_d, const uint8_t* actions_d, int8_t* reward_d, uint8_t* done_d, uint8_t* err_d,
            uint32_t* next_masks_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_STEP, n)) {
    sbw_step(&h->wctx, n, states_d, actions_d, reward_d, done_d, err_d, next_masks_d, (cudaStream_t)stream);
    LAUNCH_CHECK();
    return 0;
  }
  const int gpw = games_per_warp(h, n);
  int dense = h->dense;
  if (dense < 0) dense = n >= h->sm_count * 1536;
  if (dense)
    k_step<true><<<grid_for(n, gpw * (TPB_GAME / 32)), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, actions_d, (i8*)reward_d, done_d, err_d,
                                                                                            next_masks_d, h->d_cards, h->d_wt, gpw);
  else
    k_step<false><<<grid_for(n, gpw * (TPB_GAME / 32)), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, actions_d, (i8*)reward_d, done_d, err_d,
                                                                                             next_masks_d, h->d_cards, h->d_wt, gpw);
  LAUNCH_CHECK();
  return 0;
}
int sb_observe(SbHandle* h, int n, const uint8_t* states_d, int32_t* obs_d, uint8_t* err_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_OBSERVE, n)) { sbw_observe(&h->wctx, n, states_d, obs_d, err_d, (cudaStream_t)stream); LAUNCH_CHECK(); return 0; }
  k_observe<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, obs_d, err_d, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_features(SbHandle* h, int n, const uint8_t* states_d, double* feat_d, uint8_t* err_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_FEATURES, n)) { sbw_features(&h->wctx, n, states_d, feat_d, err_d, (cudaStream_t)stream); LAUNCH_CHECK(); return 0; }
  k_features<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(n, states_d, feat_d, err_d, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_select_action(SbHandle* h, int n, const uint8_t* states_d, const double* weights_d, uint8_t* actions_d, double* scores_d,
                     void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_SELECT, n)) { sbw_select_action(&h->wctx, n, states_d, weights_d, actions_d, scores_d, (cudaStream_t)stream); LAUNCH_CHECK(); return 0; }
  k_select_action<<<grid_for(n, WARPS_PER_CTA), WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(n, states_d, weights_d, actions_d, scores_d,
                                                                                                h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_rollout_random(SbHandle* h, int n, uint8_t* states_d, int max_steps, int32_t* steps_d, uint64_t* chain_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (use_warp_engine(h, WK_ROLLOUT_RANDOM, n)) {
    int shape = h->w_shape;
    if (shape < 0) shape = n <= h->sm_count * 32 ? 5 : 2;  // turn-synchronous 32-warp CTAs while one wave holds the batch (measured)
    sbw_rollout_random(&h->wctx, n, states_d, max_steps, steps_d, chain_d, shape, h->w_grid, (cudaStream_t)stream);
    LAUNCH_CHECK();
    return 0;
  }
  if (chain_d) launch_rollout_random<true>(h, n, states_d, max_steps, steps_d, chain_d, (cudaStream_t)stream);
  else launch_rollout_random<false>(h, n, states_d, max_steps, steps_d, nullptr, (cudaStream_t)stream);
  LAUNCH_CHECK();
  return 0;
}
int sb_set_option(SbHandle* h, const char* key, int value) {
  if (!strcmp(key, "lanes_per_game")) return 0;  // retired shape (measured slower, DESIGN.md); accepted and ignored
  if (!strcmp(key, "turn_sync")) { h->turn_sync = value; return 0; }
  if (!strcmp(key, "block_sync")) { h->block_sync = value; return 0; }
  if (!strcmp(key, "heur_wpc")) { h->heur_wpc = value; return 0; }
  if (!strcmp(key, "games_per_warp")) { h->gpw = value; return 0; }
  if (!strcmp(key, "ctas_per_sm")) { h->ctas_per_sm = value; return 0; }
  if (!strcmp(key, "refill")) { h->refill = value; return 0; }
  if (!strcmp(key, "dense")) { h->dense = value; return 0; }
  if (!strcmp(key, "refill_ctas")) { h->refill_ctas = value; return 0; }
  if (!strcmp(key, "refill_grid")) { h->refill_grid = value; return 0; }
  if (!strcmp(key, "heur_iw")) { h->heur_iw = value; return 0; }
  if (!strcmp(key, "heur_pack")) { h->heur_pack = value; return 0; }
  if (!strcmp(key, "heur_grid")) { h->heur_grid = value; return 0; }
  if (!strcmp(key, "heur_refill")) { h->heur_refill = value; return 0; }
  if (!strcmp(key, "engine")) { h->engine = value; return 0; }
  if (!strcmp(key, "w_shape")) { h->w_shape = value; return 0; }
  if (!strcmp(key, "w_grid")) { h->w_grid = value; return 0; }
  if (!strcmp(key, "w_hshape")) { h->w_hshape = value; return 0; }
  return -1;
}
int sb_rollout_heuristic(SbHandle* h, int n, uint8_t* states_d, const double* w_first_d, const double* w_second_d,
                         const int32_t* idx_first_d, const int32_t* idx_second_d, int max_steps, int8_t* result_d, int32_t* steps_d,
                         void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (use_warp_engine(h, WK_ROLLOUT_HEUR, n)) {
    sbw_rollout_heuristic(&h->wctx, n, states_d, w_first_d, w_second_d, idx_first_d, idx_second_d, max_steps, result_d, steps_d,
                          h->w_hshape < 0 ? 0 : h->w_hshape, h->w_grid, st);
    LAUNCH_CHECK();
    return 0;
  }
  const int pack = h->heur_pack < 0 ? 1 : h->heur_pack;  // auto: one game per warp in the owner / holder structure (faster at every batch size, tools/sweep_heur_pack.py)
  if (pack >= 1) {  // K games per warp, persistent grid
    int* q = h->d_queue + 1;
    cudaMemsetAsync(q, 0, sizeof(int), st);
#define HPACK(K, W, B) do { const int full = grid_for(n, (K) * (W)), resident = h->sm_count * (B); \
    const int grid = h->heur_grid > 0 ? h->heur_grid : (full < resident ? full : resident); \
    k_rollout_heuristic_packed<K, W, B><<<grid, (W) * 32, (W) * PACK_BYTES(K), st>>>(n, states_d, w_first_d, w_second_d, idx_first_d, idx_second_d, \
                                                                               max_steps, (i8*)result_d, steps_d, h->d_cards, h->d_wt, q); } while (0)
    // measured shapes (tools/sweep_heur_pack.py): K games per warp x warps per CTA x CTAs per SM
    switch (pack) {
      case 8: HPACK(8, 4, 4); break;   // 16 warps
      case 4: HPACK(4, 4, 8); break;   // 32 warps, 64 registers
      case 3: HPACK(2, 8, 6); break;   // 48 warps, 40 registers
      case 1: HPACK(1, 8, 8); break;   // 64 warps, 32 registers
      case 5: HPACK(1, 8, 6); break;   // 48 warps, 40 registers
      case 6: HPACK(1, 8, 4); break;   // 32 warps, 64 registers
      case 7: HPACK(1, 4, 16); break;  // 64 warps in 4-warp CTAs
      default: HPACK(2, 8, 8); break;  // 64 warps, 32 registers
    }
#undef HPACK
    LAUNCH_CHECK();
    return 0;
  }
  int hw = h->heur_wpc;
  if (hw < 0) hw = 4;  // auto (tools/sweep_heur.py): with the shared working-set image independent warps win at every batch size;
                       // limiting resident threads to fit L2 only loses (tools/sweep_heur_resident.py, removed knob)
  // independent warps: iw warps per CTA (4 / 8 / 16); batches beyond one wave run as a persistent grid with warp refill
  const int wave = h->sm_count * HEUR_MIN_CTAS * 4;  // resident warps = games in flight
  int refill = h->heur_refill;
  if (refill < 0) refill = n > wave;  // measured (tools/time_heur.py): 65,536 games 441 -> 404 ms, 399 ms with 8-warp CTAs
  const int iw_opt = h->heur_iw > 0 ? h->heur_iw : (refill ? 8 : 4);  // refill removes the CTA tail, so CTAs can share more
  const int iw = iw_opt >= 16 ? 16 : iw_opt >= 8 ? 8 : 4;
  int* q = nullptr;
  if (refill && hw < 8) {
    q = h->d_queue + 1;
    cudaMemsetAsync(q, 0, sizeof(int), st);
  }
#define HEUR(W, B, GRID) k_rollout_heuristic<W, B><<<GRID, W * 32, W * sizeof(G), st>>>(n, states_d, w_first_d, w_second_d, idx_first_d, \
                                                                                       idx_second_d, max_steps, (i8*)result_d, steps_d, h->d_cards, h->d_wt, q)
  if (hw >= 32) HEUR(32, true, grid_for(n, 32)); else if (hw >= 16) HEUR(16, true, grid_for(n, 16)); else if (hw >= 8) HEUR(8, true, grid_for(n, 8));
  else {
    const int full = grid_for(n, iw), resident = wave / iw;
    const int grid = q && h->heur_grid > 0 ? h->heur_grid : (q && full > resident ? resident : full);
    if (iw == 16) HEUR(16, false, grid); else if (iw == 8) HEUR(8, false, grid); else HEUR(4, false, grid);
  }
#undef HEUR
  LAUNCH_CHECK();
  return 0;
}
// The environment entries launch exactly one kernel, use no handle scratch, no atomics and no host synchronisation.  The kernel
// is fixed by the opponent kind (the "engine" option does not apply).
static int env_launch(SbHandle* h, const EnvArgs& a, const char* what, void* stream) {
  DEV_GUARD(h);
  const char* bad = a.opponent < 0 || a.opponent > 3 ? "opponent must be 0..3"
                    : a.opponent == 3 && !a.w_opp ? "opponent 3 needs a weight table"
                    : a.n_deck < 1 || a.n_deck > SB_DECK_MAX ? "n_deck must be 1..16"
                    : a.max_steps < 1 || a.max_steps > 65535 ? "max_steps must be 1..65535"
                    : a.n > 0 && (!a.states || !a.decks || !a.factions || !(a.seeds || a.actions)) ? "states, decks, factions and seeds / actions are required"
                    : nullptr;
  if (bad) { snprintf(h->err, sizeof h->err, "%s: %s", what, bad); return -1; }
  if (a.n <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (a.opponent == 3)
    k_env_step_heur<<<grid_for(a.n, WARPS_PER_CTA), WARPS_PER_CTA * 32, WARPS_PER_CTA * sizeof(G), st>>>(a, h->d_cards, h->d_wt);
  else
    k_env_step<<<grid_for(a.n, TPB_GAME), TPB_GAME, 0, st>>>(a, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_env_reset(SbHandle* h, int n, const uint64_t* seeds_d, const uint8_t* decks_d, int n_deck, int decks_shared,
                 const uint8_t* factions_d, int opponent, const uint8_t* seat_d, const double* w_opp_d,
                 const int32_t* idx_opp_d, int max_steps, uint8_t* states_d, int32_t* obs_d, uint32_t* masks_d,
                 uint8_t* obs_err_d, void* stream) {
  EnvArgs a = {n, states_d, (const unsigned long long*)seeds_d, nullptr, decks_d, n_deck, decks_shared, factions_d, opponent, seat_d,
               w_opp_d, idx_opp_d, max_steps, nullptr, nullptr, nullptr, obs_d, masks_d, obs_err_d};
  return env_launch(h, a, "sb_env_reset", stream);
}
int sb_env_step(SbHandle* h, int n, uint8_t* states_d, const uint8_t* actions_d, const uint8_t* decks_d, int n_deck,
                int decks_shared, const uint8_t* factions_d, int opponent, const uint8_t* seat_d, const double* w_opp_d,
                const int32_t* idx_opp_d, int max_steps, int8_t* result_d, int32_t* length_d, uint8_t* final_states_d,
                int32_t* obs_d, uint32_t* masks_d, uint8_t* obs_err_d, void* stream) {
  EnvArgs a = {n, states_d, nullptr, actions_d, decks_d, n_deck, decks_shared, factions_d, opponent, seat_d, w_opp_d, idx_opp_d,
               max_steps, (i8*)result_d, length_d, final_states_d, obs_d, masks_d, obs_err_d};
  return env_launch(h, a, "sb_env_step", stream);
}
// The search entries launch exactly one kernel, use no handle scratch, no atomics and no host synchronisation.
size_t sb_search_workspace_bytes(int n, int max_nodes) {
  if (n < 0 || max_nodes < 1 || max_nodes > SEARCH_MAX_NODES) return 0;
  const size_t tree = sizeof(STree) + (size_t)max_nodes * sizeof(SNode);
  return (size_t)n > SIZE_MAX / tree ? 0 : (size_t)n * tree;
}
static const char* search_bad(const SearchArgs& a, size_t ws_bytes) {
  const size_t need = sb_search_workspace_bytes(a.n, a.max_nodes);
  return a.n < 0 ? "n must be >= 0"
         : a.max_nodes < 1 || a.max_nodes > SEARCH_MAX_NODES ? "max_nodes must be 1..2^24"
         : a.n > 0 && need == 0 ? "workspace size overflows size_t"
         : a.n > 0 && !a.ws ? "workspace is NULL"
         : ((uintptr_t)a.ws & 15) ? "workspace must be 16-byte aligned"
         : ws_bytes < need ? "workspace too small (sb_search_workspace_bytes)"
         : nullptr;
}
static int search_launch(SbHandle* h, const SearchArgs& a, size_t ws_bytes, const char* bad, int which, void* stream) {
  DEV_GUARD(h);
  if (!bad) bad = search_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "%s: %s", which == 0 ? "sb_search_begin" : which == 1 ? "sb_search_simulate" : "sb_search_end", bad); return -1; }
  if (a.n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = grid_for(a.n, TPB_GAME);
  if (which == 0) k_search_begin<<<grid, TPB_GAME, 0, st>>>(a, h->d_cards, h->d_wt);
  else if (which == 1) k_search_simulate<<<grid, TPB_GAME, 0, st>>>(a, h->d_cards, h->d_wt);
  else k_search_end<<<grid, TPB_GAME, 0, st>>>(a);
  LAUNCH_CHECK();
  return 0;
}
int sb_search_begin(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const uint8_t* roots_d, int max_steps,
                    uint8_t* leaf_states_d, int32_t* obs_d, uint32_t* masks_d, uint8_t* obs_err_d, uint8_t* to_move_d,
                    uint8_t* leaf_kind_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, sizeof(STree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(SNode), roots_d,
                  max_steps, nullptr, nullptr, 0.0, 0.0, leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d,
                  nullptr, nullptr, nullptr};
  const char* bad = max_steps < 1 || max_steps > 65535 ? "max_steps must be 1..65535"
                    : n > 0 && !roots_d ? "roots are required"
                    : nullptr;
  return search_launch(h, a, ws_bytes, bad, 0, stream);
}
int sb_search_simulate(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d, const float* value_d,
                       double c_puct, double fpu, uint8_t* leaf_states_d, int32_t* obs_d, uint32_t* masks_d, uint8_t* obs_err_d,
                       uint8_t* to_move_d, uint8_t* leaf_kind_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, sizeof(STree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(SNode), nullptr,
                  0, prior_d, value_d, c_puct, fpu, leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d,
                  nullptr, nullptr, nullptr};
  const char* bad = !(c_puct >= 0.0 && c_puct <= 1.7976931348623157e308) ? "c_puct must be finite and >= 0"
                    : !(fpu >= -1.7976931348623157e308 && fpu <= 1.7976931348623157e308) ? "fpu must be finite"
                    : n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                    : nullptr;
  return search_launch(h, a, ws_bytes, bad, 1, stream);
}
int sb_search_end(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d, const float* value_d,
                  int32_t* visits_d, double* q_d, double* root_value_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, sizeof(STree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(SNode), nullptr,
                  0, prior_d, value_d, 0.0, 0.0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, visits_d, q_d, root_value_d};
  const char* bad = n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                    : n > 0 && (!visits_d || !q_d || !root_value_d) ? "visits, q and root_value are required"
                    : nullptr;
  return search_launch(h, a, ws_bytes, bad, 2, stream);
}
// The information-set search entries launch exactly one kernel, use no handle scratch, no atomics and no host synchronisation.
size_t sb_ismcts_workspace_bytes(int n, int max_nodes) {
  if (n < 0 || max_nodes < 1 || max_nodes > SEARCH_MAX_NODES) return 0;
  const size_t tree = sizeof(ITree) + (size_t)max_nodes * sizeof(INode);
  return (size_t)n > SIZE_MAX / tree ? 0 : (size_t)n * tree;
}
static const char* ismcts_bad(const SearchArgs& a, size_t ws_bytes) {
  const size_t need = sb_ismcts_workspace_bytes(a.n, a.max_nodes);
  return a.n < 0 ? "n must be >= 0"
         : a.max_nodes < 1 || a.max_nodes > SEARCH_MAX_NODES ? "max_nodes must be 1..2^24"
         : a.n > 0 && need == 0 ? "workspace size overflows size_t"
         : a.n > 0 && !a.ws ? "workspace is NULL"
         : ((uintptr_t)a.ws & 15) ? "workspace must be 16-byte aligned"
         : ws_bytes < need ? "workspace too small (sb_ismcts_workspace_bytes)"
         : nullptr;
}
static int ismcts_launch(SbHandle* h, const SearchArgs& a, size_t ws_bytes, const char* bad, int which, void* stream) {
  DEV_GUARD(h);
  if (!bad) bad = ismcts_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "%s: %s", which == 0 ? "sb_ismcts_begin" : which == 1 ? "sb_ismcts_simulate" : "sb_ismcts_end", bad); return -1; }
  if (a.n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = grid_for(a.n, TPB_GAME);
  if (which == 0) k_ismcts_begin<<<grid, TPB_GAME, 0, st>>>(a, h->d_cards, h->d_wt);
  else if (which == 1) k_ismcts_simulate<<<grid, TPB_GAME, 0, st>>>(a, h->d_cards, h->d_wt);
  else k_ismcts_end<<<grid, TPB_GAME, 0, st>>>(a);
  LAUNCH_CHECK();
  return 0;
}
static size_t ismcts_tree_bytes(int max_nodes) { return sizeof(ITree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(INode); }
int sb_ismcts_begin(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const uint8_t* det_d, int max_steps,
                    uint8_t* leaf_states_d, int32_t* obs_d, uint32_t* masks_d, uint8_t* obs_err_d, uint8_t* to_move_d,
                    uint8_t* leaf_kind_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, ismcts_tree_bytes(max_nodes), det_d, max_steps, nullptr, nullptr, 0.0, 0.0,
                  leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d, nullptr, nullptr, nullptr};
  const char* bad = max_steps < 1 || max_steps > 65535 ? "max_steps must be 1..65535"
                    : n > 0 && !det_d ? "worlds (det) are required"
                    : nullptr;
  return ismcts_launch(h, a, ws_bytes, bad, 0, stream);
}
int sb_ismcts_simulate(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const uint8_t* det_d, const float* prior_d,
                       const float* value_d, double c_puct, double fpu, uint8_t* leaf_states_d, int32_t* obs_d, uint32_t* masks_d,
                       uint8_t* obs_err_d, uint8_t* to_move_d, uint8_t* leaf_kind_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, ismcts_tree_bytes(max_nodes), det_d, 0, prior_d, value_d, c_puct, fpu,
                  leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d, nullptr, nullptr, nullptr};
  const char* bad = !(c_puct >= 0.0 && c_puct <= 1.7976931348623157e308) ? "c_puct must be finite and >= 0"
                    : !(fpu >= -1.7976931348623157e308 && fpu <= 1.7976931348623157e308) ? "fpu must be finite"
                    : n > 0 && !det_d ? "worlds (det) are required"
                    : n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                    : nullptr;
  return ismcts_launch(h, a, ws_bytes, bad, 1, stream);
}
int sb_ismcts_end(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d, const float* value_d,
                  int32_t* visits_d, double* q_d, double* root_value_d, void* stream) {
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, ismcts_tree_bytes(max_nodes), nullptr, 0, prior_d, value_d, 0.0, 0.0,
                  nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, visits_d, q_d, root_value_d};
  const char* bad = n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                    : n > 0 && (!visits_d || !q_d || !root_value_d) ? "visits, q and root_value are required"
                    : nullptr;
  return ismcts_launch(h, a, ws_bytes, bad, 2, stream);
}
// The Gumbel entries: the checks of their PUCT siblings plus the Gumbel arguments; one launch each, no handle scratch, no
// atomics and no host synchronisation.
static const char* gumbel_bad(int n, const GumbelArgs& gb, bool end) {
  const double big = 1.7976931348623157e308;
  return !(gb.c_visit >= 0.0 && gb.c_visit <= big) ? "c_visit must be finite and >= 0"
         : !(gb.c_scale >= 0.0 && gb.c_scale <= big) ? "c_scale must be finite and >= 0"
         : n > 0 && !gb.gumbel ? "gumbel is required"
         : end && n > 0 && (!gb.action || !gb.policy) ? "action and policy are required"
         : end ? nullptr
         : gb.num_simulations < 1 || gb.num_simulations > GUMBEL_MAX_SIMULATIONS ? "num_simulations must be 1..2^24"
         : gb.sim < 1 || gb.sim > gb.num_simulations ? "sim must be 1..num_simulations"
         : gb.max_considered < 1 || gb.max_considered > SB_N_ACTIONS ? "max_considered must be 1..156"
         : nullptr;
}
int sb_search_simulate_gumbel(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d,
                              const float* value_d, const float* gumbel_d, int sim, int num_simulations, int max_considered,
                              double c_visit, double c_scale, uint8_t* leaf_states_d, int32_t* obs_d, uint32_t* masks_d,
                              uint8_t* obs_err_d, uint8_t* to_move_d, uint8_t* leaf_kind_d, void* stream) {
  DEV_GUARD(h);
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, sizeof(STree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(SNode), nullptr,
                  0, prior_d, value_d, 0.0, 0.0, leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d,
                  nullptr, nullptr, nullptr};
  const GumbelArgs gb = {gumbel_d, sim, num_simulations, max_considered, c_visit, c_scale, nullptr, nullptr};
  const char* bad = gumbel_bad(n, gb, false);
  if (!bad) bad = n > 0 && (!prior_d || !value_d) ? "prior and value are required" : search_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "sb_search_simulate_gumbel: %s", bad); return -1; }
  if (n == 0) return 0;
  k_search_simulate_gumbel<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(a, gb, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_search_end_gumbel(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d, const float* value_d,
                         const float* gumbel_d, double c_visit, double c_scale, int32_t* action_d, float* policy_d,
                         int32_t* visits_d, double* q_d, double* root_value_d, void* stream) {
  DEV_GUARD(h);
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, sizeof(STree) + (size_t)(max_nodes > 0 ? max_nodes : 0) * sizeof(SNode), nullptr,
                  0, prior_d, value_d, 0.0, 0.0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, visits_d, q_d, root_value_d};
  const GumbelArgs gb = {gumbel_d, 0, 0, 0, c_visit, c_scale, action_d, policy_d};
  const char* bad = gumbel_bad(n, gb, true);
  if (!bad) bad = n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                  : n > 0 && (!visits_d || !q_d || !root_value_d) ? "visits, q and root_value are required"
                  : search_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "sb_search_end_gumbel: %s", bad); return -1; }
  if (n == 0) return 0;
  k_search_end_gumbel<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(a, gb);
  LAUNCH_CHECK();
  return 0;
}
int sb_ismcts_simulate_gumbel(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const uint8_t* det_d,
                              const float* prior_d, const float* value_d, const float* gumbel_d, int sim, int num_simulations,
                              int max_considered, double c_visit, double c_scale, uint8_t* leaf_states_d, int32_t* obs_d,
                              uint32_t* masks_d, uint8_t* obs_err_d, uint8_t* to_move_d, uint8_t* leaf_kind_d, void* stream) {
  DEV_GUARD(h);
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, ismcts_tree_bytes(max_nodes), det_d, 0, prior_d, value_d, 0.0, 0.0,
                  leaf_states_d, obs_d, masks_d, obs_err_d, to_move_d, leaf_kind_d, nullptr, nullptr, nullptr};
  const GumbelArgs gb = {gumbel_d, sim, num_simulations, max_considered, c_visit, c_scale, nullptr, nullptr};
  const char* bad = gumbel_bad(n, gb, false);
  if (!bad) bad = n > 0 && !det_d ? "worlds (det) are required" : n > 0 && (!prior_d || !value_d) ? "prior and value are required" : ismcts_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "sb_ismcts_simulate_gumbel: %s", bad); return -1; }
  if (n == 0) return 0;
  k_ismcts_simulate_gumbel<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(a, gb, h->d_cards, h->d_wt);
  LAUNCH_CHECK();
  return 0;
}
int sb_ismcts_end_gumbel(SbHandle* h, int n, int max_nodes, void* ws_d, size_t ws_bytes, const float* prior_d, const float* value_d,
                         const float* gumbel_d, double c_visit, double c_scale, int32_t* action_d, float* policy_d,
                         int32_t* visits_d, double* q_d, double* root_value_d, void* stream) {
  DEV_GUARD(h);
  SearchArgs a = {n, max_nodes, (unsigned char*)ws_d, ismcts_tree_bytes(max_nodes), nullptr, 0, prior_d, value_d, 0.0, 0.0,
                  nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, visits_d, q_d, root_value_d};
  const GumbelArgs gb = {gumbel_d, 0, 0, 0, c_visit, c_scale, action_d, policy_d};
  const char* bad = gumbel_bad(n, gb, true);
  if (!bad) bad = n > 0 && (!prior_d || !value_d) ? "prior and value are required"
                  : n > 0 && (!visits_d || !q_d || !root_value_d) ? "visits, q and root_value are required"
                  : ismcts_bad(a, ws_bytes);
  if (bad) { snprintf(h->err, sizeof h->err, "sb_ismcts_end_gumbel: %s", bad); return -1; }
  if (n == 0) return 0;
  k_ismcts_end_gumbel<<<grid_for(n, TPB_GAME), TPB_GAME, 0, (cudaStream_t)stream>>>(a, gb);
  LAUNCH_CHECK();
  return 0;
}
// One launch, no handle scratch, atomics or host synchronisation (capturable in a CUDA graph).
int sb_determinize(SbHandle* h, int n, const uint8_t* states_d, const uint8_t* observer_d, const uint64_t* keys_d, uint8_t* out_d,
                   void* stream) {
  DEV_GUARD(h);
  const char* bad = n < 0 ? "n must be >= 0" : n > 0 && (!states_d || !keys_d || !out_d) ? "states, keys and out are required" : nullptr;
  if (bad) { snprintf(h->err, sizeof h->err, "sb_determinize: %s", bad); return -1; }
  if (n == 0) return 0;
  k_determinize<<<grid_for(n, DET_WARPS), DET_WARPS * 32, 0, (cudaStream_t)stream>>>(n, states_d, observer_d,
                                                                                     (const unsigned long long*)keys_d, out_d);
  LAUNCH_CHECK();
  return 0;
}
int sb_accumulate_fitness(SbHandle* h, int n, const int8_t* result_d, const int32_t* idx_first_d, int32_t* counts_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  k_accumulate_fitness<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, (const i8*)result_d, idx_first_d, counts_d);
  LAUNCH_CHECK();
  return 0;
}

int sb_count_aborted(SbHandle* h, int n, const uint8_t* states_d, const int8_t* result_d, int32_t* out_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  k_count_aborted<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, states_d, (const i8*)result_d, out_d);
  LAUNCH_CHECK();
  return 0;
}

static inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

int sb_eval_schedule(SbHandle* h, int mode, int n_ind, int n_total, int games_per_pair, uint64_t base_seed, uint32_t generation,
                     int64_t game_lo, int n, int32_t* idx_first_d, int32_t* idx_second_d, uint64_t* seeds_d, void* stream) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  if (mode < 0 || mode > 2 || n_ind <= 0 || games_per_pair <= 0 || n_total < n_ind || (mode == 0 && n_total < 2) || (mode == 1 && n_total == n_ind)) {
    snprintf(h->err, sizeof(h->err), "sb_eval_schedule: bad schedule (mode %d, %d individuals, %d rows, %d games per pairing)", mode, n_ind,
             n_total, games_per_pair);
    return -1;
  }
  k_eval_schedule<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(mode, n_ind, n_total, games_per_pair, (unsigned long long)base_seed, generation,
                                                                    (long long)game_lo, n, idx_first_d, idx_second_d, (unsigned long long*)seeds_d);
  LAUNCH_CHECK();
  return 0;
}

// One evaluation = schedule -> new games -> whole heuristic games -> counts, chunk by chunk on `stream`, nothing on the host in
// between (no synchronisation: the caller reads counts_d when it needs them).
int sb_eval_population(SbHandle* h, int mode, int n_ind, int n_total, int games_per_pair, uint64_t base_seed, uint32_t generation,
                       int64_t game_lo, int64_t game_hi, const double* weights_d, const uint8_t* decks_d, int n_deck, const uint8_t* factions_d,
                       int max_steps, int chunk_games, int32_t* counts_d, int32_t* aborted_d, void* stream) {
  DEV_GUARD(h);
  if (game_hi <= game_lo) return 0;
  if (chunk_games <= 0) chunk_games = 262144;
  const int64_t total = game_hi - game_lo;
  const int cap = (int)(total < chunk_games ? total : chunk_games);
  const size_t o_states = 0, o_seed = al256((size_t)cap * SB_STATE_BYTES), o_i1 = o_seed + al256((size_t)cap * 8), o_i2 = o_i1 + al256((size_t)cap * 4),
               o_res = o_i2 + al256((size_t)cap * 4), bytes = o_res + al256((size_t)cap);
  if (h->eval_bytes < bytes) {
    if (h->d_eval) cudaFree(h->d_eval);
    h->d_eval = nullptr; h->eval_bytes = 0;
    CK(cudaMalloc(&h->d_eval, bytes));
    h->eval_bytes = bytes;
  }
  u8* d = h->d_eval;
  for (int64_t c0 = game_lo; c0 < game_hi; c0 += cap) {
    const int n = (int)(game_hi - c0 < cap ? game_hi - c0 : cap);
    int32_t* i1 = (int32_t*)(d + o_i1);
    int32_t* i2 = (int32_t*)(d + o_i2);
    int rc = sb_eval_schedule(h, mode, n_ind, n_total, games_per_pair, base_seed, generation, c0, n, i1, i2, (uint64_t*)(d + o_seed), stream);
    if (rc) return rc;
    rc = sb_reset(h, n, (const uint64_t*)(d + o_seed), decks_d, n_deck, 1, factions_d, d + o_states, stream);
    if (rc) return rc;
    rc = sb_rollout_heuristic(h, n, d + o_states, weights_d, mode == 2 ? nullptr : weights_d, i1, mode == 2 ? nullptr : i2, max_steps,
                              (int8_t*)(d + o_res), nullptr, stream);
    if (rc) return rc;
    rc = sb_accumulate_fitness(h, n, (const int8_t*)(d + o_res), i1, counts_d, stream);
    if (rc) return rc;
    if (aborted_d) { rc = sb_count_aborted(h, n, d + o_states, (const int8_t*)(d + o_res), aborted_d, stream); if (rc) return rc; }
  }
  return 0;
}

// ---------------------------------------------------------------- host-buffer (e2e) variants
static int ensure_stage(SbHandle* h, size_t bytes) {
  if (h->stage_bytes >= bytes) return 0;
  if (h->d_stage) cudaFree(h->d_stage);
  h->d_stage = nullptr; h->stage_bytes = 0;
  CK(cudaMalloc(&h->d_stage, bytes));
  h->stage_bytes = bytes;
  return 0;
}
int sb_step_host(SbHandle* h, int n, uint8_t* states, const uint8_t* actions, int8_t* reward, uint8_t* done, uint8_t* err,
                 uint32_t* next_masks) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  size_t o_states = 0, o_act = al256((size_t)n * SB_STATE_BYTES), o_rew = o_act + al256(n), o_done = o_rew + al256(n),
         o_err = o_done + al256(n), o_mask = o_err + al256(n), total = o_mask + al256((size_t)n * SB_MASK_WORDS * 4);
  int rc = ensure_stage(h, total);
  if (rc) return rc;
  u8* d = h->d_stage;
  cudaStream_t st = h->stream;
  CK(cudaMemcpyAsync(d + o_states, states, (size_t)n * SB_STATE_BYTES, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_act, actions, n, cudaMemcpyHostToDevice, st));
  rc = sb_step(h, n, d + o_states, d + o_act, (int8_t*)(d + o_rew), d + o_done, d + o_err, next_masks ? (uint32_t*)(d + o_mask) : nullptr, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(states, d + o_states, (size_t)n * SB_STATE_BYTES, cudaMemcpyDeviceToHost, st));
  if (reward) CK(cudaMemcpyAsync(reward, d + o_rew, n, cudaMemcpyDeviceToHost, st));
  if (done) CK(cudaMemcpyAsync(done, d + o_done, n, cudaMemcpyDeviceToHost, st));
  if (err) CK(cudaMemcpyAsync(err, d + o_err, n, cudaMemcpyDeviceToHost, st));
  if (next_masks) CK(cudaMemcpyAsync(next_masks, d + o_mask, (size_t)n * SB_MASK_WORDS * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int sb_rollout_random_host(SbHandle* h, int n, const uint64_t* seeds, const uint8_t* decks, int n_deck, const uint8_t* factions,
                           int max_steps, uint8_t* states_out, int32_t* steps_out, uint64_t* chain_out) {
  DEV_GUARD(h);
  if (n <= 0) return 0;
  size_t o_states = 0, o_seed = al256((size_t)n * SB_STATE_BYTES), o_deck = o_seed + al256((size_t)n * 8),
         o_fac = o_deck + al256((size_t)2 * n_deck), o_steps = o_fac + 256, o_chain = o_steps + al256((size_t)n * 4),
         total = o_chain + al256((size_t)n * 8);
  int rc = ensure_stage(h, total);
  if (rc) return rc;
  u8* d = h->d_stage;
  cudaStream_t st = h->stream;
  CK(cudaMemcpyAsync(d + o_seed, seeds, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_deck, decks, (size_t)2 * n_deck, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_fac, factions, 2, cudaMemcpyHostToDevice, st));
  rc = sb_reset(h, n, (const uint64_t*)(d + o_seed), d + o_deck, n_deck, 1, d + o_fac, d + o_states, st);
  if (rc) return rc;
  if (chain_out) CK(cudaMemsetAsync(d + o_chain, 0, (size_t)n * 8, st));
  rc = sb_rollout_random(h, n, d + o_states, max_steps, (int32_t*)(d + o_steps), chain_out ? (uint64_t*)(d + o_chain) : nullptr, st);
  if (rc) return rc;
  if (states_out) CK(cudaMemcpyAsync(states_out, d + o_states, (size_t)n * SB_STATE_BYTES, cudaMemcpyDeviceToHost, st));
  if (steps_out) CK(cudaMemcpyAsync(steps_out, d + o_steps, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  if (chain_out) CK(cudaMemcpyAsync(chain_out, d + o_chain, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
