// Information-set Monte-Carlo tree search (single-observer ISMCTS, Cowling, Powley & Whitehouse 2012) with a caller-supplied
// evaluator (sb_ismcts_begin / sb_ismcts_simulate / sb_ismcts_end): n trees, one tree per thread, one launch per simulation,
// as sb_search.cuh.  Tree g is built over the information set of its root's player, not over one record: every call brings
// this call's world for each root (det u8[n,512], normally sb_determinize of the root under a fresh key) and the walk replays
// the tree's moves in that world from its root.  So a node holds no record, and its edges are keyed by what a move is (a
// move code computed from the mover's hand in the current world), not by the hand slot, which holds different cards in
// different worlds.  Included by sb_kernels.cu after sb_search.cuh, whose SearchArgs (roots = this call's worlds), s_sign,
// leaf kinds and node limit it reuses.
//
// Workspace (caller-owned, sized by sb_ismcts_workspace_bytes): tree g at ws + g * tree_bytes, tree_bytes =
// 656 * (1 + max_nodes).  A tree is a 656-byte header followed by max_nodes nodes of 656 bytes each:
//   header  used nodes, pending leaf, leaf kind, max_steps, game value of a pending terminal leaf (FIRST's view), 12 B
//           padding, then root_code u32[156]: the move code of each root action id, ISM_NONE where the id is illegal or does
//           not represent its code
//   node    W f64 (FIRST's view), parent i32 (-1 at the root), first child i32, next sibling i32 (-1 = none), code u32 of the
//           edge into the node, N i32, seat to move u8 (0 FIRST / 1 SECOND) + 3 B padding, prior f32[156] (the caller's
//           prior when the node was evaluated, by the action ids of the world it was evaluated in; zero for a node created
//           terminal)
// 4,096 trees of 65 nodes (64 simulations) take 177 MB.
//
// Move codes, u32 (kind << 24 | card << 16 | x), card = hand[ci].card of the mover in the current world:
//   PLACE a < 64 (ci = a >> 4)            (0, card, a & 15)
//   SPELL 64..147 (ci, idx = (a-64) / 21, (a-64) % 21)  (1, card, idx)
//   CYCLE 148..151 (ci = a - 148)         (2, card, 0)
//   152..154 (ci = a - 151)               (3, card, hand[0].card)
//   PASS 155                              ISM_PASS
// Two legal ids with one code (copies of a card in one hand): the lowest represents the code, the others are never chosen.
//
// Fault safety: every node index read from the workspace is checked against the tree's node count before it is
// dereferenced, sibling walks and the parent chain are bounded by it, and the descent by max_nodes, so a workspace that
// was not written by sb_ismcts_begin cannot send a thread outside its own tree.  The kernels keep no per-node table on the
// stack (the children are matched to action ids by one sibling walk per level), so their frames stay below
// k_search_simulate's, which already runs the rule recursion under the 48 KB stack limit (DESIGN.md 2, 3).
#pragma once
#include "sb_search.cuh"

struct __align__(16) INode {
  double W;
  int parent, child, sibling;
  u32 code;
  int N;
  u8 seat, pad[3];
  float prior[SB_N_ACTIONS];
};
static_assert(sizeof(INode) == 656, "INode layout (header comment, DESIGN.md 8.8)");
struct __align__(16) ITree {
  int used;        // nodes in use
  int leaf;        // node emitted by the last call
  int kind;        // SEARCH_EVAL, SEARCH_TERMINAL or SEARCH_FULL (nothing pending)
  int max_steps;   // terminal rule (env_over)
  int tval;        // game value for FIRST of a pending terminal leaf in the world it was reached in
  int pad[3];
  u32 root_code[SB_N_ACTIONS];
};
static_assert(sizeof(ITree) == 656, "ITree layout (header comment, DESIGN.md 8.8)");
#define ISM_PASS (4u << 24)
#define ISM_NONE 0xFFFFFFFFu

SBD_FI ITree& ism_tree(const SearchArgs& a, int i) { return *reinterpret_cast<ITree*>(a.ws + (size_t)i * a.tree_bytes); }
SBD_FI INode* ism_nodes(const SearchArgs& a, int i) { return reinterpret_cast<INode*>(a.ws + (size_t)i * a.tree_bytes + sizeof(ITree)); }
SBD_FI bool ism_in(int j, int lim) { return (unsigned)j < (unsigned)lim; }
// the nodes of the tree that may be dereferenced: used, clamped to 0..max_nodes
SBD_FI int ism_lim(const ITree& t, int max_nodes) { const int u = t.used; return u < 0 ? 0 : u > max_nodes ? max_nodes : u; }
SBD_FI bool ism_bit(const u32* m, int a) { return m[a >> 5] >> (a & 31) & 1u; }
SBD_FI int ism_value(const G& g) { const int r = env_result(g); return r == 0 ? 1 : r == 1 ? -1 : 0; }

SBD_FI u32 ism_code(const Ply& p, int a) {
  if (a < 64) return (u32)p.hand[a >> 4].card << 16 | (u32)(a & 15);
  if (a < 148) return 1u << 24 | (u32)p.hand[(a - 64) / 21].card << 16 | (u32)((a - 64) % 21);
  if (a < 152) return 2u << 24 | (u32)p.hand[a - 148].card << 16;
  if (a < 155) return 3u << 24 | (u32)p.hand[a - 151].card << 16 | (u32)p.hand[0].card;
  return ISM_PASS;
}
// a legal id represents its code unless a lower legal id of the same kind names the same card (the ids of one kind differ
// by `stride` per hand slot; swaps start at slot 1)
SBD_FI bool ism_rep(const Ply& p, const u32* m, int a) {
  const int ci = a < 64 ? a >> 4 : a < 148 ? (a - 64) / 21 : a < 152 ? a - 148 : a < 155 ? a - 151 : -1;
  const int stride = a < 64 ? 16 : a < 148 ? 21 : 1, lo = a >= 152 && a < 155 ? 1 : 0;
  #pragma unroll 1
  for (int cj = lo; cj < ci; cj++)
    if (p.hand[cj].card == p.hand[ci].card && ism_bit(m, a - (ci - cj) * stride)) return false;
  return true;
}
// the legal action id that represents `code` in the current world (the lowest legal id with that code), -1 if none
SBD_FI int ism_action(const Ply& p, const u32* m, u32 code) {
  if (code == ISM_PASS) return ism_bit(m, SB_ACTION_PASS) ? SB_ACTION_PASS : -1;
  const int kind = (int)(code >> 24), card = (int)(code >> 16 & 255u), x = (int)(code & 0xFFFFu);
  if (kind > 3 || (kind == 0 && x > 15) || (kind == 1 && x > 20) || (kind == 2 && x != 0) || (kind == 3 && x > 255)) return -1;
  if (kind == 3 && p.hand[0].card != x) return -1;
  #pragma unroll 1
  for (int ci = kind == 3 ? 1 : 0; ci < SB_HAND_MAX; ci++) {
    if (p.hand[ci].card != card) continue;
    const int a = kind == 0 ? 16 * ci + x : kind == 1 ? 64 + 21 * ci + x : kind == 2 ? 148 + ci : 151 + ci;
    if (ism_bit(m, a)) return a;
  }
  return -1;
}

// observe()'s code without an observation buffer, in a call of its own: its 2,160-byte scratch then does not share the
// frame of k_ismcts_simulate (4,752 B against 5,296 B with the scratch inline, ptxas -v)
SBD_NI int ism_obs_err(const G& g) {
  G_LOCAL(g);
  int scratch[SB_OBS_INTS];
  return observe(g, scratch);
}
// the leaf outputs of tree i: the world's record s at the leaf, its working set g and legal mask m
SBD_FI void ism_emit(const SearchArgs& a, int i, const G& g, const SbState& s, const u32* m, int kind) {
  if (a.leaf_states) store_state(a.leaf_states + (size_t)i * SB_STATE_BYTES, s);
  if (a.masks) for (int k = 0; k < SB_MASK_WORDS; k++) a.masks[(size_t)i * SB_MASK_WORDS + k] = m[k];
  if (a.obs) {
    const int e = observe(g, a.obs + (size_t)i * SB_OBS_INTS);
    if (a.obs_err) a.obs_err[i] = (u8)e;
  } else if (a.obs_err) {
    a.obs_err[i] = (u8)ism_obs_err(g);
  }
  if (a.to_move) a.to_move[i] = g.player_sign == 1 ? 0 : 1;
  if (a.leaf_kind) a.leaf_kind[i] = (u8)kind;
}

SBD_FI void ism_zero_prior(INode& nd) {
  float4* p = reinterpret_cast<float4*>(nd.prior);
  #pragma unroll 1
  for (int k = 0; k < SB_N_ACTIONS / 4; k++) p[k] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// store the caller's prior / value for the pending leaf and add its value (FIRST's view) to every node up to the root
SBD_FI void ism_backup(const SearchArgs& a, int i, ITree& t, INode* nodes) {
  const int lim = ism_lim(t, a.max_nodes);
  if (t.kind == SEARCH_FULL || !ism_in(t.leaf, lim)) return;
  INode& leaf = nodes[t.leaf];
  double v;
  if (t.kind == SEARCH_TERMINAL) v = (double)t.tval;
  else {
    const float* p = a.prior + (size_t)i * SB_N_ACTIONS;
    #pragma unroll 1
    for (int k = 0; k < SB_N_ACTIONS; k++) leaf.prior[k] = p[k];
    v = __dmul_rn(s_sign(leaf.seat), (double)a.value[i]);
  }
  int j = t.leaf;
  #pragma unroll 1
  for (int d = 0; d < lim && ism_in(j, lim); d++) {
    nodes[j].N += 1;
    nodes[j].W = __dadd_rn(nodes[j].W, v);
    j = nodes[j].parent;
  }
}

// PUCT at node nd over the current world's legal representatives (mover's hand p, legal mask m), the formula and FP64
// order of s_select; n_a and W from the child whose code the id has.  The children are scored in one sibling walk, the ids
// without a child after it; the better score wins, ties to the lower action id (the result of s_select's scan in id order).
// child <- the chosen id's node, -1 when it has none.
SBD_FI int ism_select(const SearchArgs& a, const INode* nodes, int lim, const INode& nd, const Ply& p, const u32* m, int& child) {
  const double sgn = s_sign(nd.seat), sq = __dsqrt_rn((double)nd.N);
  u32 has[SB_MASK_WORDS] = {0, 0, 0, 0, 0};
  int best = -1, best_child = -1;
  double best_score = 0.0;
  int c = nd.child;
  #pragma unroll 1
  for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling) {
    const int act = ism_action(p, m, nodes[c].code);
    if (act < 0) continue;  // the move does not exist in this world
    has[act >> 5] |= 1u << (act & 31);
    const double score = s_score(a, nodes[c].N, __dmul_rn(sgn, nodes[c].W), nd.prior[act], sq);
    if (best < 0 || score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_child = c; }
  }
  #pragma unroll 1
  for (int w = 0; w < SB_MASK_WORDS; w++) {
    u32 r = m[w] & ~has[w];
    while (r) {
      const int act = w * 32 + __ffs(r) - 1;
      r &= r - 1;
      if (!ism_rep(p, m, act)) continue;
      const double score = s_score(a, 0, 0.0, nd.prior[act], sq);
      if (best < 0 || score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_child = -1; }
    }
  }
  child = best_child;
  return best;
}

// the header of tree i (root codes from the world's record s, unpacked to g) and the leaf outputs of its root:
// sb_ismcts_begin's tree (kept = 0: node 0 is written fresh), or one whose first `kept` nodes sb_ismcts_advance carried
// over (node 0 is already the root, and the world is not over).  m receives the root's legal mask; it is the kernel's own
// array so that the kernel's frame keeps the layout it had before this function was factored out of k_ismcts_begin.
SBD_FI void ism_start(const SearchArgs& a, int i, const G& g, const SbState& s, u32* m, int kept) {
  ITree& t = ism_tree(a, i);
  INode& root = ism_nodes(a, i)[0];
  legal_mask(g, m);
  const Ply& p = g.pl[g.local_order];
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) t.root_code[act] = ism_bit(m, act) && ism_rep(p, m, act) ? ism_code(p, act) : ISM_NONE;
  if (!kept) {
    root.W = 0.0;
    root.parent = -1;
    root.child = -1;
    root.sibling = -1;
    root.code = ISM_NONE;
    root.N = 0;
    root.seat = g.player_sign == 1 ? 0 : 1;
  }
  const bool over = env_over(g, a.max_steps);
  if (!kept && over) ism_zero_prior(root);
  t.used = kept ? kept : 1;
  t.leaf = 0;
  t.kind = over ? SEARCH_TERMINAL : SEARCH_EVAL;
  t.max_steps = a.max_steps;
  t.tval = over ? ism_value(g) : 0;
  ism_emit(a, i, g, s, m, t.kind);
}

__global__ void __launch_bounds__(TPB_GAME) k_ismcts_begin(const SearchArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  u32 m[SB_MASK_WORDS];
  ism_start(a, i, g, s, m, 0);
}

// one simulate call of tree i (k_ismcts_simulate, k_ismcts_simulate_gumbel): back up the pending leaf, unpack this call's
// world at the root (record s, working set g, legal mask m), stop when the tree is full, else replay the tree's moves in
// that world from the root and expand or emit a leaf.  select(nodes, j, lim, m, c) chooses the action at node j among the
// world's legal representatives and sets c to the child with its code (-1 = none).  Every node index is checked against
// lim and the descent is bounded by max_nodes.
template <class Select>
SBD_FI void ism_simulate(const SearchArgs& a, int i, G& g, Select select) {
  ITree& t = ism_tree(a, i);
  INode* nodes = ism_nodes(a, i);
  ism_backup(a, i, t, nodes);
  __align__(16) SbState s;
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  u32 m[SB_MASK_WORDS];
  legal_mask(g, m);
  if (t.kind == SEARCH_FULL || t.used < 1 || t.used >= a.max_nodes) {  // the tree stops: the world's root is emitted
    t.kind = SEARCH_FULL;
    ism_emit(a, i, g, s, m, SEARCH_FULL);
    return;
  }
  const int lim = t.used;
  int j = 0;
  #pragma unroll 1
  for (int d = 0; d < a.max_nodes; d++) {
    if (env_over(g, t.max_steps)) {  // terminal in this world: its game value is backed up
      t.leaf = j;
      t.kind = SEARCH_TERMINAL;
      t.tval = ism_value(g);
      ism_emit(a, i, g, s, m, SEARCH_TERMINAL);
      return;
    }
    int c;
    const int act = select(nodes, j, lim, m, c);
    if (act < 0) break;
    const u32 code = ism_code(g.pl[g.local_order], act);
    s_step(g, s, act);
    legal_mask(g, m);
    if (c < 0) {  // expand: a node for the code
      const int k = t.used++;
      INode& nd = nodes[k];
      nd.W = 0.0;
      nd.parent = j;
      nd.child = -1;
      nd.sibling = nodes[j].child;
      nd.code = code;
      nd.N = 0;
      nd.seat = g.player_sign == 1 ? 0 : 1;
      nodes[j].child = k;
      const bool over = env_over(g, t.max_steps);
      if (over) ism_zero_prior(nd);
      t.leaf = k;
      t.kind = over ? SEARCH_TERMINAL : SEARCH_EVAL;
      t.tval = over ? ism_value(g) : 0;
      ism_emit(a, i, g, s, m, t.kind);
      return;
    }
    j = c;
  }
  // only a workspace not written by sb_ismcts_begin gets here (a well-formed tree is at most max_nodes deep): the tree stops
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  legal_mask(g, m);
  t.kind = SEARCH_FULL;
  ism_emit(a, i, g, s, m, SEARCH_FULL);
}

__global__ void __launch_bounds__(TPB_GAME) k_ismcts_simulate(const SearchArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  ism_simulate(a, i, g, [&](const INode* nodes, int j, int lim, const u32* m, int& c) {
    return ism_select(a, nodes, lim, nodes[j], g.pl[g.local_order], m, c);
  });
}

// the child of node nd whose code is `code` (first in the sibling walk), -1 if none
SBD_FI int ism_find(const INode* nodes, int lim, const INode& nd, u32 code) {
  int c = nd.child;
  #pragma unroll 1
  for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling)
    if (nodes[c].code == code) return c;
  return -1;
}

// the value estimate of node s from what its children do not account for, Gumbel's vhat (sb_gumbel.cuh): every child of s
// in sibling-walk order
SBD_FI double ism_vhat(const INode* nodes, int lim, const INode& s, double sgn) {
  int sn = 0;
  double sw = 0.0;
  int c = s.child;
  #pragma unroll 1
  for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling) { sn += nodes[c].N; sw = __dadd_rn(sw, nodes[c].W); }
  const int den = s.N - sn;
  return den < 1 ? 0.0 : __ddiv_rn(__dmul_rn(sgn, __dadd_rn(s.W, -sw)), (double)den);
}

// back up the last pending leaf of tree i (the tree then holds nothing pending) and read out visits, q and root_value by
// the root's action ids; returns the node count lim, 0 when the header holds none usable (the read-out is then empty)
SBD_FI int ism_end(const SearchArgs& a, int i) {
  ITree& t = ism_tree(a, i);
  INode* nodes = ism_nodes(a, i);
  ism_backup(a, i, t, nodes);
  t.kind = SEARCH_FULL;
  const int lim = ism_lim(t, a.max_nodes);
  if (lim < 1) {
    #pragma unroll 1
    for (int act = 0; act < SB_N_ACTIONS; act++) { a.visits[(size_t)i * SB_N_ACTIONS + act] = 0; a.q[(size_t)i * SB_N_ACTIONS + act] = S_QNAN; }
    a.root_value[i] = S_QNAN;
    return 0;
  }
  const INode& root = nodes[0];
  const double sgn = s_sign(root.seat);
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) {
    const u32 code = t.root_code[act];
    const int c = code == ISM_NONE ? -1 : ism_find(nodes, lim, root, code);
    const int na = c >= 0 ? nodes[c].N : 0;
    a.visits[(size_t)i * SB_N_ACTIONS + act] = na;
    a.q[(size_t)i * SB_N_ACTIONS + act] = na ? __ddiv_rn(__dmul_rn(sgn, nodes[c].W), (double)na) : S_QNAN;
  }
  a.root_value[i] = __ddiv_rn(__dmul_rn(sgn, root.W), (double)root.N);
  return lim;
}

__global__ void __launch_bounds__(TPB_GAME) k_ismcts_end(const SearchArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < a.n) ism_end(a, i);
}
