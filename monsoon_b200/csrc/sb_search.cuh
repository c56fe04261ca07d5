// Batched Monte-Carlo tree search with a caller-supplied evaluator (sb_search_begin / sb_search_simulate / sb_search_end):
// n independent PUCT trees, one tree per thread, one launch per simulation.  The evaluator (prior over the 156 action ids
// and a value) stays with the caller; one simulate call backs up the leaf the previous call emitted, selects a new leaf,
// expands it with the engine's own game_step + end_of_step, and emits what the evaluator needs (record, observation,
// legal mask, seat to move, leaf kind).  Transitions are the records sb_step produces from the parent record, so the
// tree sees both hands and the future draws (perfect-information search, the fork semantics of the reference's own
// agent).  Included by sb_kernels.cu after the environment kernels, whose env_over / env_result it reuses.
//
// Workspace (caller-owned, sized by sb_search_workspace_bytes): tree g at ws + g * tree_bytes, tree_bytes =
// 16 + max_nodes * 1,808.  A tree is a 16-byte header {used nodes, pending leaf, leaf kind, max_steps} followed by
// max_nodes nodes of 1,808 bytes each:
//   rec     512  packed record (SbState)
//   child   624  i32[156] node index of the child per action id, 0 = none (node 0 is the root, never a child)
//   prior   624  f32[156] the caller's prior for this node (entries at illegal actions are never read)
//   mask     20  u32[5] legal mask
//   parent    4  i32, -1 at the root
//   W         8  f64 value sum from FIRST's point of view
//   N         4  i32 visits, including the node's own evaluation
//   action, seat (0 FIRST / 1 SECOND), terminal, terminal value for FIRST (+1 / -1 / 0): 1 byte each
// 4,096 trees of 65 nodes (64 simulations) take 481 MB.
#pragma once
#include "sb_engine.cuh"

struct __align__(16) SNode {
  SbState rec;
  int child[SB_N_ACTIONS];
  float prior[SB_N_ACTIONS];
  u32 mask[SB_MASK_WORDS];
  int parent;
  double W;
  int N;
  u8 action, seat, terminal;
  i8 tval;
};
static_assert(sizeof(SNode) == 1808, "SNode layout (header comment, DESIGN.md 8.6)");
struct __align__(16) STree {
  int used;        // nodes in use
  int leaf;        // node emitted by the last call
  int kind;        // SEARCH_EVAL, SEARCH_TERMINAL or SEARCH_FULL (nothing pending)
  int max_steps;   // terminal rule of the nodes (env_over)
};
static_assert(sizeof(STree) == 16, "STree layout");
#define SEARCH_EVAL 0
#define SEARCH_TERMINAL 1
#define SEARCH_FULL 2
#define SEARCH_MAX_NODES (1 << 24)

struct SearchArgs {
  int n, max_nodes;
  unsigned char* ws; size_t tree_bytes;
  const u8* roots; int max_steps;
  const float* prior; const float* value; double c_puct, fpu;
  u8* leaf_states; int* obs; u32* masks; u8* obs_err; u8* to_move; u8* leaf_kind;
  int* visits; double* q; double* root_value;
};

SBD_FI STree& s_tree(const SearchArgs& a, int i) { return *reinterpret_cast<STree*>(a.ws + (size_t)i * a.tree_bytes); }
SBD_FI SNode* s_nodes(const SearchArgs& a, int i) { return reinterpret_cast<SNode*>(a.ws + (size_t)i * a.tree_bytes + sizeof(STree)); }
SBD_FI double s_sign(int seat) { return seat ? -1.0 : 1.0; }

// node j of tree i from the working set g, which holds the record s as unpack(s) gives it
SBD_FI void s_write_node(SNode& nd, const G& g, const SbState& s, int parent, int action, int max_steps) {
  store_state(&nd.rec, s);
  int4* c = reinterpret_cast<int4*>(nd.child);
  #pragma unroll 1
  for (int k = 0; k < SB_N_ACTIONS / 4; k++) c[k] = make_int4(0, 0, 0, 0);
  u32 m[SB_MASK_WORDS];  // legal_mask works on thread-local arrays
  legal_mask(g, m);
  for (int k = 0; k < SB_MASK_WORDS; k++) nd.mask[k] = m[k];
  nd.parent = parent;
  nd.W = 0.0;
  nd.N = 0;
  nd.action = (u8)action;
  nd.seat = g.player_sign == 1 ? 0 : 1;
  const bool term = env_over(g, max_steps);
  nd.terminal = term ? 1 : 0;
  const int r = term ? env_result(g) : -1;
  nd.tval = r == 0 ? 1 : r == 1 ? -1 : 0;  // FIRST won / SECOND won / draw, timeout or engine status
}

// the leaf outputs of tree i: node nd, whose record unpacks to g
SBD_FI void s_emit(const SearchArgs& a, int i, const G& g, const SNode& nd, int kind) {
  if (a.leaf_states) store_state(a.leaf_states + (size_t)i * SB_STATE_BYTES, nd.rec);
  if (a.masks) for (int k = 0; k < SB_MASK_WORDS; k++) a.masks[(size_t)i * SB_MASK_WORDS + k] = nd.mask[k];
  if (a.obs) {
    const int e = observe(g, a.obs + (size_t)i * SB_OBS_INTS);
    if (a.obs_err) a.obs_err[i] = (u8)e;
  } else if (a.obs_err) {
    int scratch[SB_OBS_INTS];
    a.obs_err[i] = (u8)observe(g, scratch);
  }
  if (a.to_move) a.to_move[i] = nd.seat;
  if (a.leaf_kind) a.leaf_kind[i] = (u8)kind;
}
SBD_FI bool s_needs_record(const SearchArgs& a) { return a.obs || a.obs_err; }
// emit an existing node: unpack its record only when the observation is asked for
SBD_FI void s_emit_node(const SearchArgs& a, int i, G& g, const SNode& nd, int kind) {
  if (s_needs_record(a)) {
    __align__(16) SbState s;
    load_state(s, &nd.rec);
    unpack(g, s);
  }
  s_emit(a, i, g, nd, kind);
}

// store the caller's prior / value for the pending leaf and add its value (FIRST's view) to every node up to the root
SBD_FI void s_backup(const SearchArgs& a, int i, STree& t, SNode* nodes) {
  if (t.kind == SEARCH_FULL) return;
  SNode& leaf = nodes[t.leaf];
  double v;
  if (t.kind == SEARCH_TERMINAL) v = (double)leaf.tval;
  else {
    const float* p = a.prior + (size_t)i * SB_N_ACTIONS;
    #pragma unroll 1
    for (int k = 0; k < SB_N_ACTIONS; k++) leaf.prior[k] = p[k];
    v = __dmul_rn(s_sign(leaf.seat), (double)a.value[i]);
  }
  #pragma unroll 1
  for (int j = t.leaf; j >= 0; j = nodes[j].parent) {
    nodes[j].N += 1;
    nodes[j].W = __dadd_rn(nodes[j].W, v);
  }
}

// PUCT at a non-terminal node: score = q + u, q = sgn * W(child) / n_a (fpu when n_a = 0),
// u = ((c_puct * P) * sqrt(N)) / (1 + n_a); correctly rounded FP64 in this order, ties to the lowest action id
SBD_FI int s_select(const SearchArgs& a, const SNode* nodes, const SNode& nd) {
  const double sgn = s_sign(nd.seat), sq = __dsqrt_rn((double)nd.N);
  int best = -1;
  double best_score = 0.0;
  #pragma unroll 1
  for (int w = 0; w < SB_MASK_WORDS; w++) {
    u32 m = nd.mask[w];
    while (m) {
      const int act = w * 32 + __ffs(m) - 1;
      m &= m - 1;
      const int c = nd.child[act];
      const int na = c ? nodes[c].N : 0;
      const double q = na ? __ddiv_rn(__dmul_rn(sgn, nodes[c].W), (double)na) : a.fpu;
      const double u = __ddiv_rn(__dmul_rn(__dmul_rn(a.c_puct, (double)nd.prior[act]), sq), (double)(1 + na));
      const double score = __dadd_rn(q, u);
      if (best < 0 || score > best_score) { best = act; best_score = score; }
    }
  }
  return best;
}

// the header of tree i and the leaf outputs of its root, whose record s unpacks to g: sb_search_begin's tree (kept = 0:
// node 0 is written from s), or one whose first `kept` nodes sb_search_advance carried over (node 0 already holds s)
SBD_FI void s_start(const SearchArgs& a, int i, const G& g, const SbState& s, int kept) {
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  if (!kept) s_write_node(nodes[0], g, s, -1, SB_ACTION_PASS, a.max_steps);
  t.used = kept ? kept : 1;
  t.leaf = 0;
  t.kind = nodes[0].terminal ? SEARCH_TERMINAL : SEARCH_EVAL;
  t.max_steps = a.max_steps;
  s_emit(a, i, g, nodes[0], t.kind);
}

__global__ void __launch_bounds__(TPB_GAME) k_search_begin(const SearchArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  s_start(a, i, g, s, 0);
}

__global__ void __launch_bounds__(TPB_GAME) k_search_simulate(const SearchArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  s_backup(a, i, t, nodes);
  if (t.kind == SEARCH_FULL || t.used >= a.max_nodes) {  // the tree stops: the root is emitted, nothing is pending
    t.kind = SEARCH_FULL;
    s_emit_node(a, i, g, nodes[0], SEARCH_FULL);
    return;
  }
  int j = 0;
  #pragma unroll 1
  while (!nodes[j].terminal) {
    const int act = s_select(a, nodes, nodes[j]);
    const int c = nodes[j].child[act];
    if (!c) {  // expand: the child is the record sb_step(parent, act) produces
      __align__(16) SbState s;
      load_state(s, &nodes[j].rec);
      unpack(g, s);
      game_step(g, act);
      end_of_step(g);
      pack(g, s);
      unpack(g, s);  // the working set as the next sb_* call would unpack it from the child's record
      const int k = t.used++;
      s_write_node(nodes[k], g, s, j, act, t.max_steps);
      nodes[j].child[act] = k;
      t.leaf = k;
      t.kind = nodes[k].terminal ? SEARCH_TERMINAL : SEARCH_EVAL;
      s_emit(a, i, g, nodes[k], t.kind);
      return;
    }
    j = c;
  }
  t.leaf = j;  // an existing terminal node (or a terminal root): its game value is backed up again
  t.kind = SEARCH_TERMINAL;
  s_emit_node(a, i, g, nodes[j], SEARCH_TERMINAL);
}

// one simulation's walk after the backup, as k_search_simulate's but checked (the Gumbel kernel): select(j, c) chooses the
// action at the non-terminal node j and sets c to its child (0 = none), already checked against the node count; the
// descent stops after max_nodes levels, and a selection without an action (act < 0) stops the tree, as sb_ismcts does.
template <class Select>
SBD_FI void s_walk(const SearchArgs& a, int i, G& g, STree& t, SNode* nodes, Select select) {
  int j = 0;
  #pragma unroll 1
  for (int d = 0; !nodes[j].terminal; d++) {
    int c;
    const int act = d < a.max_nodes ? select(j, c) : -1;
    if (act < 0) {  // only a workspace not written by sb_search_begin gets here: the tree stops
      t.kind = SEARCH_FULL;
      s_emit_node(a, i, g, nodes[0], SEARCH_FULL);
      return;
    }
    if (!c) {  // expand: the child is the record sb_step(parent, act) produces
      __align__(16) SbState s;
      load_state(s, &nodes[j].rec);
      unpack(g, s);
      game_step(g, act);
      end_of_step(g);
      pack(g, s);
      unpack(g, s);  // the working set as the next sb_* call would unpack it from the child's record
      const int k = t.used++;
      s_write_node(nodes[k], g, s, j, act, t.max_steps);
      nodes[j].child[act] = k;
      t.leaf = k;
      t.kind = nodes[k].terminal ? SEARCH_TERMINAL : SEARCH_EVAL;
      s_emit(a, i, g, nodes[k], t.kind);
      return;
    }
    j = c;
  }
  t.leaf = j;  // an existing terminal node (or a terminal root): its game value is backed up again
  t.kind = SEARCH_TERMINAL;
  s_emit_node(a, i, g, nodes[j], SEARCH_TERMINAL);
}

// visits, q and root_value of tree i (sb_search_end)
SBD_FI void s_read_out(const SearchArgs& a, int i, const SNode* nodes) {
  const SNode& root = nodes[0];
  const double sgn = s_sign(root.seat);
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) {
    const int c = root.child[act];
    const int na = c ? nodes[c].N : 0;
    a.visits[(size_t)i * SB_N_ACTIONS + act] = na;
    a.q[(size_t)i * SB_N_ACTIONS + act] = na ? __ddiv_rn(__dmul_rn(sgn, nodes[c].W), (double)na) : __longlong_as_double(0x7FF8000000000000ll);
  }
  a.root_value[i] = __ddiv_rn(__dmul_rn(sgn, root.W), (double)root.N);
}

// back up the last pending leaf (the tree then holds nothing pending) and read out the root's edges
__global__ void __launch_bounds__(TPB_GAME) k_search_end(const SearchArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  s_backup(a, i, t, nodes);
  t.kind = SEARCH_FULL;
  s_read_out(a, i, nodes);
}
