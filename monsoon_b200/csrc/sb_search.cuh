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
//
// Fault safety, the one rule of every kernel over these trees (PUCT here, Gumbel in sb_gumbel.cuh, batch in
// sb_search_batch.cuh): every index read from the workspace is checked before it is dereferenced.  The node count must lie in
// 1..max_nodes (sb_count), the pending leaf below it, and a parent below its child, so every walk up ends at the root
// (sb_add_path).  Every child is created after its parent, so a child link the selection reads must be 0 (none) or lie
// above its node and below the count; every walk down then moves to higher indices and ends within the count.  A failed
// check stops the tree: kind SEARCH_FULL, the root emitted, nothing pending.  The read-out (s_read_out) counts a root child link
// outside 1..count-1 as none.  The advance (sb_reuse.cuh) checks what it reads from its source workspace by its own rules.
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

// the arguments of every search kernel; an entry point sets the fields its call uses, the others stay null / 0
struct SearchArgs {
  int n, max_nodes;
  unsigned char* ws; size_t tree_bytes;
  const u8* roots = nullptr; int max_steps = 0;
  const float* prior = nullptr; const float* value = nullptr; double c_puct = 0.0, fpu = 0.0;
  u8* leaf_states = nullptr; int* obs = nullptr; u32* masks = nullptr; u8* obs_err = nullptr; u8* to_move = nullptr;
  u8* leaf_kind = nullptr;
  int* visits = nullptr; double* q = nullptr; double* root_value = nullptr;
  SearchArgs(int n_, int max_nodes_, void* ws_, size_t tree_bytes_)
      : n(n_), max_nodes(max_nodes_), ws((unsigned char*)ws_), tree_bytes(tree_bytes_) {}
};

#define S_QNAN __longlong_as_double(0x7FF8000000000000ll)  // q of an edge without visits, root_value of an empty read-out

SBD_FI STree& s_tree(const SearchArgs& a, int i) { return *reinterpret_cast<STree*>(a.ws + (size_t)i * a.tree_bytes); }
SBD_FI SNode* s_nodes(const SearchArgs& a, int i) { return reinterpret_cast<SNode*>(a.ws + (size_t)i * a.tree_bytes + sizeof(STree)); }
SBD_FI double s_sign(int seat) { return seat ? -1.0 : 1.0; }
// PUCT's score of an edge with n_a visits and prior p at a node with sq = sqrt(N): q + u, q = x / n_a (fpu when n_a = 0;
// x is the edge's value sum from the node's point of view), u = ((c_puct * p) * sq) / (1 + n_a), correctly rounded FP64
SBD_FI double s_score(const SearchArgs& a, int na, double x, float p, double sq) {
  const double q = na ? __ddiv_rn(x, (double)na) : a.fpu;
  return __dadd_rn(q, __ddiv_rn(__dmul_rn(__dmul_rn(a.c_puct, (double)p), sq), (double)(1 + na)));
}
// sb_step on the working set g after action act: g and s become what the next sb_* call unpacks from the child's record
SBD_FI void s_step(G& g, SbState& s, int act) {
  game_step(g, act);
  end_of_step(g);
  pack(g, s);
  unpack(g, s);
}

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

// the node count of tree t, 0 when it is not in 1..max_nodes
SBD_FI int sb_count(const STree& t, int max_nodes) { return t.used >= 1 && t.used <= max_nodes ? t.used : 0; }

// add v to W and 1 to N of node j and every node above it, leaf up to root; false on a parent link that is not below its child
SBD_FI bool sb_add_path(SNode* nodes, int j, double v) {
  #pragma unroll 1
  while (true) {
    nodes[j].N += 1;
    nodes[j].W = __dadd_rn(nodes[j].W, v);
    if (j == 0) return true;
    const int p = nodes[j].parent;
    if (p < 0 || p >= j) return false;
    j = p;
  }
}

// store row r's prior / value as node k's (kind EVAL; TERMINAL: its game value) and add the value (FIRST's view) to every
// node up to the root; false on a bad index
SBD_FI bool sb_backup_node(const SearchArgs& a, SNode* nodes, int used, size_t r, int k, int kind) {
  if (k < 0 || k >= used) return false;
  SNode& leaf = nodes[k];
  double v;
  if (kind == SEARCH_TERMINAL) v = (double)leaf.tval;
  else {
    const float* p = a.prior + r * SB_N_ACTIONS;
    #pragma unroll 1
    for (int x = 0; x < SB_N_ACTIONS; x++) leaf.prior[x] = p[x];
    v = __dmul_rn(s_sign(leaf.seat), (double)a.value[r]);
  }
  return sb_add_path(nodes, k, v);
}

// back up the leaf the header of tree i holds pending, with row i's prior / value; returns the node count, 0 when nothing
// was pending or a check failed (the tree then stops: kind SEARCH_FULL)
SBD_FI int s_backup(const SearchArgs& a, int i, STree& t, SNode* nodes) {
  if (t.kind == SEARCH_FULL) return 0;
  const int used = sb_count(t, a.max_nodes);
  if (used > 0 && sb_backup_node(a, nodes, used, i, t.leaf, t.kind)) return used;
  t.kind = SEARCH_FULL;
  return 0;
}

// the child link of nd at act, 0 (none) when it lies outside lo+1..used-1
SBD_FI int s_child(const SNode& nd, int act, int lo, int used) { const int c = nd.child[act]; return c > lo && c < used ? c : 0; }

// PUCT at the non-terminal node j, with the virtual visits V of a batch call (Virt: virt; else V = 0, 8.6's scores bit for
// bit, as x - vl * 0 and sqrt(N + 0) are exact; a compile-time flag, so neither search tests it per edge): n_a = N(c) + V(c), q = ((sgn * W(c)) - (vl * V(c))) / n_a (fpu when n_a = 0),
// u = ((c_puct * P) * sqrt(N(j) + V(j))) / (1 + n_a), score = q + u; correctly rounded FP64 in this order, ties to the lowest
// action id.  Returns the action, child <- its child link (0 = none); -1 when no action is legal or a child link is neither 0 nor
// in j+1..used-1.
template <bool Virt>
SBD_FI int s_select(const SearchArgs& a, const SNode* nodes, const int* virt, double vl, int j, int used, int& child) {
  const SNode& nd = nodes[j];
  const double sgn = s_sign(nd.seat), sq = __dsqrt_rn((double)(nd.N + (Virt ? virt[j] : 0)));
  int best = -1, best_c = 0;
  double best_score = 0.0;
  #pragma unroll 1
  for (int w = 0; w < SB_MASK_WORDS; w++) {
    u32 m = nd.mask[w];
    while (m) {
      const int act = w * 32 + __ffs(m) - 1;
      m &= m - 1;
      const int c = nd.child[act];
      if (c != 0 && (c <= j || c >= used)) return -1;
      const int vc = Virt && c ? virt[c] : 0;
      const int na = c ? nodes[c].N + vc : 0;
      double x = 0.0;
      if (na) x = Virt ? __dsub_rn(__dmul_rn(sgn, nodes[c].W), __dmul_rn(vl, (double)vc)) : __dmul_rn(sgn, nodes[c].W);
      const double score = s_score(a, na, x, nd.prior[act], sq);
      if (best < 0 || score > best_score) { best = act; best_c = c; best_score = score; }
    }
  }
  child = best_c;
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

// node k of tree i, child of p by act, becomes the record sb_step(p's record, act) produces: written, and emitted at row r
// (working set g); returns its leaf kind
SBD_FI int s_expand(const SearchArgs& a, int r, G& g, const STree& t, SNode* nodes, int k, int p, int act) {
  __align__(16) SbState s;
  load_state(s, &nodes[p].rec);
  unpack(g, s);
  s_step(g, s, act);
  s_write_node(nodes[k], g, s, p, act, t.max_steps);
  const int kind = nodes[k].terminal ? SEARCH_TERMINAL : SEARCH_EVAL;
  s_emit(a, r, g, nodes[k], kind);
  return kind;
}

// one simulate call of tree i (k_search_simulate, k_search_simulate_gumbel): back up the pending leaf, stop when the tree
// is full, else walk down from the root and expand or emit a leaf.  select(nodes, j, used, c) chooses the action at the
// non-terminal node j and sets c to its child link, 0 (none) or in j+1..used-1; a selection without an action (act < 0)
// stops the tree.  As every step goes to a higher node index, the walk ends within the node count.
template <class Select>
SBD_FI void s_simulate(const SearchArgs& a, int i, G& g, Select select) {
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  const int used = s_backup(a, i, t, nodes);
  bool stop = used == 0 || used >= a.max_nodes;
  int j = 0;
  #pragma unroll 1
  while (!stop && !nodes[j].terminal) {
    int c;
    const int act = select(nodes, j, used, c);
    if (act < 0) {
      stop = true;
      break;
    }
    if (!c) {
      const int k = t.used++;
      const int kind = s_expand(a, i, g, t, nodes, k, j, act);
      nodes[j].child[act] = k;
      t.leaf = k;
      t.kind = kind;
      return;
    }
    j = c;
  }
  // one emit outside the walk: a stopped tree (full, or a check failed) emits its root with nothing pending; an existing
  // terminal node (or a terminal root) is the leaf, and its game value is backed up again
  if (stop) j = 0;
  else t.leaf = j;
  t.kind = stop ? SEARCH_FULL : SEARCH_TERMINAL;
  s_emit_node(a, i, g, nodes[j], t.kind);
}

__global__ void __launch_bounds__(TPB_GAME) k_search_simulate(const SearchArgs a, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  s_simulate(a, i, g, [&](const SNode* nodes, int j, int used, int& c) { return s_select<false>(a, nodes, nullptr, 0.0, j, used, c); });
}

// visits, q and root_value of tree i whose node count is used (0: none usable); a root child link outside 1..used-1 counts
// as none
SBD_FI void s_read_out(const SearchArgs& a, int i, const SNode* nodes, int used) {
  const SNode& root = nodes[0];
  const double sgn = s_sign(root.seat);
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) {
    const int c = s_child(root, act, 0, used);
    const int na = c ? nodes[c].N : 0;
    a.visits[(size_t)i * SB_N_ACTIONS + act] = na;
    a.q[(size_t)i * SB_N_ACTIONS + act] = na ? __ddiv_rn(__dmul_rn(sgn, nodes[c].W), (double)na) : S_QNAN;
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
  s_read_out(a, i, nodes, sb_count(t, a.max_nodes));
}
