// Gumbel MuZero search (Danihelka, Guez, Schrittwieser & Silver, "Policy improvement by planning with Gumbel", ICLR 2022)
// for both tree searches: sb_search_simulate_gumbel / sb_search_end_gumbel over the perfect-information trees of
// sb_search.cuh, sb_ismcts_simulate_gumbel / sb_ismcts_end_gumbel over the information-set trees of sb_ismcts.cuh.  A search
// is the existing begin, S Gumbel simulate calls and the Gumbel end; backup, expansion, leaf emission, the workspaces and
// the begin kernels are those of PUCT.  Only the selection rule and the read-out differ (DESIGN.md 8.9):
//
//   at a non-terminal node s with seat sign sgn, legal set A (8.6: the node's legal ids; 8.8: the world's legal
//   representative ids, children matched by move code), n_a / W_a the N / W of a's child (0 without one), q_a = sgn W_a / n_a:
//   vhat   = sgn (W(s) - sum W(c)) / (N(s) - sum N(c)) over all children c of s; 0 when the denominator is < 1
//   vmix   = (vhat + sumN * (sum_{n_a>0} pt_a q_a / sum_{n_a>0} pt_a)) / (1 + sumN), sumN = sum_A n_a, pt_a = max(p_a, 2^-126)
//            (the product term is 0 when no a has n_a > 0)
//   qbar_a = q_a if n_a > 0 else vmix;  qhat_a = (qbar_a - min_A qbar) / max(max_A qbar - min_A qbar, 1e-8)
//   sigma_a = ((c_visit + max_A n_a) * c_scale) * qhat_a;  logit_a = es_log(p_a) if p_a > 0 else -1e9
//   interior: z_a = logit_a + sigma_a, e_a = es_exp(z_a - max_A z) (0 when that is < -700), pi_a = e_a / sum_A e,
//             choose argmax_A (pi_a - n_a / (1 + sumN))
//   root (node 0) at call k = 1..S: m = min(max_considered, |A|), c = seq(m, S)[k - 1], E = {a in A : n_a = c} (A if empty),
//             choose argmax_E max(-1e9, (g_a + logit_a) + sigma_a), g the caller's Gumbel noise
//   end:      action = argmax over {a in A : n_a = max_A n} of (g_a + logit_a) + sigma_a (255 when max_A n = 0),
//             policy = f32(pi) with the final counts, 0 outside A
// Every operation is a correctly rounded FP64 __d*_rn in the order written; log / exp are es_log / es_exp (sb_es.cuh, the
// oracle's sbo_det_log / sbo_det_exp).  Sums run in the order the edges are visited: 8.6 in increasing id order; 8.8 during
// simulate over the children in sibling-walk order (newest first), then the ids without a child in increasing order, and at
// the end in increasing root id order.  max(x, y) is x > y ? x : y, so a NaN never wins a comparison; arg-max ties go to the
// lowest id; an arg-max in which nothing scores takes the lowest id of its set, so a selection over a non-empty A always
// returns a legal id.
//
// seq(m, S), mctx's get_sequence_of_considered_visits, the visit count the root's chosen action has before call k:
//   if m <= 1: return 0, 1, ..., S-1
//   L = ceil(log2 m); visits = [0]*m; k = m; out = []
//   while len(out) < S:
//       extra = max(1, S // (L * k))
//       repeat extra times: out += visits[:k]; visits[i] += 1 for i < k
//       k = max(2, k // 2)
//   return out[:S]
// The first k entries of visits are always equal, so gb_seq replays this with one counter, per tree and call, in O(log S).
//
// Fault safety: every node index read from the workspace by the selection and the read-out is checked against the tree's
// node count, and the descents are bounded by max_nodes (s_walk, ism_walk); 8.6's backup is s_backup, unchanged, which like
// the PUCT kernels trusts the parent chain of a workspace written by sb_search_begin.  The 8.8 kernels compute the per-node
// quantities in bounded sibling-walk passes plus a pass over the ids without a child and keep no per-id table on the stack.
#pragma once
#include "sb_es.cuh"
#include "sb_ismcts.cuh"

struct GumbelArgs {
  const float* gumbel;                        // f32[n,156], the same for every call of one search
  int sim, num_simulations, max_considered;   // call index k (1..S) of simulate, S, the root's considered actions
  double c_visit, c_scale;
  int* action; float* policy;                 // end: i32[n], f32[n,156]
};
#define GUMBEL_MAX_SIMULATIONS (1 << 24)
#define GUMBEL_NO_ACTION 255

// seq(m, S)[k], 0 <= k < S
SBD_FI int gb_seq(int m, int S, int k) {
  if (m <= 1) return k;
  int L = 0;
  while ((1 << L) < m) L++;
  int pos = 0, v = 0, w = m;
  #pragma unroll 1
  for (;;) {
    const int q = S / (L * w), extra = q > 1 ? q : 1;
    if (k < pos + extra * w) return v + (k - pos) / w;
    pos += extra * w;
    v += extra;
    w = w / 2 > 2 ? w / 2 : 2;
  }
}
SBD_FI double gb_logit(float p) { const double d = (double)p; return d > 0.0 ? es_log(d) : -1e9; }
SBD_FI double gb_ptilde(float p) { const double d = (double)p, tiny = 1.1754943508222875e-38; return d > tiny ? d : tiny; }

// the per-node quantities of the rule, from passes over the edges of one node
struct GbNode {
  double sgn, vmix, qmin, qden, sig, zmax, esum;
  int sum_n, max_n, count, lo, lo_child, considered;  // considered: edges with n_a == the root's target count
};
SBD_FI double gb_q(const GbNode& s, int n, double w) { return n > 0 ? __ddiv_rn(__dmul_rn(s.sgn, w), (double)n) : s.vmix; }
SBD_FI double gb_sigma(const GbNode& s, int n, double w) {
  return __dmul_rn(s.sig, __ddiv_rn(__dadd_rn(gb_q(s, n, w), -s.qmin), s.qden));
}
SBD_FI double gb_e(const GbNode& s, double z) {
  const double d = __dadd_rn(z, -s.zmax);
  return d >= -700.0 ? es_exp(d) : 0.0;
}

// Edges: each(f) calls f(act, n, W, child) once per a in A in the summation order; vhat(nd) the node value.
// target: the root's considered visit count (-1 elsewhere); softmax: also compute max z and sum e.
template <class Edges, class Node>
SBD_FI void gb_node(GbNode& s, const Edges& E, const Node& nd, double c_visit, double c_scale, int target, bool softmax) {
  s.sgn = s_sign(nd.seat);
  int sum_n = 0, max_n = 0, count = 0, lo = SB_N_ACTIONS, lo_child = 0, considered = 0;
  bool visited = false;
  double sp = 0.0, spq = 0.0;
  E.each([&](int act, int n, double w, int c) {
    count++;
    sum_n += n;
    if (n > max_n) max_n = n;
    if (act < lo) { lo = act; lo_child = c; }
    if (n == target) considered++;
    if (n > 0) {
      const double pt = gb_ptilde(nd.prior[act]);
      visited = true;
      sp = __dadd_rn(sp, pt);
      spq = __dadd_rn(spq, __dmul_rn(pt, __ddiv_rn(__dmul_rn(s.sgn, w), (double)n)));
    }
  });
  s.sum_n = sum_n; s.max_n = max_n; s.count = count; s.lo = lo; s.lo_child = lo_child; s.considered = considered;
  const double vhat = E.vhat(nd, s.sgn);
  const double mix = visited ? __dmul_rn((double)sum_n, __ddiv_rn(spq, sp)) : 0.0;
  s.vmix = __ddiv_rn(__dadd_rn(vhat, mix), (double)(1 + sum_n));
  double qmin = __longlong_as_double(0x7FF0000000000000ll), qmax = -qmin;
  E.each([&](int act, int n, double w, int c) {
    const double q = gb_q(s, n, w);
    if (q < qmin) qmin = q;
    if (q > qmax) qmax = q;
  });
  const double d = __dadd_rn(qmax, -qmin);
  s.qmin = qmin;
  s.qden = d > 1e-8 ? d : 1e-8;
  s.sig = __dmul_rn(__dadd_rn(c_visit, (double)max_n), c_scale);
  s.zmax = -__longlong_as_double(0x7FF0000000000000ll);
  s.esum = 0.0;
  if (!softmax) return;
  double zmax = s.zmax;
  E.each([&](int act, int n, double w, int c) {
    const double z = __dadd_rn(gb_logit(nd.prior[act]), gb_sigma(s, n, w));
    if (z > zmax) zmax = z;
  });
  s.zmax = zmax;
  double esum = 0.0;
  E.each([&](int act, int n, double w, int c) {
    esum = __dadd_rn(esum, gb_e(s, __dadd_rn(gb_logit(nd.prior[act]), gb_sigma(s, n, w))));
  });
  s.esum = esum;
}

// the selection at node nd (root: tree i's call gb.sim), child <- the chosen id's child (the edge set's "none" when it has
// none); -1 when A is empty
template <class Edges, class Node>
SBD_FI int gb_select(const GumbelArgs& gb, int i, const Edges& E, const Node& nd, bool root, int& child) {
  GbNode s;
  if (!root) {
    gb_node(s, E, nd, gb.c_visit, gb.c_scale, -1, true);
    if (s.count == 0) return -1;
    int best = -1, best_child = s.lo_child;
    double best_score = -__longlong_as_double(0x7FF0000000000000ll);
    const double inv = (double)(1 + s.sum_n);
    E.each([&](int act, int n, double w, int c) {
      const double pi = __ddiv_rn(gb_e(s, __dadd_rn(gb_logit(nd.prior[act]), gb_sigma(s, n, w))), s.esum);
      const double score = __dadd_rn(pi, -__ddiv_rn((double)n, inv));
      if (score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_child = c; }
    });
    if (best < 0) { child = s.lo_child; return s.lo; }
    child = best_child;
    return best;
  }
  // the root: the considered count needs |A|, so one counting pass first
  int count = 0;
  E.each([&](int act, int n, double w, int c) { count++; });
  if (count == 0) return -1;
  const int m = gb.max_considered < count ? gb.max_considered : count;
  const int target = gb_seq(m, gb.num_simulations, gb.sim - 1);
  gb_node(s, E, nd, gb.c_visit, gb.c_scale, target, false);
  const bool all = s.considered == 0;
  const float* g = gb.gumbel + (size_t)i * SB_N_ACTIONS;
  int best = -1, best_child = s.lo_child;
  double best_score = -__longlong_as_double(0x7FF0000000000000ll);
  E.each([&](int act, int n, double w, int c) {
    if (!all && n != target) return;
    const double x = __dadd_rn(__dadd_rn((double)g[act], gb_logit(nd.prior[act])), gb_sigma(s, n, w));
    const double score = x > -1e9 ? x : -1e9;
    if (score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_child = c; }
  });
  if (best < 0) { child = s.lo_child; return s.lo; }
  child = best_child;
  return best;
}

// the read-out of tree i after the last backup: policy row and action over the root's edges E (nd the root)
template <class Edges, class Node>
SBD_FI void gb_read_out(const GumbelArgs& gb, int i, const Edges& E, const Node& nd) {
  float* pol = gb.policy + (size_t)i * SB_N_ACTIONS;
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) pol[act] = 0.f;
  GbNode s;
  gb_node(s, E, nd, gb.c_visit, gb.c_scale, -1, true);
  int best = -1, lo = GUMBEL_NO_ACTION;
  double best_score = -__longlong_as_double(0x7FF0000000000000ll);
  const float* g = gb.gumbel + (size_t)i * SB_N_ACTIONS;
  E.each([&](int act, int n, double w, int c) {
    const double z = __dadd_rn(gb_logit(nd.prior[act]), gb_sigma(s, n, w));
    pol[act] = (float)__ddiv_rn(gb_e(s, z), s.esum);
    if (n != s.max_n || n == 0) return;
    if (act < lo) lo = act;
    const double score = __dadd_rn(__dadd_rn((double)g[act], gb_logit(nd.prior[act])), gb_sigma(s, n, w));
    if (score > best_score || (score == best_score && act < best)) { best = act; best_score = score; }
  });
  gb.action[i] = best >= 0 ? best : lo;
}

// ---------------------------------------------------------------- 8.6: the perfect-information trees
// A = the node's legal ids in increasing order; a child index outside 1..lim-1 counts as none (0)
struct GbSearchEdges {
  const SNode* nodes;
  const SNode& nd;
  int lim;
  SBD_FI int child(int act) const { const int c = nd.child[act]; return c > 0 && c < lim ? c : 0; }
  template <class F> SBD_FI void each(F f) const {
    #pragma unroll 1
    for (int w = 0; w < SB_MASK_WORDS; w++) {
      u32 m = nd.mask[w];
      while (m) {
        const int act = w * 32 + __ffs(m) - 1;
        m &= m - 1;
        const int c = child(act);
        f(act, c ? nodes[c].N : 0, c ? nodes[c].W : 0.0, c);
      }
    }
  }
  // every child of a node sits at a legal id, so the children are those of the legal ids, in increasing id order
  SBD_FI double vhat(const SNode& s, double sgn) const {
    int sn = 0;
    double sw = 0.0;
    #pragma unroll 1
    for (int w = 0; w < SB_MASK_WORDS; w++) {
      u32 m = s.mask[w];
      while (m) {
        const int c = child(w * 32 + __ffs(m) - 1);
        m &= m - 1;
        if (c) { sn += nodes[c].N; sw = __dadd_rn(sw, nodes[c].W); }
      }
    }
    const int den = s.N - sn;
    return den < 1 ? 0.0 : __ddiv_rn(__dmul_rn(sgn, __dadd_rn(s.W, -sw)), (double)den);
  }
};

__global__ void __launch_bounds__(TPB_GAME) k_search_simulate_gumbel(const SearchArgs a, const GumbelArgs gb, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  if (t.used < 1 || t.used > a.max_nodes || (t.kind != SEARCH_FULL && (t.leaf < 0 || t.leaf >= t.used))) t.kind = SEARCH_FULL;
  s_backup(a, i, t, nodes);
  if (t.kind == SEARCH_FULL || t.used >= a.max_nodes) {  // the tree stops: the root is emitted, nothing is pending
    t.kind = SEARCH_FULL;
    s_emit_node(a, i, g, nodes[0], SEARCH_FULL);
    return;
  }
  const int lim = t.used;
  s_walk(a, i, g, t, nodes, [&](int j, int& c) {
    const GbSearchEdges E{nodes, nodes[j], lim};
    return gb_select(gb, i, E, nodes[j], j == 0, c);
  });
}

__global__ void __launch_bounds__(TPB_GAME) k_search_end_gumbel(const SearchArgs a, const GumbelArgs gb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  if (t.used < 1 || t.used > a.max_nodes || (t.kind != SEARCH_FULL && (t.leaf < 0 || t.leaf >= t.used))) t.kind = SEARCH_FULL;
  s_backup(a, i, t, nodes);
  t.kind = SEARCH_FULL;
  const int lim = t.used < 1 ? 1 : t.used > a.max_nodes ? a.max_nodes : t.used;
  const SNode& root = nodes[0];
  const GbSearchEdges E{nodes, root, lim};
  #pragma unroll 1
  for (int act = 0; act < SB_N_ACTIONS; act++) {  // sb_search_end's read-out, over the checked child indices
    const int c = E.child(act);
    const int na = c ? nodes[c].N : 0;
    a.visits[(size_t)i * SB_N_ACTIONS + act] = na;
    a.q[(size_t)i * SB_N_ACTIONS + act] = na ? __ddiv_rn(__dmul_rn(s_sign(root.seat), nodes[c].W), (double)na) : __longlong_as_double(0x7FF8000000000000ll);
  }
  a.root_value[i] = __ddiv_rn(__dmul_rn(s_sign(root.seat), root.W), (double)root.N);
  if (root.terminal) {  // A is empty: a terminal root never stores a prior
    #pragma unroll 1
    for (int act = 0; act < SB_N_ACTIONS; act++) gb.policy[(size_t)i * SB_N_ACTIONS + act] = 0.f;
    gb.action[i] = GUMBEL_NO_ACTION;
    return;
  }
  gb_read_out(gb, i, E, root);
}

// ---------------------------------------------------------------- 8.8: the information-set trees
// simulate: A = the current world's legal representatives; the children with a code legal in this world first (sibling
// walk, newest first), then the representative ids without a child in increasing order
struct GbIsmEdges {
  const INode* nodes;
  const INode& nd;
  int lim;
  const Ply& p;
  const u32* m;
  template <class F> SBD_FI void each(F f) const {
    u32 has[SB_MASK_WORDS] = {0, 0, 0, 0, 0};
    int c = nd.child;
    #pragma unroll 1
    for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling) {
      const int act = ism_action(p, m, nodes[c].code);
      if (act < 0 || ism_bit(has, act)) continue;  // the move does not exist in this world (or a repeated code)
      has[act >> 5] |= 1u << (act & 31);
      f(act, nodes[c].N, nodes[c].W, c);
    }
    #pragma unroll 1
    for (int w = 0; w < SB_MASK_WORDS; w++) {
      u32 r = m[w] & ~has[w];
      while (r) {
        const int act = w * 32 + __ffs(r) - 1;
        r &= r - 1;
        if (ism_rep(p, m, act)) f(act, 0, 0.0, -1);
      }
    }
  }
  SBD_FI double vhat(const INode& s, double sgn) const { return gb_ism_vhat(nodes, lim, s, sgn); }
  // every child of s in sibling-walk order
  static SBD_FI double gb_ism_vhat(const INode* nodes, int lim, const INode& s, double sgn) {
    int sn = 0;
    double sw = 0.0;
    int c = s.child;
    #pragma unroll 1
    for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling) { sn += nodes[c].N; sw = __dadd_rn(sw, nodes[c].W); }
    const int den = s.N - sn;
    return den < 1 ? 0.0 : __ddiv_rn(__dmul_rn(sgn, __dadd_rn(s.W, -sw)), (double)den);
  }
};
// end: A = the root ids whose stored code is set, in increasing id order, each with the child of its code
struct GbIsmRootEdges {
  const INode* nodes;
  const INode& nd;
  int lim;
  const ITree& t;
  template <class F> SBD_FI void each(F f) const {
    #pragma unroll 1
    for (int act = 0; act < SB_N_ACTIONS; act++) {
      const u32 code = t.root_code[act];
      if (code == ISM_NONE) continue;
      const int c = ism_find(nodes, lim, nd, code);
      f(act, c >= 0 ? nodes[c].N : 0, c >= 0 ? nodes[c].W : 0.0, c);
    }
  }
  SBD_FI double vhat(const INode& s, double sgn) const { return GbIsmEdges::gb_ism_vhat(nodes, lim, s, sgn); }
};

__global__ void __launch_bounds__(TPB_GAME) k_ismcts_simulate_gumbel(const SearchArgs a, const GumbelArgs gb, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  G g;
  init_g(g, s_cards, wt);
  ITree& t = ism_tree(a, i);
  INode* nodes = ism_nodes(a, i);
  ism_backup(a, i, t, nodes);
  __align__(16) SbState s;
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);  // this call's world at the root
  unpack(g, s);
  u32 m[SB_MASK_WORDS];
  legal_mask(g, m);
  if (t.kind == SEARCH_FULL || t.used < 1 || t.used >= a.max_nodes) {  // the tree stops: the world's root is emitted
    t.kind = SEARCH_FULL;
    ism_emit(a, i, g, s, m, SEARCH_FULL);
    return;
  }
  ism_walk(a, i, g, t, nodes, s, m, [&](int j, int lim, int& c) {
    const GbIsmEdges E{nodes, nodes[j], lim, g.pl[g.local_order], m};
    return gb_select(gb, i, E, nodes[j], j == 0, c);
  });
}

__global__ void __launch_bounds__(TPB_GAME) k_ismcts_end_gumbel(const SearchArgs a, const GumbelArgs gb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  ITree& t = ism_tree(a, i);
  INode* nodes = ism_nodes(a, i);
  ism_backup(a, i, t, nodes);
  t.kind = SEARCH_FULL;
  const int lim = ism_lim(t, a.max_nodes);
  if (lim < 1) {
    ism_read_out_empty(a, i);
    #pragma unroll 1
    for (int act = 0; act < SB_N_ACTIONS; act++) gb.policy[(size_t)i * SB_N_ACTIONS + act] = 0.f;
    gb.action[i] = GUMBEL_NO_ACTION;
    return;
  }
  ism_read_out(a, i, t, nodes, lim);
  const GbIsmRootEdges E{nodes, nodes[0], lim, t};
  gb_read_out(gb, i, E, nodes[0]);
}
