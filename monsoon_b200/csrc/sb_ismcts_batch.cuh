// Several leaves per tree per call for the information-set search, under virtual loss (sb_ismcts_simulate_batch /
// sb_ismcts_end_batch, DESIGN.md 8.12).  8.11's contract over 8.8's tree, with one world per slot: a batch call backs up the
// L leaves the previous call left pending, then slot l walks from the root through its own world l (det row g * L + l), as
// ism_simulate does, counting the paths of the earlier slots of the same call as virtual visits V that carry a loss.  The
// definition is sequential, slot by slot; the kernel below computes it in parallel.
//
// Workspace: sb_ismcts_workspace_bytes(n, max_nodes) bytes of 8.8's layout (tree g at ws + g * tree_bytes), then tree g's
// tail at ws + n * tree_bytes + g * tail_bytes, tail_bytes = 16-byte multiple of 16 * L + 4 * max_nodes:
//   slot  int4[L]           pending slot l: {node index, slot kind, game value for FIRST of a TERMINAL slot in its world, 0}
//   virt  i32[max_nodes]    virtual visits V of this call, zero between calls
// A tree is in header form (ITree.kind 0, 1 or 2, one pending leaf) after begin, advance or a plain simulate, and in batch
// form (kind SEARCH_BATCH, the L slots pending) after a batch call.  A batch call on a header-form tree backs up its single
// leaf from slot 0's row and zeroes V.
//
// One launch per call (k_ismcts_simulate_batch), a wavefront: one lane per slot, the lanes of a tree in one CTA (L rounded up
// to a power of two, ISM_BATCH_CTA threads per CTA, or one CTA of 128 / 256 lanes per tree for L > 64).  In step t, lane l
// takes its decision at depth t - l in its own world and steps that world.  Slot l's decision at depth d reads only what the
// slots below l did down to depth d + 1, which they did in earlier steps, so the result is the sequential one after L +
// depth steps, with two CTA barriers per step.  What a step reads and what it writes are split by a barrier, and a node at
// depth d is marked by slot l only in step l + d - 1, so no two lanes write one counter in one step (no atomics).  Edges the
// walks need are recorded in a per-call table in shared memory, entry l = slot l's edge (parent, move code, V); a later slot
// that picks the code of an earlier slot's entry at the same parent stops there (COLLISION).  Once the wavefront is done,
// lane 0 of each tree takes the new nodes in slot order and links each at the head of its parent's children, so node
// indices, sibling order and the FULL cut-off follow slot order, not wavefront time.  Each lane still holds its world at the
// leaf and emits it in the same launch.  sb_ismcts_end_batch is one launch (k_ismcts_end_batch): backup, kind SEARCH_FULL,
// ism_end's read-out.  No handle scratch, no atomics, no host synchronisation.
//
// Fault safety: 8.8's rule (sb_ismcts.cuh): every node index read from the workspace is checked against the node count
// before it is dereferenced, sibling walks and parent chains are bounded by it, the descent by max_nodes; in addition a
// pending slot's node must lie below the count.  A failed check stops the tree: kind SEARCH_FULL, every slot FULL, the
// world's root emitted (a stopped tree's V is never read again, the next header-form call zeroes it).
#pragma once
#include "sb_ismcts.cuh"
#include "sb_search_batch.cuh"

#define ISM_BATCH_CTA 64        // threads per CTA of k_ismcts_simulate_batch when a tree's lanes fit in it
#define ISM_BATCH_MAX_CTA 256   // one tree of 256 lanes
#define ISM_WALK -1             // lane states besides the slot kinds: still walking,
#define ISM_NEW 4               // the walk needs a node for the edge it recorded in the table,
#define ISM_FAIL 5              // a check failed or no representative is legal (the tree stops)

struct IsmBatchArgs {
  int leaves, lanes;        // L, and L rounded up to a power of two
  double vl;                // virtual loss per virtual visit
  unsigned char* tail;      // ws + n * tree_bytes
  size_t tail_bytes;
};

SBD_FI int4* ib_slots(const IsmBatchArgs& b, int i) { return reinterpret_cast<int4*>(b.tail + (size_t)i * b.tail_bytes); }
SBD_FI int* ib_virt(const IsmBatchArgs& b, int i) { return reinterpret_cast<int*>(b.tail + (size_t)i * b.tail_bytes + 16 * (size_t)b.leaves); }

// ism_backup of node k: row r's prior / value (EVAL) or the game value tval (TERMINAL) added to every node up to the root;
// false on a node or parent index outside the count
SBD_FI bool ib_backup_node(const SearchArgs& a, INode* nodes, int lim, size_t r, int k, int kind, int tval) {
  if (!ism_in(k, lim)) return false;
  INode& leaf = nodes[k];
  double v;
  if (kind == SEARCH_TERMINAL) v = (double)tval;
  else {
    const float* p = a.prior + r * SB_N_ACTIONS;
    #pragma unroll 1
    for (int x = 0; x < SB_N_ACTIONS; x++) leaf.prior[x] = p[x];
    v = __dmul_rn(s_sign(leaf.seat), (double)a.value[r]);
  }
  int j = k;
  #pragma unroll 1
  for (int d = 0; d < lim && ism_in(j, lim); d++) {
    nodes[j].N += 1;
    nodes[j].W = __dadd_rn(nodes[j].W, v);
    j = nodes[j].parent;
  }
  return j == -1;
}

// what the previous call left pending in tree i: the header-form leaf (slot 0's row) or the L slots in ascending order.
// Returns the node count, 0 when the tree is (or now is) stopped; header <- the tree was in header form (V to be zeroed).
SBD_FI int ib_backup(const SearchArgs& a, const IsmBatchArgs& b, int i, ITree& t, INode* nodes, bool& header) {
  const int used = t.used;
  const size_t row = (size_t)i * b.leaves;
  header = t.kind == SEARCH_EVAL || t.kind == SEARCH_TERMINAL;
  if (t.kind == SEARCH_FULL) return 0;
  bool ok = used >= 1 && used <= a.max_nodes;
  if (ok && header) ok = ib_backup_node(a, nodes, used, row, t.leaf, t.kind, t.tval);
  else if (ok && t.kind == SEARCH_BATCH) {
    const int4* slot = ib_slots(b, i);
    #pragma unroll 1
    for (int l = 0; l < b.leaves && ok; l++) {
      const int4 s = slot[l];
      if (s.y == SEARCH_EVAL || s.y == SEARCH_TERMINAL) ok = ib_backup_node(a, nodes, used, row + l, s.x, s.y, s.z);
    }
  } else ok = false;
  if (!ok) { t.kind = SEARCH_FULL; return 0; }
  t.leaf = 0;  // stays a valid index: a plain call on a batch-form tree computes wrong numbers but stays inside the tree
  t.kind = SEARCH_BATCH;
  return used;
}

// PUCT at node j for slot l: ism_select over the world's legal representatives (mover's hand p, legal mask m) with the
// virtual visits of the earlier slots, scored as s_select<true> (n_a = N + V, x = (sgn * W) - (vl * V)).  The candidates are
// j's children (nodes that existed before the call, V in virt), the table entries of earlier slots at j (N = W = 0, V =
// ev[q]) and the ids without either; ties go to the lower id.  vj is V(j).  Returns the action; c <- its child (-1 = none),
// e <- its table entry (-1 = none).
SBD_FI int ib_select(const SearchArgs& a, double vl, const INode* nodes, int lim, const int* virt, const int* ep, const u32* ec,
                     const int* ev, int l, int j, int vj, const Ply& p, const u32* m, int& c_out, int& e_out) {
  const INode& nd = nodes[j];
  const double sgn = s_sign(nd.seat), sq = __dsqrt_rn((double)(nd.N + vj));
  u32 has[SB_MASK_WORDS] = {0, 0, 0, 0, 0};
  int best = -1, best_c = -1, best_e = -1;
  double best_score = 0.0;
  int c = nd.child;
  #pragma unroll 1
  for (int k = 0; k < lim && ism_in(c, lim); k++, c = nodes[c].sibling) {
    const int act = ism_action(p, m, nodes[c].code);
    if (act < 0) continue;
    has[act >> 5] |= 1u << (act & 31);
    const int vc = virt[c], na = nodes[c].N + vc;
    const double x = na ? __dsub_rn(__dmul_rn(sgn, nodes[c].W), __dmul_rn(vl, (double)vc)) : 0.0;
    const double score = s_score(a, na, x, nd.prior[act], sq);
    if (best < 0 || score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_c = c; best_e = -1; }
  }
  #pragma unroll 1
  for (int q = 0; q < l; q++) {
    if (ep[q] != j) continue;
    const int act = ism_action(p, m, ec[q]);
    if (act < 0) continue;
    has[act >> 5] |= 1u << (act & 31);
    const int na = ev[q];
    const double x = __dsub_rn(__dmul_rn(sgn, 0.0), __dmul_rn(vl, (double)na));
    const double score = s_score(a, na, x, nd.prior[act], sq);
    if (best < 0 || score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_c = -1; best_e = q; }
  }
  #pragma unroll 1
  for (int w = 0; w < SB_MASK_WORDS; w++) {
    u32 r = m[w] & ~has[w];
    while (r) {
      const int act = w * 32 + __ffs(r) - 1;
      r &= r - 1;
      if (!ism_rep(p, m, act)) continue;
      const double score = s_score(a, 0, 0.0, nd.prior[act], sq);
      if (best < 0 || score > best_score || (score == best_score && act < best)) { best = act; best_score = score; best_c = -1; best_e = -1; }
    }
  }
  c_out = best_c;
  e_out = best_e;
  return best;
}

__global__ void __launch_bounds__(ISM_BATCH_MAX_CTA) k_ismcts_simulate_batch(const SearchArgs a, const IsmBatchArgs b, const DCard* cards,
                                                                          const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  __shared__ int e_parent[ISM_BATCH_MAX_CTA], e_v[ISM_BATCH_MAX_CTA], e_kind[ISM_BATCH_MAX_CTA], e_node[ISM_BATCH_MAX_CTA];
  __shared__ u32 e_code[ISM_BATCH_MAX_CTA];
  __shared__ int t_start[ISM_BATCH_MAX_CTA], t_cut[ISM_BATCH_MAX_CTA];  // per tree, at its lane 0's index
  stage_cards(s_cards, cards);
  const int x = threadIdx.x, base = x & -b.lanes, l = x - base;
  const int i = (blockIdx.x * blockDim.x + x) / b.lanes;
  const bool tree = i < a.n, live = tree && l < b.leaves;
  const size_t row = (size_t)i * b.leaves + l;
  ITree& t = ism_tree(a, tree ? i : 0);
  INode* nodes = ism_nodes(a, tree ? i : 0);
  int* virt = ib_virt(b, tree ? i : 0);
  bool header = false;
  if (l == 0) {
    int used = tree ? ib_backup(a, b, i, t, nodes, header) : 0;
    if (used >= a.max_nodes) { t.kind = SEARCH_FULL; used = 0; }  // no free node at the start: the tree stops, as 8.8's
    t_start[x] = used;
    t_cut[x] = 0;
    e_kind[x] = header;
  }
  __syncthreads();
  const int start = t_start[base];
  if (start > 0 && e_kind[base]) {
    #pragma unroll 1
    for (int k = l; k < a.max_nodes; k += b.lanes) virt[k] = 0;
  }
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  u32 m[SB_MASK_WORDS];
  if (live) {
    load_state(s, a.roots + row * SB_STATE_BYTES);
    unpack(g, s);
    legal_mask(g, m);
  }
  e_parent[x] = -1;
  e_v[x] = 0;
  int j = 0, d = 0, tval = 0, kind = live && start > 0 ? ISM_WALK : SEARCH_FULL;
  // the wavefront: lane l walks in steps l, l + 1, ...; a step's reads come before the barrier, its writes after it
  #pragma unroll 1
  for (int step = 0; __syncthreads_or(kind == ISM_WALK); step++) {
    int mark = -1, hit = -1;
    bool make = false;
    u32 code = 0;
    if (kind == ISM_WALK && step >= l) {
      if (env_over(g, t.max_steps)) {  // terminal in this world: its game value is backed up
        kind = SEARCH_TERMINAL;
        tval = ism_value(g);
      } else if (d >= a.max_nodes) {
        kind = ISM_FAIL;
      } else {
        int c, e;
        const Ply& p = g.pl[g.local_order];
        const int act = ib_select(a, b.vl, nodes, start, virt, e_parent + base, e_code + base, e_v + base, l, j, d ? virt[j] - 1 : l, p, m, c, e);
        if (act < 0) kind = ISM_FAIL;
        else {
          code = ism_code(p, act);
          s_step(g, s, act);
          legal_mask(g, m);
          if (e >= 0) { kind = SEARCH_COLLISION; hit = e; }
          else if (c >= 0) mark = c;
          else { kind = ISM_NEW; make = true; }
        }
      }
    }
    __syncthreads();
    if (mark >= 0) {  // V(j) then counts this slot too (read back as virt[j] - 1)
      virt[mark] += 1;
      j = mark;
      d++;
    } else if (hit >= 0) {
      e_v[base + hit] += 1;
    } else if (make) {
      e_parent[x] = j;
      e_code[x] = code;
      e_v[x] = 1;
    }
  }
  // every read of V is done: each lane clears its path (the root's V is implicit: slot l counts l earlier slots there)
  if (live && start > 0) {
    int k = j;
    #pragma unroll 1
    for (int q = 0; q < start && k > 0 && k < start; q++) { virt[k] = 0; k = nodes[k].parent; }
  }
  e_kind[x] = kind;
  __syncthreads();
  if (l == 0 && start > 0) {  // new nodes in slot order; the first slot without a free node cuts the call, a failed one stops the tree
    int used = start, cut = b.leaves;
    bool stop = false;
    #pragma unroll 1
    for (int q = 0; q < b.leaves; q++) {
      const int kq = e_kind[base + q];
      if (kq == ISM_FAIL) { stop = true; break; }
      if (kq != ISM_NEW) continue;
      if (used >= a.max_nodes) { cut = q; break; }
      const int p = e_parent[base + q];
      INode& nd = nodes[used];
      nd.parent = p;
      nd.code = e_code[base + q];
      nd.sibling = nodes[p].child;
      nodes[p].child = used;
      e_node[base + q] = used++;
    }
    if (stop) t.kind = SEARCH_FULL;
    else t.used = used;
    t_cut[x] = stop ? 0 : cut;
  }
  __syncthreads();
  if (!live) return;
  int4& slot = ib_slots(b, i)[l];
  if (l >= t_cut[base] || kind == SEARCH_COLLISION) {  // the world's root is emitted and nothing is backed up
    kind = l >= t_cut[base] ? SEARCH_FULL : SEARCH_COLLISION;
    slot = make_int4(0, kind, 0, 0);
    load_state(s, a.roots + row * SB_STATE_BYTES);
    unpack(g, s);
    legal_mask(g, m);
  } else if (kind == SEARCH_TERMINAL) {
    slot = make_int4(j, kind, tval, 0);
  } else {  // ISM_NEW: the node lane 0 took for this slot, written from the world at the leaf
    const int k = e_node[x];
    INode& nd = nodes[k];
    nd.W = 0.0;
    nd.child = -1;
    nd.N = 0;
    nd.seat = g.player_sign == 1 ? 0 : 1;
    const bool over = env_over(g, t.max_steps);
    if (over) ism_zero_prior(nd);
    kind = over ? SEARCH_TERMINAL : SEARCH_EVAL;
    slot = make_int4(k, kind, over ? ism_value(g) : 0, 0);
  }
  ism_emit(a, (int)row, g, s, m, kind);
}

// back up what is pending, mark the tree finished and read out the root's edges (ism_end)
__global__ void __launch_bounds__(TPB_GAME) k_ismcts_end_batch(const SearchArgs a, const IsmBatchArgs b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  ITree& t = ism_tree(a, i);
  bool header;
  ib_backup(a, b, i, t, ism_nodes(a, i), header);
  t.kind = SEARCH_FULL;
  ism_end(a, i);
}
