// Several leaves per tree per call for the perfect-information search, under virtual loss (sb_search_simulate_batch /
// sb_search_end_batch, DESIGN.md 8.11).  One batch call backs up the L leaves the previous call left pending, selects L new
// leaves one after another in each tree (each selection counts the earlier paths of the same call as extra visits carrying
// a loss), then expands and emits all n * L leaves in parallel.  The tree is 8.6's; the new state lives in a tail after
// 8.6's workspace.
//
// Workspace: sb_search_workspace_bytes(n, max_nodes) bytes of 8.6's layout (tree g at ws + g * tree_bytes), then tree g's
// tail at ws + n * tree_bytes + g * tail_bytes, tail_bytes = 16-byte multiple of 8 * L + 4 * max_nodes:
//   slot  int2[L]           pending slot l: {node index, slot kind}
//   virt  i32[max_nodes]    virtual visits V of this call, zero between calls
// Slot l of tree g is row g * L + l of every input and leaf output.  A tree is in header form (STree.kind 0, 1 or 2, one
// pending leaf) after begin, advance or a plain simulate, and in batch form (kind SEARCH_BATCH, the L slots pending) after a
// batch call.  A batch call on a header-form tree backs up its single leaf from slot 0's row and zeroes V.
//
// Two launches per call:
//   k_search_batch_select  one thread per tree, SB_SELECT_THREADS per CTA: backup, then the L selections.  A walk that
//                          needs a new edge takes the next free node at once (parent, action, N = 0, W = 0 and the parent's
//                          child link), so later slots see it as pending: a walk that reaches a pending node stops there
//                          (COLLISION), one that needs a node when none is left makes this and every later slot FULL.
//   k_search_batch_expand  one thread per slot, TPB_GAME per CTA: a new node becomes the record sb_step(parent, action)
//                          (s_write_node), every slot emits 8.6's leaf outputs at its row.
// sb_search_end_batch is one launch (k_search_end_batch): backup, kind SEARCH_FULL, 8.6's read-out.  No handle scratch, no
// atomics, no host synchronisation: the expansion writes only its own new node and reads records of nodes that existed
// before the call (a walk never continues below a pending node).
//
// Fault safety: 8.6's rule (sb_search.cuh), with the same checks (sb_count, sb_backup_node, s_select, s_read_out); in
// addition a pending slot's node must lie below the node count and a new node's action below 156.  A failed check stops the
// tree: kind SEARCH_FULL, every slot FULL, the root emitted (a stopped tree's V is never read again, the next header-form
// call zeroes it).
#pragma once
#include "sb_search.cuh"

#define SEARCH_BATCH 3        // STree.kind of a batch-form tree: the tail's L slots are pending
#define SEARCH_COLLISION 3    // slot kind: the walk reached a node allocated earlier in the same call
#define SEARCH_MAX_LEAVES 256
#define SB_SELECT_THREADS 32  // trees per CTA of the selection pass: more CTAs on the chip for a few thousand trees

struct BatchArgs {
  int leaves;
  double vl;                // virtual loss per virtual visit
  unsigned char* tail;      // ws + n * tree_bytes
  size_t tail_bytes;
};

SBD_FI int2* sb_slots(const BatchArgs& b, int i) { return reinterpret_cast<int2*>(b.tail + (size_t)i * b.tail_bytes); }
SBD_FI int* sb_virt(const BatchArgs& b, int i) { return reinterpret_cast<int*>(b.tail + (size_t)i * b.tail_bytes + 8 * (size_t)b.leaves); }
// set (d = 0) or add d to (d = 1) V of node j and every node above it; false on a bad parent link
SBD_FI bool sb_mark_path(const SNode* nodes, int* virt, int j, int d) {
  #pragma unroll 1
  while (true) {
    virt[j] = d ? virt[j] + 1 : 0;
    if (j == 0) return true;
    const int p = nodes[j].parent;
    if (p < 0 || p >= j) return false;
    j = p;
  }
}

// what the previous call left pending in tree i: the header-form leaf (slot 0's row) or the L slots in ascending order.
// Returns the node count, 0 when the tree is (or now is) stopped.  A header-form tree becomes batch form with V zero.
SBD_FI int sb_backup(const SearchArgs& a, const BatchArgs& b, int i, STree& t, SNode* nodes) {
  const int used = sb_count(t, a.max_nodes);
  const size_t row = (size_t)i * b.leaves;
  bool ok = used > 0;
  if (t.kind == SEARCH_FULL) return 0;
  if (ok && (t.kind == SEARCH_EVAL || t.kind == SEARCH_TERMINAL)) {
    ok = sb_backup_node(a, nodes, used, row, t.leaf, t.kind);
    int* virt = sb_virt(b, i);
    #pragma unroll 1
    for (int k = 0; k < a.max_nodes; k++) virt[k] = 0;
  } else if (ok && t.kind == SEARCH_BATCH) {
    const int2* slot = sb_slots(b, i);
    #pragma unroll 1
    for (int l = 0; l < b.leaves && ok; l++) {
      const int2 s = slot[l];
      if (s.y == SEARCH_EVAL || s.y == SEARCH_TERMINAL) ok = sb_backup_node(a, nodes, used, row + l, s.x, s.y);
    }
  } else ok = false;
  if (!ok) { t.kind = SEARCH_FULL; return 0; }
  t.leaf = 0;  // stays a valid index: a plain call on a batch-form tree computes wrong numbers but stays inside the tree
  t.kind = SEARCH_BATCH;
  return used;
}

__global__ void __launch_bounds__(SB_SELECT_THREADS) k_search_batch_select(const SearchArgs a, const BatchArgs b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  int2* slot = sb_slots(b, i);
  int* virt = sb_virt(b, i);
  int used = sb_backup(a, b, i, t, nodes);
  if (used >= a.max_nodes) { t.kind = SEARCH_FULL; used = 0; }  // no free node at the start: the tree stops, as 8.6's
  const int start = used;
  int l = 0;
  bool ok = used > 0;
  #pragma unroll 1
  for (; l < b.leaves && ok; l++) {
    int j = 0, kind = -1;
    #pragma unroll 1
    for (int d = 0; kind < 0; d++) {
      if (j >= start) kind = SEARCH_COLLISION;
      else if (nodes[j].terminal) kind = SEARCH_TERMINAL;
      else {
        int c;
        const int act = d < a.max_nodes ? s_select<true>(a, nodes, virt, b.vl, j, used, c) : -1;
        if (act < 0) { ok = false; break; }
        if (!c) {
          if (used >= a.max_nodes) break;  // no free node: this and every later slot are FULL
          const int k = used++;
          nodes[k].parent = j;
          nodes[k].action = (u8)act;
          nodes[k].N = 0;
          nodes[k].W = 0.0;
          nodes[j].child[act] = k;
          j = k;
          kind = SEARCH_EVAL;  // the expansion pass makes it TERMINAL when the new record is over
        } else j = c;
      }
    }
    if (kind < 0) break;
    slot[l] = make_int2(j, kind);
    if (!sb_mark_path(nodes, virt, j, 1)) { ok = false; break; }
  }
  if (!ok) t.kind = SEARCH_FULL;  // a bad index or no legal action: the tree stops
  else {
    t.used = used;
    #pragma unroll 1
    for (int x = 0; x < l; x++) sb_mark_path(nodes, virt, slot[x].x, 0);
  }
  #pragma unroll 1
  for (int x = ok ? l : 0; x < b.leaves; x++) slot[x] = make_int2(0, SEARCH_FULL);
}

__global__ void __launch_bounds__(TPB_GAME) k_search_batch_expand(const SearchArgs a, const BatchArgs b, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  stage_cards(s_cards, cards);
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.n * b.leaves) return;
  const int i = r / b.leaves, l = r - i * b.leaves;
  G g;
  init_g(g, s_cards, wt);
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  int2& slot = sb_slots(b, i)[l];
  const int used = sb_count(t, a.max_nodes), k = slot.x, kind = slot.y;
  if (kind == SEARCH_EVAL && k > 0 && k < used && nodes[k].parent >= 0 && nodes[k].parent < k && nodes[k].action < SB_N_ACTIONS) {
    slot.y = s_expand(a, r, g, t, nodes, k, nodes[k].parent, nodes[k].action);
  } else if (kind == SEARCH_TERMINAL && k >= 0 && k < used) {
    s_emit_node(a, r, g, nodes[k], SEARCH_TERMINAL);
  } else if (kind == SEARCH_COLLISION || kind == SEARCH_FULL) {
    s_emit_node(a, r, g, nodes[0], kind);
  } else {  // a bad slot: the tree stops (every thread of the tree that gets here writes the same value)
    t.kind = SEARCH_FULL;
    slot = make_int2(0, SEARCH_FULL);
    s_emit_node(a, r, g, nodes[0], SEARCH_FULL);
  }
}

// back up what is pending, mark the tree finished and read out the root's edges
__global__ void __launch_bounds__(TPB_GAME) k_search_end_batch(const SearchArgs a, const BatchArgs b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  STree& t = s_tree(a, i);
  SNode* nodes = s_nodes(a, i);
  sb_backup(a, b, i, t, nodes);
  t.kind = SEARCH_FULL;
  s_read_out(a, i, nodes, sb_count(t, a.max_nodes));
}
