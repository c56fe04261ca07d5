// Tree reuse between moves for both PUCT searches (sb_search_advance / sb_ismcts_advance, DESIGN.md 8.10): an advance is
// the matching begin, except that it may carry the subtree of the new root over from a finished search.  It reads the
// finished workspace (ws_src, consumed) and writes the next one (ws_dst, a.ws), which then holds, for each tree, either
// exactly what the begin would write (kept 0) or the first `keep` nodes of the matched node's subtree in creation order
// (increasing node index), the matched node becoming node 0.  A tree is reused only when its source header says finished
// (kind SEARCH_FULL: ended or stopped full, nothing pending) with this call's max_steps, and its rule finds a node j:
//   8.6 (k_search_advance): the lowest-index node whose 512-byte record equals this call's root byte for byte;
//   8.8 (k_ismcts_advance): the child of the source root with the move code the source header stores for the root action
//        id played (played[g] in 0..155, that code not ISM_NONE), when world 0 of the new root is not over and its seat to
//        move is the child's and the source root's (the tree is over one player's information set: a PASS, or any move
//        that hands the turn over, starts fresh).
//
// One CTA of RS_THREADS threads covers TPB_GAME trees in three phases.  (8.8 only: each of the first TPB_GAME threads unpacks
// its tree's world and notes its seat to move, -1 when it is over.)  Each of the 8 warps then carries over 8 of the CTA's
// trees, one at a time: its 32 lanes compare a 16-byte prefix (Philox key, turn, draw, steps) of 32 nodes' records at once
// and the whole 512-byte record only on a candidate, with a ballot; then one ascending pass over the source nodes from j
// maps each parent through the index map, keeps the node while fewer than `keep` are kept and its parent is kept, copies it
// as 16-byte chunks with its child links cleared and its parent remapped, links it into its new parent and writes its new
// index (-1 if dropped) into the source node's parent field, which is the map its children read.  Last, each of the first
// TPB_GAME threads writes its tree's header and emits the root with the begin's code (s_start / ism_start), which also
// writes node 0 when nothing was kept.
//
// Fault safety: the source header's node count is clamped to 0..max_nodes and bounds every index read from ws_src: the
// prefix scan and the pass stop at it, a parent is used only when it lies in [j, k), a map entry only when it lies in
// [0, kept so far), 8.8's sibling walk (ism_find) is bounded by it, and 8.6 links a child only at an action id below 156.
// Every write lands in node 0 .. keep-1 of tree g of ws_dst, in the parent field of a source node below the count, or in
// the source header's node count, which the pass sets to 0 (rs_consume): a consumed workspace reads as empty.
#pragma once
#include "sb_gumbel.cuh"

// threads per CTA: 8 warps carry over the CTA's TPB_GAME trees (the pass is bound by the latency of its dependent loads, so
// more warps per tree hide more of it); the first TPB_GAME threads then write and emit one tree each
#define RS_THREADS 256

struct ReuseArgs {
  unsigned char* src;  // the finished search's workspace, same n, max_nodes and layout as a.ws; consumed
  int keep;            // nodes kept at most, 1..max_nodes
  int* kept;           // i32[n] nodes kept (0: a fresh root), nullable
  const int* played;   // i32[n] root action id played since the source search (sb_ismcts_advance)
};

SBD_FI int4 rs_shfl(int4 v, int src) {
  return make_int4(__shfl_sync(0xFFFFFFFFu, v.x, src), __shfl_sync(0xFFFFFFFFu, v.y, src), __shfl_sync(0xFFFFFFFFu, v.z, src),
                   __shfl_sync(0xFFFFFFFFu, v.w, src));
}
SBD_FI bool rs_eq(int4 a, int4 b) { return a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w; }

// the warp's pass over source nodes j .. lim-1 (see the header comment); fix(c, v, mp) adjusts chunk c of a kept node whose
// new parent is mp, link(k, mk, mp) runs on lane 0 after the copy.  Returns the number of nodes kept (>= 1).
template <class Node, class Fix, class Link>
SBD_FI int rs_pass(Node* src, Node* dst, int j, int lim, int keep, int lane, Fix fix, Link link) {
  int cnt = 0;
  #pragma unroll 1
  for (int k = j; k < lim && cnt < keep; k++) {
    int mp = -1;
    bool kept = k == j;
    if (!kept) {
      const int p = src[k].parent;
      if (p >= j && p < k) {
        mp = src[p].parent;  // the map entry lane 0 wrote for p
        kept = mp >= 0 && mp < cnt;
      }
    }
    const int mk = kept ? cnt : -1;
    if (kept) {
      const int4* s4 = reinterpret_cast<const int4*>(&src[k]);
      int4* d4 = reinterpret_cast<int4*>(&dst[mk]);
      #pragma unroll 1
      for (int c = lane; c < (int)(sizeof(Node) / 16); c += 32) d4[c] = fix(c, s4[c], mp);
      cnt++;
    }
    __syncwarp();
    if (lane == 0) {
      if (kept && mp >= 0) link(k, mk, mp);
      src[k].parent = mk;
    }
    __syncwarp();
  }
  return cnt;
}

// source tree i after its pass: its node count (the first int of both tree headers) becomes 0, so a second advance from
// the same workspace (a replayed graph capture) starts every tree fresh instead of reading the index map as a tree, and a
// simulate or end on it dereferences no node (warp-wide; i may be past n)
SBD_FI void rs_consume(const SearchArgs& a, const ReuseArgs& r, int i, int lane) {
  __syncwarp();
  if (lane == 0 && i < a.n) *reinterpret_cast<int*>(r.src + (size_t)i * a.tree_bytes) = 0;
}

// the first of source tree i's nodes whose record equals this call's root (-1 if none), warp-wide
SBD_FI int s_match(const SearchArgs& a, const SNode* src, int lim, int i, int lane) {
  const int4 want = reinterpret_cast<const int4*>(a.roots + (size_t)i * SB_STATE_BYTES)[lane];
  const int4 head = rs_shfl(want, 0);
  #pragma unroll 1
  for (int b = 0; b < lim; b += 32) {
    const int k = b + lane;
    u32 cand = __ballot_sync(0xFFFFFFFFu, k < lim && rs_eq(reinterpret_cast<const int4*>(&src[k].rec)[0], head));
    while (cand) {
      const int c = b + __ffs(cand) - 1;
      cand &= cand - 1;
      if (__all_sync(0xFFFFFFFFu, rs_eq(reinterpret_cast<const int4*>(&src[c].rec)[lane], want))) return c;
    }
  }
  return -1;
}

#define RS_S_CHILD0 ((int)(offsetof(SNode, child) / 16))
#define RS_S_CHILD1 ((int)(offsetof(SNode, prior) / 16))
#define RS_S_PARENT ((int)(offsetof(SNode, parent) / 16))
static_assert(offsetof(STree, used) == 0 && offsetof(ITree, used) == 0, "rs_consume: the node count opens both tree headers");
static_assert(offsetof(SNode, child) % 16 == 0 && offsetof(SNode, prior) % 16 == 0 && offsetof(SNode, parent) % 16 == 4,
              "sb_search_advance's chunk copy: child links fill whole chunks, parent is .y of its chunk");

// 8.6: carry tree i over into a.ws; returns the nodes kept, 0 for a fresh root (warp-uniform)
SBD_FI int s_carry(const SearchArgs& a, const ReuseArgs& r, int i, int lane) {
  const STree& ts = *reinterpret_cast<const STree*>(r.src + (size_t)i * a.tree_bytes);
  SNode* src = reinterpret_cast<SNode*>(r.src + (size_t)i * a.tree_bytes + sizeof(STree));
  const int u = ts.used, lim = u < 0 ? 0 : u > a.max_nodes ? a.max_nodes : u;
  if (ts.kind != SEARCH_FULL || ts.max_steps != a.max_steps || lim < 1) return 0;
  const int j = s_match(a, src, lim, i, lane);
  if (j < 0) return 0;
  SNode* dst = s_nodes(a, i);
  return rs_pass(src, dst, j, lim, r.keep, lane,
                 [](int c, int4 v, int mp) {
                   if (c >= RS_S_CHILD0 && c < RS_S_CHILD1) v = make_int4(0, 0, 0, 0);
                   if (c == RS_S_PARENT) v.y = mp;
                   return v;
                 },
                 [&](int k, int mk, int mp) {
                   const int act = src[k].action;
                   if (act < SB_N_ACTIONS) dst[mp].child[act] = mk;
                 });
}

__global__ void __launch_bounds__(RS_THREADS) k_search_advance(const SearchArgs a, const ReuseArgs r, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  __shared__ int s_kept[TPB_GAME];
  stage_cards(s_cards, cards);
  const int lane = threadIdx.x & 31, base = blockIdx.x * TPB_GAME;
  #pragma unroll 1
  for (int t = threadIdx.x >> 5; t < TPB_GAME; t += RS_THREADS / 32) {
    const int kept = base + t < a.n ? s_carry(a, r, base + t, lane) : 0;
    rs_consume(a, r, base + t, lane);
    if (lane == 0) s_kept[t] = kept;
  }
  __syncthreads();
  const int i = base + threadIdx.x;
  if (threadIdx.x >= TPB_GAME || i >= a.n) return;
  const int kept = s_kept[threadIdx.x];
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
  unpack(g, s);
  s_start(a, i, g, s, kept);
  if (r.kept) r.kept[i] = kept;
}

static_assert(offsetof(INode, parent) == 8 && offsetof(INode, child) == 12 && offsetof(INode, sibling) == 16 &&
              offsetof(INode, code) == 20, "sb_ismcts_advance's chunk copy: parent / child are .z / .w of chunk 0, "
              "sibling / code .x / .y of chunk 1");

// 8.8: carry tree i over into a.ws when world 0 of its new root has `seat` to move (-1: the world is over); returns the
// nodes kept, 0 for a fresh root (warp-uniform)
SBD_FI int ism_carry(const SearchArgs& a, const ReuseArgs& r, int i, int lane, int seat) {
  const ITree& ts = *reinterpret_cast<const ITree*>(r.src + (size_t)i * a.tree_bytes);
  INode* src = reinterpret_cast<INode*>(r.src + (size_t)i * a.tree_bytes + sizeof(ITree));
  const int lim = ism_lim(ts, a.max_nodes), played = r.played[i];
  if (seat < 0 || ts.kind != SEARCH_FULL || ts.max_steps != a.max_steps || lim < 1 || played < 0 || played >= SB_N_ACTIONS) return 0;
  const u32 code = ts.root_code[played];
  const int j = code == ISM_NONE ? -1 : ism_find(src, lim, src[0], code);
  if (j < 0 || src[j].seat != seat || src[0].seat != seat) return 0;  // the same observer: no PASS, no turn over
  INode* dst = ism_nodes(a, i);
  return rs_pass(src, dst, j, lim, r.keep, lane,
                 [](int c, int4 v, int mp) {
                   if (c == 0) { v.z = mp; v.w = -1; }  // parent, no child yet
                   if (c == 1) { v.x = -1; if (mp < 0) v.y = (int)ISM_NONE; }  // no sibling yet; the root has no code
                   return v;
                 },
                 [&](int, int mk, int mp) {  // prepend: ascending creation order keeps the source's newest-first sibling order
                   dst[mk].sibling = dst[mp].child;
                   dst[mp].child = mk;
                 });
}

__global__ void __launch_bounds__(RS_THREADS) k_ismcts_advance(const SearchArgs a, const ReuseArgs r, const DCard* cards, const double* wt) {
  __shared__ DCard s_cards[SBC_COUNT];
  __shared__ int s_seat[TPB_GAME], s_kept[TPB_GAME];
  stage_cards(s_cards, cards);
  const int lane = threadIdx.x & 31, base = blockIdx.x * TPB_GAME, i = base + threadIdx.x;
  const bool mine = threadIdx.x < TPB_GAME && i < a.n;  // this thread writes and emits tree i
  G g;
  init_g(g, s_cards, wt);
  __align__(16) SbState s;
  if (mine) {
    load_state(s, a.roots + (size_t)i * SB_STATE_BYTES);
    unpack(g, s);
    s_seat[threadIdx.x] = env_over(g, a.max_steps) ? -1 : g.player_sign == 1 ? 0 : 1;
  }
  __syncthreads();
  #pragma unroll 1
  for (int t = threadIdx.x >> 5; t < TPB_GAME; t += RS_THREADS / 32) {
    const int kept = base + t < a.n ? ism_carry(a, r, base + t, lane, s_seat[t]) : 0;
    rs_consume(a, r, base + t, lane);
    if (lane == 0) s_kept[t] = kept;
  }
  __syncthreads();
  if (!mine) return;
  const int kept = s_kept[threadIdx.x];
  u32 m[SB_MASK_WORDS];
  ism_start(a, i, g, s, m, kept);
  if (r.kept) r.kept[i] = kept;
}
