// Determinization of packed records for information-set sampling (sb_determinize): rewrite each record so that everything
// the observer sees stays byte-identical and everything hidden from the observer is resampled.  Hidden from observer o are
// (a) which of the other seat r = 1 - o's cards sit in r's hand and which in r's deck at which slot, and (b) the Philox key,
// which fixes every future draw and random target.  The kernel shuffles r's (card, cost, flags) triples over r's movable
// slots and sets the key; r's card multiset, n_hand, n_deck and the deck's weight profile (deck_wn stays with its slot) are
// kept.  Movable slots: hand 0..n_hand-1, then deck 0..n_deck-1 (clamped to 4 / 16), skipping records flagged SB_CF_OBJ,
// which ext[91..107] addresses by (order, in_deck, index).  Fisher-Yates from the end over that list, j = umulhi(w0, i + 1)
// with w0 of philox(counter=(t, 0, 0xDE7E, 0), key) for the t-th swap: the call shape of the engine's shuffle / rng_below
// on a stream of its own (the game's stream is (draw, turn, 0, 0), the random agent's 0xA6E7, the deck schedule's 0xDEC4,
// the ES operators' 0xE5..0xE7).  Included by sb_kernels.cu.
//
// One warp per record, straight on the packed bytes (no unpack): one 128-bit load per lane into a 512-byte shared image,
// lane s < 20 owns slot s (hand 0..3, deck 4..19), lane t computes the t-th Philox block, every lane follows its own
// triple through the swaps (a swap is a transposition of positions, so each element's final position needs only the
// swap list), the triples are written to their final slots in the image, and one 128-bit store per lane writes it out.
#pragma once
#include "sb_engine.cuh"

#define DET_TAG 0xDE7Eu
#define DET_WARPS 4  // records per CTA

// byte offset of the card of slot s (0..3 hand, 4..19 deck) within SbPlayer; cost and flags follow at +stride, +2 stride
SBD_FI int det_card_off(int s) { return s < SB_HAND_MAX ? 12 + s : 24 + (s - SB_HAND_MAX); }
SBD_FI int det_stride(int s) { return s < SB_HAND_MAX ? SB_HAND_MAX : SB_DECK_MAX; }

__global__ void __launch_bounds__(DET_WARPS * 32) k_determinize(int n, const u8* states, const u8* observer,
                                                               const unsigned long long* keys, u8* out) {
  __shared__ int4 s_img[DET_WARPS][SB_STATE_BYTES / 16];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * DET_WARPS + w;
  if (i >= n) return;  // warp-uniform
  s_img[w][lane] = reinterpret_cast<const int4*>(states + i * SB_STATE_BYTES)[lane];
  __syncwarp();
  u8* b = reinterpret_cast<u8*>(s_img[w]);
  const int o = observer ? (observer[i] != 0) : (b[14] != 0);  // local_order
  const int p = 32 + (1 - o) * (int)sizeof(SbPlayer);          // pl[r]
  const int nh = min((int)b[p + 8], SB_HAND_MAX), nd = min((int)b[p + 9], SB_DECK_MAX);
  const int s = lane, off = p + det_card_off(s < 20 ? s : 0), st = det_stride(s);
  const bool valid = s < SB_HAND_MAX ? s < nh : s < 20 && s - SB_HAND_MAX < nd;
  u8 card = 0, cost = 0, flags = 0;
  if (valid) { card = b[off]; cost = b[off + st]; flags = b[off + 2 * st]; }
  const bool movable = valid && !(flags & SB_CF_OBJ);
  const unsigned bal = __ballot_sync(0xFFFFFFFFu, movable);
  const int m = __popc(bal);
  const unsigned long long k = keys[i];
  const u32 k_lo = (u32)k, k_hi = (u32)(k >> 32);
  u32 jt = 0;  // swap t exchanges positions m-1-t and jt
  if (lane < m - 1) {
    u32 w0, w1;
    philox((u32)lane, 0u, DET_TAG, 0u, k_lo, k_hi, w0, w1);
    jt = __umulhi(w0, (u32)(m - lane));
  }
  int pos = __popc(bal & ((1u << lane) - 1u));  // this lane's triple starts at position pos of the movable list
  #pragma unroll 1
  for (int t = 0; t < m - 1; t++) {
    const int a = m - 1 - t, j = (int)__shfl_sync(0xFFFFFFFFu, jt, t);
    pos = pos == a ? j : pos == j ? a : pos;
  }
  __syncwarp();  // every lane has read its triple before any is overwritten
  if (movable) {
    unsigned rest = bal;
    #pragma unroll 1
    for (int q = 0; q < pos; q++) rest &= rest - 1;
    const int d = __ffs(rest) - 1, doff = p + det_card_off(d), dst = det_stride(d);
    b[doff] = card; b[doff + dst] = cost; b[doff + 2 * dst] = flags;
  }
  if (lane == 0) {
    reinterpret_cast<u32*>(b)[0] = k_lo;
    reinterpret_cast<u32*>(b)[1] = k_hi;
  }
  __syncwarp();
  reinterpret_cast<int4*>(out + i * SB_STATE_BYTES)[lane] = s_img[w][lane];
}
