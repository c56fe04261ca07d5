// sbw_effects.cuh -- the card effects of the warp-per-game engine (reference cards/<id>.py activate_ability).
//
// Most cards are one row of a compact OPCODE table (w_effect_ops): query -> selection -> verb, interpreted by
// w_run_op() with uniform control flow; the irregular ones (temples, hand / deck surgery, pushes) are bespoke handlers
// behind the same dispatcher.  p[] = the card's ability_* attributes exported by tools/gen_card_table.py.
#pragma once
#include "sbw_core.cuh"

#define WCUR(wg) ((wg)->current_order)

SBW_FI int w_need(WG* wg, int pt) {  // board.at(pt) dereferenced without a None check -> AttributeError (Q11)
  int id = w_at_pt(wg, pt);
  if (id < 0) WERR(wg, SB_ERR_NONE_TARGET);
  return id;
}
SBW_FI int w_choice_tl(WG* wg, TL t) {
  const int n = tl_n(t);
  if (n <= 0) { WERR(wg, SB_ERR_EMPTY_CHOICE); return PT_NONE; }
  return tl_nth(t, w_rng_below(wg, n));
}
SBW_FI int w_choice_pl(WG* wg, PL p) {
  if (p.n <= 0) { WERR(wg, SB_ERR_EMPTY_CHOICE); return PT_NONE; }
  return pl_get(p, w_rng_below(wg, p.n));
}
// a tile list into the scratch array, in list order
SBW_FI int w_expand(WG* wg, TL t) {
  int n = 0;
#pragma unroll 1
  for (;;) { const int pt = tl_pop(t); if (pt == PT_NONE) break; wg->scr[n++] = (i8)pt; }
  return n;
}
template <class F> SBW_FI u32 w_or_tiles(const WG* wg, u32 tiles, F f) {  // OR of f(slot) over the on-board entities standing on `tiles`
  u32 m = 0;
  const int ne = wg->n_ent;
#pragma unroll 1
  for (int base = 0; base < ne; base += 32)
    m |= w_or([&](int l) -> u32 { const int s = base + l; return (s < ne && (wg->e_fl[s] & WEF_ONB) && ((tiles >> wg->e_pos[s]) & 1u)) ? (u32)f(s) : 0u; });
  return m;
}
template <class F> SBW_FI int w_min_tiles(const WG* wg, u32 tiles, F f) {
  int r = 0x7FFFFFFF;
  const int ne = wg->n_ent;
#pragma unroll 1
  for (int base = 0; base < ne; base += 32) {
    const int v = w_min([&](int l) -> int { const int s = base + l; return (s < ne && (wg->e_fl[s] & WEF_ONB) && ((tiles >> wg->e_pos[s]) & 1u)) ? (int)f(s) : 0x7FFFFFFF; });
    r = v < r ? v : r;
  }
  return r;
}
// list.sort(key=lambda t: (k1(t), random.random()), reverse=desc): one random() per element in list order, then a stable
// sort (cards/b002.py:20, b008.py:24, b009.py:20, b104.py:19, s101.py:21).  Only the first one or two elements are ever
// used: selection instead of a sort.  k1 = Point.y (by_strength = false) or the entity's strength.
SBW_NI PL w_keyed_take(WG* wg, TL t, bool by_strength, bool desc, int take) {
  W_SHARED(wg);
  PL out; out.v = 0; out.n = 0;
  const int n = w_expand(wg, t);  // at most 20 points: no keyed query includes a base
#pragma unroll 1
  for (int i = 0; i < n && i < DECK_W; i++) wg->scr_d[i] = w_rng_random(wg);
  u32 taken = 0;
#pragma unroll 1
  for (int s = 0; s < take && s < n; s++) {
    int best = -1, bk = 0;
    double br = 0.0;
#pragma unroll 1
    for (int i = 0; i < n; i++) {
      if ((taken >> i) & 1u) continue;
      const int pt = wg->scr[i];
      const int k = by_strength ? (int)wg->e_str[wg->board[pt]] : wpt_y(pt);
      const double r = wg->scr_d[i];
      const bool before = best < 0 || (desc ? (k > bk || (k == bk && r > br)) : (k < bk || (k == bk && r < br)));
      if (before) { best = i; bk = k; br = r; }
    }
    taken |= 1u << best;
    pl_push(out, wg->scr[best]);
  }
  return out;
}
SBW_NI int w_count_types_friendly(WG* wg) {  // cards/up02.py:13-19, up03.py:14-20
  W_SHARED(wg);
  const TL t = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_FRIENDLY), PT_NONE);
  const DCard* cards = wg->cards;
  W_SHARED(cards);
  return w_popc(w_or_tiles(wg, t.m, [&](int s) -> u32 { return cards[wg->e_card[s]].types; }));
}

// ---- Temple of Time memories (cards/b005.py:13,24-33): a forest of deep copies, see WMem / Mem in sb_engine.cuh
SBW_NI int w_mem_push_entity(WG* wg, int temple, int parent, int pos, int src) {
  W_SHARED(wg);
  if (wg->n_mem >= NMEM) { WERR(wg, SB_ERR_OVERFLOW); return -1; }
  const int me = wg->n_mem;
  WMem m;
  m.b005 = (i8)temple; m.parent = (i8)parent; m.pos = (u8)pos; m.card = wg->e_card[src];
  m.fl = wg->e_fl[src] & (WEF_OWNER | WEF_STRUCT | WEF_FIXED);
  m.strength = wg->e_str[src];
#pragma unroll
  for (int k = 0; k < 5; k++) m.st[k] = (u8)w_st(wg, src, k);
#pragma unroll
  for (int k = 0; k < 4; k++) m.pad[k] = 0;
  wg->mem[me] = m;
  wg->n_mem = (u8)(me + 1);
  return me;
}
// deep copy of the subtree rooted at mem[src] under new_parent (iterative: parents precede children in the array)
SBW_NI int w_mem_copy_subtree(WG* wg, int src, int new_parent, int limit) {
  W_SHARED(wg);
  i8* map = wg->scr;
#pragma unroll 1
  for (int q = 0; q < NMEM; q++) map[q] = -1;
  int root = -1;
#pragma unroll 1
  for (int q = src; q < limit; q++) {
    const int par = wg->mem[q].parent;
    const bool is_root = (q == src);
    if (!is_root && (par < 0 || map[par] < 0)) continue;
    if (wg->n_mem >= NMEM) { WERR(wg, SB_ERR_OVERFLOW); return -1; }
    const int me = wg->n_mem;
    wg->n_mem = (u8)(me + 1);
    WMem m = wg->mem[q];
    m.b005 = -1;
    m.fl |= WEF_SINGLE;  // detached: deep-copied below another temple's copy (lives on a cloned board once restored)
    m.parent = (i8)(is_root ? new_parent : map[par]);
    wg->mem[me] = m;
    map[q] = (i8)me;
    if (is_root) root = me;
  }
  return root;
}
SBW_NI void w_mem_delete_temple(WG* wg, int temple) {  // self.ability_remembered = []
  W_SHARED(wg);
  i8* keep = wg->scr;
  i8* nidx = wg->scr + 12;
  int w = 0;
  const int nm = wg->n_mem;
#pragma unroll 1
  for (int i = 0; i < nm; i++) {
    const WMem& m = wg->mem[i];
    const bool k = m.parent < 0 ? (m.b005 != temple) : (keep[m.parent] != 0);
    keep[i] = k; nidx[i] = k ? (i8)w++ : (i8)-1;
  }
#pragma unroll 1
  for (int i = 0; i < nm; i++) if (keep[i]) {
    WMem m = wg->mem[i];
    if (m.parent >= 0) m.parent = nidx[m.parent];
    wg->mem[nidx[i]] = m;
  }
  wg->n_mem = (u8)w;
}

// ---------------------------------------------------------------- the opcode table
// One 32-bit word per regular card:
//   bits  0-3  region   WR_*      where the targets come from
//   bits  4-5  kind     TK_*
//   bits  6-7  side     TS_*
//   bits  8-11 select   WS_*      which of them are taken, in which order
//   bits 12-16 verb     WV_*      what happens to each taken target
//   bits 17-19 amount   WA_*      where the verb's amount comes from
//   bits 20-22 filter   WF_*      extra Target filter
//   bit  23    pov = the entity's owner (else board.current_player)
//   bit  24    exclude the entity's own tile
//   bit  25    include bases
//   bits 26-28 after    WX_*      what the entity does to itself afterwards
//   bits 29-31 cond     WC_*      precondition
enum { WR_ALL = 1, WR_SURROUND, WR_BORDER, WR_AHEAD, WR_BEHIND, WR_SELF, WR_NONE };
enum { WS_ALL = 0, WS_CHOICE, WS_FIRST, WS_SHUFFLE_P0, WS_SHUFFLE_P1, WS_FRONTMOST1, WS_FRONTMOST_P0_SHUFFLED };
enum { WV_NONE = 0, WV_DAMAGE_PT, WV_HEAL, WV_HEAL_VITALIZE, WV_VITALIZE, WV_POISON, WV_FREEZE, WV_CONFUSE, WV_DESTROY, WV_PUSH,
       WV_COMMAND, WV_DECONFUSE_COMMAND, WV_FORCE_ATTACK, WV_DAMAGE_POISON_GUARDED, WV_DAMAGE_HEAL_SELF, WV_DAMAGE_RANDINT };
enum { WA_P0 = 0, WA_P1, WA_ONE, WA_DMG };
enum { WF_NONE = 0, WF_CONSTRUCT, WF_DRAGON, WF_X_DRAGON, WF_X_CONFUSED, WF_FROZEN, WF_POISONED, WF_LIMIT_SELF };
enum { WX_NONE = 0, WX_HEAL_P0, WX_VITALIZE, WX_DESTROY, WX_GAIN_SPEED_2 };
enum { WC_NONE = 0, WC_ATTACKING_UNIT, WC_ATTACKING_FROZEN_UNIT, WC_REPEAT_P0, WC_REPEAT_DMG };
#define WOP(region, kind, side, select, verb, amount, filter, povme, exself, base, after, cond) \
  ((u32)(region) | ((u32)(kind) << 4) | ((u32)(side) << 6) | ((u32)(select) << 8) | ((u32)(verb) << 12) | ((u32)(amount) << 17) | \
   ((u32)(filter) << 20) | ((u32)(povme) << 23) | ((u32)(exself) << 24) | ((u32)(base) << 25) | ((u32)(after) << 26) | ((u32)(cond) << 29))

// returns 0 when the card has no table row (bespoke handler or no ability)
SBW_FI u32 w_effect_op(int card) {
  switch (card) {
    //                            region       kind          side         select           verb                   amount filter        me xs bs after          cond
    case SBC_B002: return WOP(WR_ALL,      TK_ANY,  TS_ENEMY,    WS_FRONTMOST1,   WV_DAMAGE_PT,          WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/b002.py:13-21
    case SBC_B004: return WOP(WR_ALL,      TK_ANY,  TS_ENEMY,    WS_ALL,          WV_DAMAGE_PT,          WA_P0, WF_NONE,      0, 0, 1, WX_DESTROY,    WC_NONE);  // cards/b004.py:13-22
    case SBC_B009: return WOP(WR_ALL,      TK_UNIT, TS_ENEMY,    WS_FRONTMOST_P0_SHUFFLED, WV_CONFUSE,   WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/b009.py:13-24
    case SBC_B104: return WOP(WR_ALL,      TK_UNIT, TS_ENEMY,    WS_FRONTMOST1,   WV_FREEZE,             WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/b104.py:12-20
    case SBC_B203: return WOP(WR_AHEAD,    TK_UNIT, TS_FRIENDLY, WS_ALL,          WV_DECONFUSE_COMMAND,  WA_P0, WF_NONE,      1, 0, 0, WX_NONE,       WC_NONE);  // cards/b203.py:12-21
    case SBC_U007: return WOP(WR_SURROUND, TK_UNIT, TS_ENEMY,    WS_CHOICE,       WV_HEAL_VITALIZE,      WA_P0, WF_NONE,      1, 0, 0, WX_NONE,       WC_NONE);  // cards/u007.py:13-21
    case SBC_U021: return WOP(WR_ALL,      TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_P0, WF_NONE,      0, 1, 0, WX_NONE,       WC_NONE);  // cards/u021.py:13-19
    case SBC_U026: return WOP(WR_BEHIND,   TK_ANY,  TS_ENEMY,    WS_FIRST,        WV_DAMAGE_PT,          WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/u026.py:13-16
    case SBC_U055: return WOP(WR_AHEAD,    TK_UNIT, TS_ENEMY,    WS_ALL,          WV_CONFUSE,            WA_P0, WF_X_CONFUSED, 0, 0, 0, WX_NONE,      WC_NONE);  // cards/u055.py:12-19
    case SBC_U074: return WOP(WR_AHEAD,    TK_UNIT, TS_ENEMY,    WS_FIRST,        WV_FORCE_ATTACK,       WA_P0, WF_NONE,      1, 0, 0, WX_NONE,       WC_NONE);  // cards/u074.py:12-19
    case SBC_U101: return WOP(WR_SURROUND, TK_UNIT, TS_ENEMY,    WS_ALL,          WV_DAMAGE_PT,          WA_P0, WF_FROZEN,    1, 0, 0, WX_NONE,       WC_ATTACKING_FROZEN_UNIT);  // cards/u101.py:13-26
    case SBC_U103: return WOP(WR_BORDER,   TK_UNIT, TS_ENEMY,    WS_ALL,          WV_FREEZE,             WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/u103.py:12-18
    case SBC_U111: return WOP(WR_SURROUND, TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_ONE, WF_NONE,     1, 0, 0, WX_NONE,       WC_REPEAT_P0);  // cards/u111.py:13-21
    case SBC_U306: return WOP(WR_ALL,      TK_ANY,  TS_FRIENDLY, WS_CHOICE,       WV_DAMAGE_PT,          WA_P0, WF_NONE,      0, 1, 0, WX_NONE,       WC_NONE);  // cards/u306.py:13-20
    case SBC_U313: return WOP(WR_SURROUND, TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_P0, WF_NONE,      0, 0, 0, WX_HEAL_P0,    WC_NONE);  // cards/u313.py:13-21
    case SBC_U314: return WOP(WR_AHEAD,    TK_UNIT, TS_FRIENDLY, WS_FIRST,        WV_PUSH,               WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/u314.py:11-17
    case SBC_U316: return WOP(WR_SURROUND, TK_UNIT, TS_FRIENDLY, WS_SHUFFLE_P0,   WV_VITALIZE,           WA_P0, WF_NONE,      0, 0, 0, WX_VITALIZE,   WC_NONE);  // cards/u316.py:13-23
    case SBC_U320: return WOP(WR_SURROUND, TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_P0, WF_NONE,      1, 0, 0, WX_NONE,       WC_NONE);  // cards/u320.py:13-19
    case SBC_U401: return WOP(WR_BORDER,   TK_UNIT, TS_ANY,      WS_ALL,          WV_DAMAGE_POISON_GUARDED, WA_P0, WF_NONE,   0, 0, 0, WX_NONE,       WC_NONE);  // cards/u401.py:13-22
    case SBC_U405: return WOP(WR_BORDER,   TK_UNIT, TS_ANY,      WS_ALL,          WV_DAMAGE_HEAL_SELF,   WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/u405.py:13-21
    case SBC_U411: return WOP(WR_ALL,      TK_UNIT, TS_ENEMY,    WS_SHUFFLE_P0,   WV_POISON,             WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/u411.py:13-22
    case SBC_UD01: return WOP(WR_ALL,      TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_P0, WF_DRAGON,    1, 0, 0, WX_NONE,       WC_NONE);  // cards/ud01.py:13-19
    case SBC_UD02: return WOP(WR_AHEAD,    TK_UNIT, TS_ANY,      WS_ALL,          WV_DAMAGE_PT,          WA_P0, WF_X_DRAGON,  0, 0, 0, WX_NONE,       WC_NONE);  // cards/ud02.py:13-19
    case SBC_UD31: return WOP(WR_SURROUND, TK_UNIT, TS_FRIENDLY, WS_CHOICE,       WV_HEAL,               WA_P0, WF_DRAGON,    1, 0, 0, WX_HEAL_P0,    WC_ATTACKING_UNIT);  // cards/ud31.py:13-24
    case SBC_UE01: return WOP(WR_ALL,      TK_UNIT, TS_ENEMY,    WS_CHOICE,       WV_DAMAGE_PT,          WA_ONE, WF_NONE,     1, 0, 0, WX_NONE,       WC_REPEAT_DMG);  // cards/ue01.py:11-19
    case SBC_UE12: return WOP(WR_AHEAD,    TK_UNIT, TS_ENEMY,    WS_ALL,          WV_DESTROY,            WA_P0, WF_NONE,      1, 0, 0, WX_NONE,       WC_NONE);  // cards/ue12.py:11-18
    case SBC_UE21: return WOP(WR_ALL,      TK_UNIT, TS_FRIENDLY, WS_ALL,          WV_COMMAND,            WA_P0, WF_LIMIT_SELF, 1, 1, 0, WX_NONE,      WC_NONE);  // cards/ue21.py:11-18
    case SBC_UE22: return WOP(WR_ALL,      TK_UNIT, TS_FRIENDLY, WS_SHUFFLE_P0,   WV_HEAL,               WA_DMG, WF_NONE,     1, 1, 0, WX_NONE,       WC_NONE);  // cards/ue22.py:12-22
    // spells (pov = board.current_player; no own tile)
    case SBC_S003: return WOP(WR_ALL,      TK_ANY,  TS_ENEMY,    WS_ALL,          WV_DAMAGE_RANDINT,     WA_P0, WF_NONE,      0, 0, 0, WX_NONE,       WC_NONE);  // cards/s003.py:14-19
    case SBC_S302: return WOP(WR_ALL,      TK_ANY,  TS_ENEMY,    WS_SHUFFLE_P1,   WV_DAMAGE_PT,          WA_P0, WF_NONE,      0, 0, 1, WX_NONE,       WC_NONE);  // cards/s302.py:14-22
    case SBC_S403: return WOP(WR_ALL,      TK_UNIT, TS_FRIENDLY, WS_ALL,          WV_HEAL_VITALIZE,      WA_P0, WF_POISONED,  0, 0, 0, WX_NONE,       WC_NONE);  // cards/s403.py:13-22
    default: return 0u;
  }
}

// The interpreter.  id = acting entity (-1 for a spell), p = the card's parameters.
SBW_NI void w_run_op(WG* wg, u32 op, int id, const i8* p, int pos_pt) {
  W_SHARED(wg);
  const int region = op & 15, kind = (op >> 4) & 3, side = (op >> 6) & 3, select = (op >> 8) & 15, verb = (op >> 12) & 31;
  const int amount_src = (op >> 17) & 7, filter = (op >> 20) & 7, after = (op >> 26) & 7, cond = (op >> 29) & 7;
  const int me = id >= 0 ? w_owner(wg, id) : 0;
  const int ex = id >= 0 ? w_ex(wg, id) : 0, ey = id >= 0 ? w_ey(wg, id) : 0;
  const int pov = ((op >> 23) & 1u) ? me : WCUR(wg);
  int repeat = 1;
  if (cond == WC_ATTACKING_UNIT || cond == WC_ATTACKING_FROZEN_UNIT) {
    if (pos_pt < 0 || pos_pt >= 20) return;
    const int tid = w_at_pt(wg, pos_pt);
    if (tid < 0 || w_is_struct(wg, tid)) return;
    if (cond == WC_ATTACKING_FROZEN_UNIT && !w_st(wg, tid, SB_ST_FROZEN)) return;
  } else if (cond == WC_REPEAT_P0) repeat = p[0];
  else if (cond == WC_REPEAT_DMG) repeat = wg->e_dmg[id];
  int amount = amount_src == WA_P0 ? p[0] : amount_src == WA_P1 ? p[1] : amount_src == WA_ONE ? 1 : (int)wg->e_dmg[id];
  TQ q = w_mkT(kind, side);
  if (filter == WF_CONSTRUCT) q = tq_types(q, 1u << UT_CONSTRUCT);
  else if (filter == WF_DRAGON) q = tq_types(q, 1u << UT_DRAGON);
  else if (filter == WF_X_DRAGON) q = tq_xtypes(q, 1u << UT_DRAGON);
  else if (filter == WF_X_CONFUSED) q = tq_xstatus(q, 1u << SB_ST_CONFUSED);
  else if (filter == WF_FROZEN) q = tq_status(q, 1u << SB_ST_FROZEN);
  else if (filter == WF_POISONED) q = tq_status(q, 1u << SB_ST_POISONED);
  else if (filter == WF_LIMIT_SELF) q = tq_limit(q, wg->e_str[id]);
  if ((op >> 25) & 1u) q = tq_base(q);
  const int exclude = ((op >> 24) & 1u) ? ey * 4 + ex : PT_NONE;
#pragma unroll 1
  for (int rep = 0; rep < repeat; rep++) {
    TL t;
    if (region == WR_ALL) t = w_targets(wg, pov, q, exclude);
    else if (region == WR_SURROUND) t = w_surrounding_t(wg, ex, ey, pov, q);
    else if (region == WR_BORDER) t = w_bordering_t(wg, ex, ey, pov, q);
    else t = w_column_targets(wg, ex, ey, pov, q, region == WR_AHEAD);
    // selection -> up to 22 points in `sel` (a tile list in order) or `few` (an explicit short list)
    PL few; few.v = 0; few.n = 0;
    bool use_few = true;
    const int n = tl_n(t);
    if (select == WS_ALL) use_few = false;
    else if (select == WS_CHOICE) { if (n > 0) pl_push(few, w_choice_tl(wg, t)); }
    else if (select == WS_FIRST) { if (n > 0) pl_push(few, tl_nth(t, 0)); }
    else if (select == WS_SHUFFLE_P0 || select == WS_SHUFFLE_P1) {
      // cards/s302.py shuffles even an empty list (no draw is consumed for n <= 1 either way)
      const int take = select == WS_SHUFFLE_P0 ? p[0] : p[1];
      if (n > 0) {
        w_expand(wg, t);
        w_shuffle(wg, wg->scr, n);
#pragma unroll 1
        for (int i = 0; i < n && i < take && i < 8; i++) pl_push(few, wg->scr[i]);
      }
    } else if (select == WS_FRONTMOST1) { if (n > 0) few = w_keyed_take(wg, t, false, true, 1); }
    else if (select == WS_FRONTMOST_P0_SHUFFLED) {
      if (n > 0) {
        few = w_keyed_take(wg, t, false, true, p[0] < 8 ? p[0] : 8);
        const int k = few.n;
        for (int i = 0; i < k; i++) wg->scr[i] = (i8)pl_get(few, i);
        w_shuffle(wg, wg->scr, k);
        few.v = 0; few.n = 0;
        for (int i = 0; i < k; i++) pl_push(few, wg->scr[i]);
      }
    }
    int i = 0;
#pragma unroll 1
    for (;;) {
      int pt;
      if (use_few) { if (i >= few.n) break; pt = pl_get(few, i++); }
      else { pt = tl_pop(t); if (pt == PT_NONE) break; }
      int tid;
      switch (verb) {
        case WV_DAMAGE_PT: w_deal_damage_pt(wg, pt, amount, 1); if (wg->err) return; break;
        case WV_DAMAGE_RANDINT:  // cards/s003.py:18-19: randint(p[1], p[0] + 1) per target
          if (w_need(wg, pt) < 0) return;
          w_deal_damage_pt(wg, pt, p[1] + w_rng_below(wg, p[0] + 1 - p[1]), 1);
          if (wg->err) return;
          break;
        case WV_DAMAGE_HEAL_SELF: {  // cards/u405.py:19-21
          const int dealt = w_deal_damage_pt(wg, pt, amount, 1);
          if (wg->err) return;
          wv_heal(wg, id, dealt);
          break; }
        case WV_DAMAGE_POISON_GUARDED:  // cards/u401.py:19-22: the only effect that guards board.at() against None
          tid = w_at_pt(wg, pt);
          if (tid >= 0) {
            w_deal_damage(wg, tid, amount, 0, 1);
            if (w_is_struct(wg, tid)) { WERR(wg, SB_ERR_NONE_TARGET); return; }
            wv_poison(wg, tid);
          }
          break;
        default:
          tid = w_need(wg, pt);
          if (tid < 0) return;
          switch (verb) {
            case WV_HEAL: wv_heal(wg, tid, amount); break;
            case WV_HEAL_VITALIZE: wv_heal(wg, tid, amount); wv_vitalize(wg, tid); break;
            case WV_VITALIZE: wv_vitalize(wg, tid); break;
            case WV_POISON: wv_poison(wg, tid); break;
            case WV_FREEZE: wv_freeze(wg, tid); break;
            case WV_CONFUSE: wv_confuse(wg, tid); break;
            case WV_DESTROY: w_destroy(wg, tid, 1); break;
            case WV_PUSH: wv_push(wg, tid, ex, ey); break;
            case WV_FORCE_ATTACK: wv_force_attack(wg, id, wpt_x(pt), wpt_y(pt)); break;
            case WV_COMMAND:
            case WV_DECONFUSE_COMMAND:
              if (w_is_struct(wg, tid)) { WERR(wg, SB_ERR_NONE_TARGET); return; }
              if (verb == WV_DECONFUSE_COMMAND && w_st(wg, tid, SB_ST_CONFUSED)) w_st_remove(wg, tid, SB_ST_CONFUSED);
              wv_command(wg, tid);
              break;
            default: break;
          }
          break;
      }
    }
  }
  if (after == WX_HEAL_P0) wv_heal(wg, id, p[0]);
  else if (after == WX_VITALIZE) wv_vitalize(wg, id);
  else if (after == WX_DESTROY) w_destroy(wg, id, 1);
}

// The bespoke handlers of the cards that the default decks do not hold, out of line: the handlers that the bench's
// games run (and the dispatch to them) then stay together in a few instruction-cache lines of w_effect instead of
// being spread over the 69 KB of all handlers (tools/hot_footprint.py, DESIGN.md section 10).  Same rules either way.
SBW_NI void w_effect_rare(WG* wg, int id, int pos_pt, int has_source) {
  W_SHARED(wg);
  const int card = wg->e_card[id];
  const DCard& cd = WCARD(wg, card);
  const i8* p = cd.p;
  const int me = w_owner(wg, id);
  const int ex = w_ex(wg, id), ey = w_ey(wg, id);
  int tid;
  TL t;
  switch (card) {
    case SBC_B005: {  // cards/b005.py:15-33, including the memories of remembered temple copies (deepcopy)
      t = w_surrounding_t(wg, ex, ey, WCUR(wg), w_mkT(TK_ANY, TS_FRIENDLY));
      int mine = 0;
#pragma unroll 1
      for (int i = 0; i < wg->n_mem; i++) if (wg->mem[i].parent < 0 && wg->mem[i].b005 == id) mine++;
      if (mine == 0) {
#pragma unroll 1
        for (;;) {
          const int pt = tl_pop(t);
          if (pt == PT_NONE) break;
          tid = w_need(wg, pt);
          if (tid < 0) return;
          const int r = w_mem_push_entity(wg, id, -1, pt, tid);
          if (r < 0) return;
          if (wg->e_card[tid] == SBC_B005) {  // the copy carries a deep copy of that temple's own memories
            const int nm0 = wg->n_mem;
#pragma unroll 1
            for (int q = 0; q < nm0; q++)
              if (wg->mem[q].parent < 0 && wg->mem[q].b005 == tid && w_mem_copy_subtree(wg, q, r, nm0) < 0) return;
          }
        }
      } else {
        int count = 0;
        const int nm0 = wg->n_mem;
#pragma unroll 1
        for (int i = 0; i < nm0 && count < p[0]; i++) {
          const WMem m = wg->mem[i];
          if (m.parent >= 0 || m.b005 != id) continue;
          const int occ = w_at_pt(wg, m.pos);
          if (occ < 0 || (wg->e_card[occ] == m.card && ((wg->e_fl[occ] ^ m.fl) & (WEF_OWNER | WEF_STRUCT)) == 0)) {
            if (m.fl & WEF_SINGLE) { WERR(wg, SB_ERR_UNSUPPORTED); return; }  // detached copy: not modelled (DESIGN.md)
            const int c = w_new_ent(wg, m.card, m.fl & WEF_OWNER, m.strength);
            wg->e_fl[c] = (u8)((wg->e_fl[c] & ~WEF_FIXED) | (m.fl & WEF_FIXED));
            u32 w = 0;
#pragma unroll
            for (int k = 0; k < 5; k++) w |= (u32)(m.st[k] > 63 ? 63 : m.st[k]) << (SB_ST_BITS * k);
            wg->e_st[c] = w;
            w_set_xy(wg, wpt_x(m.pos), wpt_y(m.pos), c);
#pragma unroll 1
            for (int q = i + 1; q < nm0; q++)  // the restored object keeps its own ability_remembered
              if (wg->mem[q].parent == i) { wg->mem[q].parent = -1; wg->mem[q].b005 = (i8)c; }
            count++;
          }
        }
        w_mem_delete_temple(wg, id);
      }
      break; }
    case SBC_B006: {  // cards/b006.py:14-39: ability_strength, ability_targets
      t = w_targets(wg, WCUR(wg), tq_xstatus(w_mkT(TK_UNIT, TS_FRIENDLY), 1u << SB_ST_VITALIZED), PT_NONE);
      const int ns = w_expand(wg, t);
      w_shuffle(wg, wg->scr, ns);
      PL few; few.v = 0; few.n = 0;
#pragma unroll 1
      for (int i = 0; i < ns && i < p[1] && i < 8; i++) pl_push(few, wg->scr[i]);
#pragma unroll 1
      for (int i = 0; i < few.n; i++) { tid = w_need(wg, pl_get(few, i)); if (tid < 0) return; wv_vitalize(wg, tid); }
      PL tiles; tiles.v = 0; tiles.n = 0;
      const int fr = w_column_first_tile(wg, ex, ey, WCUR(wg), true);
      const int bh = w_column_first_tile(wg, ex, ey, WCUR(wg), false);
      if (fr != PT_NONE && w_at_pt(wg, fr) < 0 && w_within_front_line(wg, me, wpt_y(fr))) pl_push(tiles, fr);
      if (bh != PT_NONE && w_at_pt(wg, bh) < 0) pl_push(tiles, bh);
      if (tiles.n > 0) {
        const int c = w_new_ent(wg, card, me, p[0]);
        const int where = w_choice_pl(wg, tiles);
        w_struct_play(wg, c, wpt_x(where), wpt_y(where));
      }
      break; }
    case SBC_B007: {  // cards/b007.py:12-19
      const int opp = w_opponent_of(wg, me);
      if (wg->pl[me].base == wg->pl[opp].base) return;
      const int stronger = wg->pl[me].base > wg->pl[opp].base ? me : opp;
      w_player_damage(wg, stronger, p[0]);
      const int o2 = w_opponent_of(wg, stronger);
      wg->pl[o2].base = (i16)(wg->pl[o2].base + p[0]);
      break; }
    case SBC_B008: {  // cards/b008.py:14-26
      WPly& pl = wg->pl[me];
      if (pl.n_hand > 0 && WCARD(wg, pl.hand[0].card).kind == KIND_UNIT) pl.hand[0].flags ^= SB_CF_FIXED;
      t = w_targets(wg, WCUR(wg), tq_status(w_mkT(TK_UNIT, TS_ANY), 1u << SB_ST_CONFUSED), PT_NONE);
      if (tl_n(t) > 0) {
        const PL first = w_keyed_take(wg, t, true, false, 1);
        tid = w_need(wg, pl_get(first, 0));
        if (tid >= 0) w_destroy(wg, tid, 1);
      }
      break; }
    case SBC_B305: {  // cards/b305.py:16-45: ability_amount, ability_mana, original_cost
      t = w_targets(wg, WCUR(wg), w_mkT(TK_STRUCTURE, TS_FRIENDLY), ey * 4 + ex);
#pragma unroll 1
      for (int i = 0; i < p[0]; i++) {
        const int pt = tl_pop(t);
        if (pt == PT_NONE) break;
        tid = w_need(wg, pt);
        if (tid < 0) return;
        if (wg->e_card[tid] == card) {
          const int tx = wpt_x(pt), ty = wpt_y(pt);
          TL sp = w_surrounding_t(wg, tx, ty, WCUR(wg), w_mkT(TK_UNIT, TS_ANY));
#pragma unroll 1
          for (;;) {
            const int s = tl_pop(sp);
            if (s == PT_NONE) break;
            const int nx = wpt_x(s) - tx + ex, ny = wpt_y(s) - ty + ey;
            if (w_valid_xy(nx, ny)) { const int u = w_need(wg, s); if (u < 0) return; wv_teleport(wg, u, nx, ny); }
          }
          w_destroy(wg, tid, 1);
          WPly& pl = wg->pl[me];
          if (pl.n_deck == 0) { WERR(wg, SB_ERR_INDEX); return; }
          pl.deck[pl.n_deck - 1].cost = p[2];
          return;
        }
      }
      {  // no other temple: the BOARD INSTANCE itself goes to the hand with cost 2 (a live link)
        WPly& pl = wg->pl[me];
        const bool single = (wg->e_fl[id] & WEF_SINGLE) != 0;
        if (!single) { if (pl.n_deck == 0) { WERR(wg, SB_ERR_INDEX); return; } pl.n_deck = (u8)(pl.n_deck - 1); }
        if (pl.n_hand >= HAND_W) { WERR(wg, SB_ERR_OVERFLOW); return; }
        WCard r; r.card = (u8)card; r.cost = p[1]; r.flags = (u8)((single ? SB_CF_SINGLE_USE : 0) | SB_CF_OBJ); r.link = (i8)id; r.wn = 0; r.xstr = 0;
        const int nh = pl.n_hand;
        pl.hand[nh] = r;
        pl.n_hand = (u8)(nh + 1);
        wg->n_obj = (u8)(wg->n_obj + 1);
      }
      break; }
    case SBC_U017: {  // cards/u017.py:18-34
      WPly& pl = wg->pl[me];
      int nc = 0;
#pragma unroll 1
      for (int i = 0; i < pl.n_hand; i++) if (WCARD(wg, pl.hand[i].card).kind == KIND_SPELL && pl.hand[i].cost <= 8) wg->scr[nc++] = (i8)i;
      if (nc > 0) {
        w_shuffle(wg, wg->scr, nc);
        int remaining = 8;
        PL chosen; chosen.v = 0; chosen.n = 0;
#pragma unroll 1
        for (int i = 0; i < nc; i++) { const int h = wg->scr[i]; if (pl.hand[h].cost <= remaining) { pl_push(chosen, h); remaining -= pl.hand[h].cost; } }
#pragma unroll 1
        for (int i = 0; i < chosen.n; i++) {
          const int idx = pl_get(chosen, i);
          const DCard& c = WCARD(wg, pl.hand[idx].card);
          int where = PT_NONE;
          if (c.flags & DCF_TARGET) {
            where = w_choice_tl(wg, w_targets(wg, WCUR(wg), w_card_target(c), PT_NONE));
            if (wg->err) return;
          }
          w_player_play(wg, me, idx, where);
          if (wg->err) return;
          PL fixed; fixed.v = 0; fixed.n = 0;  // later hand indices shift down past the removed card
#pragma unroll 1
          for (int k = 0; k < chosen.n; k++) { const int v = pl_get(chosen, k); pl_push(fixed, (k > i && v > idx) ? v - 1 : v); }
          chosen = fixed;
        }
      }
      break; }
    case SBC_U018: {  // cards/u018.py:13-26
      t = w_surrounding_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ANY));
      const DCard* cards = wg->cards;
      W_SHARED(cards);
      const int cnt = w_popc(w_or_tiles(wg, t.m, [&](int s) -> u32 { return 1u << cards[wg->e_card[s]].first_type; }));
#pragma unroll 1
      for (int k = 0; k < cnt; k++) {
        const int where = w_choice_tl(wg, w_targets(wg, WCUR(wg), tq_base(w_mkT(TK_ANY, TS_ENEMY)), PT_NONE));
        if (wg->err) return;
        w_deal_damage_pt(wg, where, p[0], 1);
        if (wg->err) return;
      }
      break; }
    case SBC_U036:  // cards/u036.py:12-14
      if (wg->pl[me].n_hand == 0) { tid = w_need(wg, ey * 4 + ex); if (tid >= 0) wv_heal(wg, tid, p[0]); }
      break;
    case SBC_U040:  // cards/u040.py:13-22 (the print is dropped); respawn unit.py:384-402
      if (has_source) {
        const PL sl = w_surround_list(ex, ey);
        if (sl.n > 0) {
          const int where = w_choice_pl(wg, sl);
          const int c = w_new_ent(wg, card, me, p[0]);
          w_set_xy(wg, wpt_x(where), wpt_y(where), c);
        }
      }
      break;
    case SBC_U050:  // cards/u050.py:13-15
      if (ey == 4) w_gain_speed(wg, id, p[0]);
      break;
    case SBC_U051:  // cards/u051.py:14-21: ability_movement, ability_strength
      if (tl_n(w_bordering_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ANY))) == 0) w_gain_speed(wg, id, p[0]);
      else wv_heal(wg, id, p[1]);
      break;
    case SBC_U076:  // cards/u076.py:14-26: ability_damage, ability_strength
      t = w_surrounding_t(wg, ex, ey, WCUR(wg), tq_xtypes(w_mkT(TK_UNIT, TS_ANY), 1u << UT_DRAGON));
      if (tl_n(t) > 0) {
        tid = w_need(wg, w_choice_tl(wg, t));
        if (tid < 0) return;
        w_deal_damage(wg, tid, p[0], 0, 1);
        if (wg->e_str[tid] <= 0) w_spawn_token_unit(wg, me, wg->e_pos[tid], p[1], UT_DRAGON);
      }
      break;
    case SBC_U106:  // cards/u106.py:13-18
      if (tl_n(w_bordering_t(wg, ex, ey, WCUR(wg), w_mkT(TK_STRUCTURE, TS_FRIENDLY))) > 0 || ey == 4) wv_heal(wg, id, p[0]);
      break;
    case SBC_U117: wv_freeze(wg, id); break;          // cards/u117.py:11-12
    case SBC_U216: w_player_damage(wg, me, p[0]); break;  // cards/u216.py:12-13
    case SBC_U217: {  // cards/u217.py:13-17
      const TL row = tl_tiles(0xF0000u & ~wg->occ, true);
      if (tl_n(row) > 0) w_spawn_token_unit(wg, me, w_choice_tl(wg, row), p[0], UT_SATYR);
      break; }
    case SBC_U310: {  // cards/u310.py:12-41
      t = w_bordering_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ENEMY));
      const u32 m = t.m;
      const int behind = (ey < 4 && ((m >> ((ey + 1) * 4 + ex)) & 1u)) ? (ey + 1) * 4 + ex : PT_NONE;
      const int right = (ex < 3 && ((m >> (ey * 4 + ex + 1)) & 1u)) ? ey * 4 + ex + 1 : PT_NONE;
      const int left = (ex > 0 && ((m >> (ey * 4 + ex - 1)) & 1u)) ? ey * 4 + ex - 1 : PT_NONE;
      const int front = (ey > 0 && ((m >> ((ey - 1) * 4 + ex)) & 1u)) ? (ey - 1) * 4 + ex : PT_NONE;
      int target = PT_NONE;
      if (behind != PT_NONE && wpt_y(behind) < 4 && w_at_xy(wg, wpt_x(behind), wpt_y(behind) + 1) < 0) target = behind;
      else if (left != PT_NONE && wpt_x(left) > 0 && w_at_xy(wg, wpt_x(left) - 1, wpt_y(left)) < 0) target = left;
      else if (right != PT_NONE && wpt_x(right) < 3 && w_at_xy(wg, wpt_x(right) + 1, wpt_y(right)) < 0) target = right;
      else if (front != PT_NONE && wpt_y(front) > 0 && w_at_xy(wg, wpt_x(front), wpt_y(front) - 1) < 0) target = front;
      if (target == PT_NONE) { WERR(wg, SB_ERR_INDEX); return; }  // UnboundLocalError
      tid = w_need(wg, target);
      if (tid >= 0) wv_push(wg, tid, ex, ey);
      break; }
    case SBC_U403: {  // cards/u403.py:14-24: ability_amount, ability_strength
      t = w_surrounding_t(wg, ex, ey, WCUR(wg), tq_status(w_mkT(TK_UNIT, TS_ANY), 1u << SB_ST_POISONED));
#pragma unroll 1
      for (;;) {
        const int pt = tl_pop(t);
        if (pt == PT_NONE) break;
        const PL em = pl_empty_of(wg, w_border_list(wpt_x(pt), wpt_y(pt)));
#pragma unroll 1
        for (int k = 0; k < em.n; k++) wg->scr[k] = (i8)pl_get(em, k);
        w_shuffle(wg, wg->scr, em.n);
        PL few; few.v = 0; few.n = 0;
#pragma unroll 1
        for (int k = 0; k < em.n && k < p[0]; k++) pl_push(few, wg->scr[k]);
#pragma unroll 1
        for (int k = 0; k < few.n; k++) w_spawn_token_unit(wg, me, pl_get(few, k), p[1], UT_TOAD);
      }
      break; }
    case SBC_U406: {  // cards/u406.py:13-20
      const PL em = pl_empty_of(wg, w_border_list(ex, ey));
      if (em.n > 0) { const int where = w_choice_pl(wg, em); w_spawn_token_unit(wg, w_opponent_of(wg, me), where, p[0], UT_RAVEN); }
      break; }
    case SBC_UA03: {  // cards/ua03.py:12-15
      PL row; row.v = 0; row.n = 0;
#pragma unroll 1
      for (int x = 0; x < 4; x++) if (wg->board[ey * 4 + x] < 0) pl_push(row, ey * 4 + x);
      pl_push(row, ey * 4 + ex);
      const int where = w_choice_pl(wg, row);
      wv_teleport(wg, id, wpt_x(where), wpt_y(where));
      break; }
    case SBC_UA04: {  // cards/ua04.py:12-33
      const TL lp = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_FRIENDLY), PT_NONE);
      const TL rp = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_ENEMY), PT_NONE);
      const int nl = tl_n(lp), nr = tl_n(rp);
      if (nl != nr) {
        TL src = nl > nr ? lp : rp;
        const int mn = w_min_tiles(wg, src.m, [&](int s) -> int { return wg->e_str[s]; });
        src.m &= w_tilemask(wg, [&](int s) -> bool { return wg->e_str[s] == mn; });
        if (tl_n(src) > 0) w_destroy(wg, w_at_pt(wg, tl_nth(src, w_rng_below(wg, tl_n(src)))), 1);
      }
      break; }
    case SBC_UA05: {  // cards/ua05.py:13-19
      const PL em = pl_empty_of(wg, w_side_list(ex, ey));
#pragma unroll 1
      for (int k = 0; k < em.n; k++) w_spawn_token_unit(wg, me, pl_get(em, k), p[0], UT_ANCIENT);
      break; }
    case SBC_UA20:  // cards/ua20.py:21-32: ability_cost, ability_level
      if (tl_n(w_column_targets(wg, ex, ey, me, w_mkT(TK_UNIT, TS_ENEMY), true)) == 0) {
        WPly& pl = wg->pl[me];
        const int k = w_rng_below(wg, 4);
        const int c = k == 0 ? SBC_B005 : k == 1 ? SBC_B006 : k == 2 ? SBC_B203 : SBC_B305;
        if (pl.n_deck >= DECK_W) { WERR(wg, SB_ERR_OVERFLOW); return; }
        WCard r; r.card = (u8)c; r.cost = p[0]; r.flags = SB_CF_SINGLE_USE; r.link = -1; r.wn = 0; r.xstr = 0;
        const int nd = pl.n_deck;
        pl.deck[nd] = r;
        pl.n_deck = (u8)(nd + 1);
      }
      break;
    case SBC_UE03: {  // cards/ue03.py:11-17
      const PL em = pl_empty_of(wg, w_border_list(ex, ey));
      if (em.n > 0) w_spawn_token_unit(wg, me, w_choice_pl(wg, em), wg->e_str[id], UT_ELDER);
      break; }
    case SBC_UE04: {  // cards/ue04.py:12-18
      t = w_targets(wg, me, w_mkT(TK_UNIT, TS_ENEMY), PT_NONE);
      const int mine = wg->e_str[id];
      const int c = w_popc(t.m & w_tilemask(wg, [&](int s) -> bool { return wg->e_str[s] > mine; }));
      wv_heal(wg, id, c * p[0]);
      break; }
    case SBC_UE05: {  // cards/ue05.py:12-19
      const int mine = wg->e_str[id];
      t = w_targets(wg, me, tq_limit(w_mkT(TK_UNIT, TS_FRIENDLY), mine - 1), ey * 4 + ex);
#pragma unroll 1
      for (int i = 0; i < p[0]; i++) { const int pt = tl_pop(t); if (pt == PT_NONE) break; wg->e_str[wg->board[pt]] = (i16)mine; }
      break; }
    case SBC_UE11: wv_heal(wg, id, p[0]); break;  // cards/ue11.py:12-13
    case SBC_UE31: wg->e_str[id] = p[0]; break;  // cards/ue31.py:12-13
    case SBC_UE32: {  // cards/ue32.py:12-22
      const int damage = wg->e_str[id] < 6 ? (int)wg->e_str[id] : 6;
      t = w_column_targets(wg, ex, ey, me, w_mkT(TK_ANY, TS_ENEMY), true);
      if (tl_n(t) > 0) w_deal_damage_pt(wg, tl_nth(t, 0), damage, 1);
      else w_player_damage(wg, w_opponent_of(wg, me), damage);
      break; }
    case SBC_UE41: wv_convert(wg, id); break;  // cards/ue41.py:10-11
    case SBC_UE42: {  // cards/ue42.py:12-15
      const int amount = wg->e_dmg[id] < p[0] ? (int)wg->e_dmg[id] : (int)p[0];
      wv_heal(wg, id, w_player_damage(wg, w_opponent_of(wg, me), amount));
      break; }
    case SBC_UP02: wv_heal(wg, id, p[0] * w_count_types_friendly(wg)); break;  // cards/up02.py:12-20
    case SBC_UP03: {  // cards/up03.py:12-28
      const int c = w_count_types_friendly(wg);
      t = w_surrounding_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ENEMY));
#pragma unroll 1
      for (;;) {
        const int pt = tl_pop(t);
        if (pt == PT_NONE) break;
        tid = w_need(wg, pt);
        if (tid < 0) return;
        const int s = wg->e_str[tid] - p[0] * c;
        wg->e_str[tid] = (i16)(s > 1 ? s : 1);  // unit.py:233-234 reduce
      }
      break; }
    default: break;
  }
}

SBW_NI void w_effect(WG* wg, int id, int pos_pt, int has_source) {
  W_SHARED(wg);
  const int card = wg->e_card[id];
  const DCard& cd = WCARD(wg, card);
  const i8* p = cd.p;
  const u32 op = w_effect_op(card);
  if (op) { w_run_op(wg, op, id, p, pos_pt); return; }
  const int me = w_owner(wg, id);
  const int ex = w_ex(wg, id), ey = w_ey(wg, id);
  int tid;
  TL t;
  switch (card) {
    case SBC_B304:  // cards/b304.py:12-13
      w_deal_damage(wg, id, p[0], 0, 1);
      break;
    case SBC_U053:  // cards/u053.py:14-24: ability_amount=1, ability_movement=2
      if (tl_n(w_surrounding_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ANY))) == 0) w_gain_speed(wg, id, p[1]);
      else if (tl_n(w_bordering_t(wg, ex, ey, WCUR(wg), w_mkT(TK_UNIT, TS_ANY))) == 0) w_gain_speed(wg, id, p[0]);
      break;
    case SBC_U061:  // cards/u061.py:12-23
      wv_confuse(wg, id);
      t = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_FRIENDLY), ey * 4 + ex);
      if (tl_n(t) > 0) { tid = w_need(wg, w_choice_tl(wg, t)); if (tid < 0) return; wv_confuse(wg, tid); }
      w_gain_speed(wg, id, 2);
      break;
    case SBC_U071: {  // cards/u071.py:12-27
      t = w_bordering_t(wg, ex, ey, me, tq_xstatus(w_mkT(TK_UNIT, TS_ENEMY), 1u << SB_ST_CONFUSED));
      if (tl_n(t) > 0) {
        tid = w_need(wg, w_choice_tl(wg, t));
        if (tid < 0) return;
        wv_confuse(wg, tid);
        const int fr = w_column_first_tile(wg, ex, ey, WCUR(wg), true);
        if (fr != PT_NONE && w_at_pt(wg, fr) < 0) wv_teleport(wg, id, wpt_x(fr), wpt_y(fr));
      }
      break; }
    case SBC_U206: w_player_damage(wg, me, p[0]); break;  // cards/u206.py:12-13
    case SBC_U211: {  // cards/u211.py:14-19: ability_max_strength, ability_min_strength
      const int fr = w_column_first_tile(wg, ex, ey, WCUR(wg), true);
      if (fr != PT_NONE && w_at_pt(wg, fr) < 0) {
        const int s = p[1] + w_rng_below(wg, p[0] + 1 - p[1]);
        w_spawn_token_unit(wg, me, fr, s, UT_SATYR);
      }
      break; }
    case SBC_U302:  // cards/u302.py:12-23
      if (pos_pt < 0 || pos_pt >= 20) return;
      tid = w_at_pt(wg, pos_pt);
      if (tid < 0 || w_is_struct(wg, tid)) return;
      if (wg->e_str[tid] > wg->e_str[id]) {
        w_deal_damage(wg, tid, p[0], 0, 1);
        if (wg->e_str[tid] > 0) wv_push(wg, tid, w_ex(wg, id), w_ey(wg, id));
      }
      break;
    case SBC_U305:  // cards/u305.py:13-21: +p0 to a bordering friendly CONSTRUCT and to itself, only if there is one
      t = w_bordering_t(wg, ex, ey, WCUR(wg), tq_types(w_mkT(TK_UNIT, TS_FRIENDLY), 1u << UT_CONSTRUCT));
      if (tl_n(t) > 0) { tid = w_need(wg, w_choice_tl(wg, t)); if (tid < 0) return; wv_heal(wg, tid, p[0]); wv_heal(wg, id, p[0]); }
      break;
    case SBC_UA07:  // cards/ua07.py:11-22
      switch (w_rng_below(wg, 5)) {
        case 0: wv_freeze(wg, id); break;
        case 1: wv_poison(wg, id); break;
        case 2: wv_vitalize(wg, id); break;
        case 3: wv_confuse(wg, id); break;
        case 4: wv_disable(wg, id); break;
      }
      break;
    default: w_effect_rare(wg, id, pos_pt, has_source); break;
  }
}

SBW_NI void w_spell_effect(WG* wg, int card, int caster, int pos_pt) {
  W_SHARED(wg);
  const i8* p = WCARD(wg, card).p;
  const u32 op = w_effect_op(card);
  if (op) { w_run_op(wg, op, -1, p, pos_pt); return; }
  int tid;
  TL t;
  switch (card) {
    case SBC_S001: w_deal_damage_pt(wg, pos_pt, p[0], 1); break;  // cards/s001.py:13-14
    case SBC_S004: {  // cards/s004.py:14-23: ability_max_amount, ability_min_amount
      TL tl = w_within_front_line_tiles(wg, caster);
      tl.m &= ~wg->occ;
      const int ne = tl_n(tl);
      if (ne > 0) {
        w_expand(wg, tl);
        w_shuffle(wg, wg->scr, ne);
        const int amount = p[1] + w_rng_below(wg, p[0] + 1 - p[1]);
        PL few; few.v = 0; few.n = 0;
#pragma unroll 1
        for (int i = 0; i < ne && i < amount && i < 8; i++) pl_push(few, wg->scr[i]);
#pragma unroll 1
        for (int i = 0; i < few.n; i++) w_spawn_token_unit(wg, caster, pl_get(few, i), 1, UT_TOAD);
      }
      break; }
    case SBC_S007:  // cards/s007.py:13-16
      tid = w_need(wg, pos_pt);
      if (tid < 0) return;
      wv_heal(wg, tid, p[0]); wv_vitalize(wg, tid);
      break;
    case SBC_S012: {  // cards/s012.py:13-18
      TL tl = w_within_front_line_tiles(wg, caster);
      tl.m &= ~wg->occ;
      if (tl_n(tl) > 0) w_spawn_token_unit(wg, caster, w_choice_tl(wg, tl), p[0], UT_KNIGHT);
      break; }
    case SBC_S013: {  // cards/s013.py:13-27
      u32 taken = 0;
      int nc = 0;
      u64 order = 0, order2 = 0;  // chosen points in pick order, 5 bits each (12 per word; 16 unit types -> two words)
#pragma unroll 1
      for (int ut = 0; ut < 16; ut++) {
        t = w_targets(wg, WCUR(wg), tq_types(w_mkT(TK_UNIT, TS_ANY), 1u << ut), PT_NONE);
        t.m &= ~taken;
        if (tl_n(t) > 0) {
          const int c = w_choice_tl(wg, t);
          if (nc < 12) order |= (u64)c << (5 * nc); else order2 |= (u64)c << (5 * (nc - 12));
          nc++;
          taken |= 1u << c;
        }
      }
#pragma unroll 1
      for (int i = 0; i < nc; i++) {
        const int pt = (int)((i < 12 ? (order >> (5 * i)) : (order2 >> (5 * (i - 12)))) & 31u);
        w_deal_damage_pt(wg, pt, p[0], 1);
        if (wg->err) return;
      }
      break; }
    case SBC_S021:  // cards/s021.py:13-25
      tid = w_need(wg, pos_pt);
      if (tid < 0) return;
      wv_confuse(wg, tid);
      t = w_targets(wg, WCUR(wg), tq_types(w_mkT(TK_UNIT, TS_FRIENDLY), 1u << UT_FELINE), PT_NONE);
      if (tl_n(t) > 0) {
        const int mn = w_min_tiles(wg, t.m, [&](int s) -> int { return wg->e_str[s]; });
        t.m &= w_tilemask(wg, [&](int s) -> bool { return wg->e_str[s] == mn; });
        tid = w_need(wg, w_choice_tl(wg, t));
        if (tid >= 0) wv_heal(wg, tid, p[0]);
      }
      break;
    case SBC_S101: {  // cards/s101.py:14-22: ability_mana, ability_strength
      wg->pl[caster].mana = (i16)(wg->pl[caster].mana + p[0]);
      t = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_FRIENDLY), PT_NONE);
      if (tl_n(t) == 0) { WERR(wg, SB_ERR_INDEX); return; }
      const PL first = w_keyed_take(wg, t, true, false, 1);
      tid = w_need(wg, pl_get(first, 0));
      if (tid >= 0) wv_heal(wg, tid, p[1]);
      break; }
    case SBC_S104:  // cards/s104.py:13-19
      tid = w_need(wg, pos_pt);
      if (tid < 0) return;
      if (w_st(wg, tid, SB_ST_FROZEN)) w_deal_damage(wg, tid, p[0], 0, 1); else wv_freeze(wg, tid);
      break;
    case SBC_S105:  // cards/s105.py:13-14
      tid = w_need(wg, pos_pt);
      if (tid >= 0) wv_heal(wg, tid, p[0]);
      break;
    case SBC_S203: {  // cards/s203.py:14-30; list(set(...)) order is str-hash dependent upstream (Q14): canonical first-occurrence order
      // first-occurrence order over the surrounding queries of every friendly unit: up to 20 tiles + 2 bases, 5 bits each
      u64 lo = 0, hi = 0;
      int na = 0;
      u32 seen = 0;
      TL fr = w_targets(wg, WCUR(wg), w_mkT(TK_UNIT, TS_FRIENDLY), PT_NONE);
#pragma unroll 1
      for (;;) {
        const int f = tl_pop(fr);
        if (f == PT_NONE) break;
        TL sp = w_surrounding_t(wg, wpt_x(f), wpt_y(f), WCUR(wg), tq_base(w_mkT(TK_ANY, TS_ENEMY)));
#pragma unroll 1
        for (;;) {
          const int s = tl_pop(sp);
          if (s == PT_NONE) break;
          if (!((seen >> s) & 1u)) {
            seen |= 1u << s;
            if (na < 12) lo |= (u64)s << (5 * na); else hi |= (u64)s << (5 * (na - 12));
            na++;
          }
        }
      }
#pragma unroll 1
      for (int i = 0; i < na; i++) {
        const int pt = (int)((i < 12 ? (lo >> (5 * i)) : (hi >> (5 * (i - 12)))) & 31u);
        w_deal_damage_pt(wg, pt, p[0], 1);
        if (wg->err) return;
      }
      break; }
    default: break;
  }
}
