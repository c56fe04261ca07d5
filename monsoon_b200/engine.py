"""Batched Stormbound on one B200: device-resident packed states + the kernels of libsb_b200.so.

torch is plumbing only (device memory, streams, torch.distributed); every rule, draw and score is
computed by the CUDA kernels behind the C ABI (include/sb_b200.h).  No CPU path exists.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._card_table import CARDS

STATE_BYTES = 512
N_ACTIONS = 156
MASK_WORDS = 5
PASS = 155

CARD_INDEX = {c["name"]: i for i, c in enumerate(CARDS)}
# games/stormbound.py:295-302
DEFAULT_DECKS = (
    ["UA07", "U007", "U306", "U061", "B304", "U305", "U320", "U302", "U313", "UA02", "UT32", "U316"],
    ["UA07", "U007", "U001", "U053", "UE01", "U211", "U206", "U071", "U020", "S013", "B001", "U061"],
)
DEFAULT_FACTIONS = (3, 2)  # Faction.IRONCLAD, Faction.SWARM


def deck_indices(names):
    return [CARD_INDEX[n.upper()] for n in names]


class Engine:
    """One handle per device (sb_create).  All tensors passed in must live on that device."""

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise _lib.SbError("no CUDA device: the B200 simulator has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        h = ctypes.c_void_p()
        rc = self.lib.sb_create(self.device.index, ctypes.byref(h))
        if rc != 0:
            msg = self.lib.sb_last_error(h).decode() if h else "sb_create failed"
            raise _lib.SbError("sb_create(%d) -> %d: %s" % (self.device.index, rc, msg))
        self.h = h  # the caller's current device is left alone: every sb_* entry switches to the handle's device and back
        self._default_decks = None
        self.sm_count = self.lib.sb_sm_count(h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.sb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    # ------------------------------------------------------------------ helpers
    def _check(self, rc, what):
        if rc != 0:
            raise _lib.SbError("%s -> %d: %s" % (what, rc, self.lib.sb_last_error(self.h).decode()))

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _p(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    def _dev(self, t, dtype):
        assert t.device == self.device and t.dtype == dtype and t.is_contiguous(), (t.device, t.dtype)
        return t

    @property
    def launches(self):
        return int(self.lib.sb_launch_count(self.h))

    def set_option(self, key, value):
        """sb_set_option: tuning knobs of the rollout kernels (include/sb_b200.h)"""
        self._check(self.lib.sb_set_option(self.h, key.encode(), int(value)), "sb_set_option(%s)" % key)

    def empty_states(self, n):
        return torch.empty((n, STATE_BYTES), dtype=torch.uint8, device=self.device)

    # ------------------------------------------------------------------ C ABI wrappers (device tensors)
    def reset(self, seeds, decks=None, factions=None, out=None):
        """seeds: int64/uint64 tensor [n] on device.  decks: None (default decks), [2,k] shared or [n,2,k]."""
        n = seeds.numel()
        seeds = self._dev(seeds.view(torch.int64) if seeds.dtype != torch.int64 else seeds, torch.int64)
        if decks is None:
            if self._default_decks is None:  # built once: two pageable H2D copies per call otherwise
                self._default_decks = (torch.tensor([deck_indices(d) for d in DEFAULT_DECKS], dtype=torch.uint8, device=self.device),
                                       torch.tensor(DEFAULT_FACTIONS, dtype=torch.uint8, device=self.device))
            decks, factions = self._default_decks
        decks = self._dev(decks, torch.uint8)
        shared = 1 if decks.dim() == 2 else 0
        n_deck = decks.shape[-1]
        if factions is None:
            factions = torch.zeros((2,) if shared else (n, 2), dtype=torch.uint8, device=self.device)
        factions = self._dev(factions, torch.uint8)
        assert (factions.dim() == 1) == bool(shared)
        states = out if out is not None else self.empty_states(n)
        self._check(self.lib.sb_reset(self.h, n, self._p(seeds), self._p(decks), n_deck, shared, self._p(factions),
                                      self._p(states), self._stream()), "sb_reset")
        return states

    def generate_decks(self, seeds, generation, mode, n_preserve=0, q=0.0, archetypes=None, arch_factions=None, factions=None):
        """sb_generate_decks: per-game deck pairs of DeckEvolutionConfig.get_deck_configuration (utils.py:121-241).
        Returns (decks u8[n,2,12], factions u8[n,2]) on the device, ready for reset()."""
        seeds = torch.as_tensor(np.asarray(seeds, dtype=np.int64) if not torch.is_tensor(seeds) else seeds).to(self.device, torch.int64).contiguous()
        n = seeds.numel()
        arch = None if archetypes is None else np.ascontiguousarray(np.asarray(archetypes, dtype=np.uint8).reshape(24))
        af = None if arch_factions is None else np.ascontiguousarray(np.asarray(arch_factions, dtype=np.uint8).reshape(2))
        if factions is not None:
            factions = torch.as_tensor(factions).to(self.device, torch.uint8).contiguous()
            assert factions.shape == (n, 2)
        decks = torch.empty((n, 2, 12), dtype=torch.uint8, device=self.device)
        fout = torch.empty((n, 2), dtype=torch.uint8, device=self.device)
        self._check(self.lib.sb_generate_decks(self.h, n, self._p(seeds), int(generation), int(mode), int(n_preserve), float(q),
                                               None if arch is None else arch.ctypes.data, None if af is None else af.ctypes.data,
                                               self._p(factions), self._p(decks), self._p(fout), self._stream()), "sb_generate_decks")
        return decks, fout

    # ---- evolution-strategy operators on a resident population (include/sb_b200.h, sb_es_*)
    def es_offspring(self, seed, generation, mu, lam, tau, tau_prime, min_sigma, w, s, parents=None):
        assert w.shape == s.shape and w.shape[0] >= mu + lam and w.dtype == torch.float64 and w.is_contiguous() and s.is_contiguous()
        self._check(self.lib.sb_es_offspring(self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(generation), mu, lam, w.shape[1], float(tau),
                                             float(tau_prime), float(min_sigma), self._p(w), self._p(s), self._p(parents), self._stream()),
                    "sb_es_offspring")

    def es_select(self, mu, fitness, w, s, want_order=False):
        total, nf = w.shape
        fitness = torch.as_tensor(fitness, dtype=torch.float64).to(self.device).contiguous()
        assert fitness.numel() == total
        wo = torch.empty((mu, nf), dtype=torch.float64, device=self.device)
        so = torch.empty_like(wo)
        fo = torch.empty(mu, dtype=torch.float64, device=self.device)
        order = torch.empty(mu, dtype=torch.int32, device=self.device) if want_order else None
        self._check(self.lib.sb_es_select(self.h, total, mu, nf, self._p(fitness), self._p(w), self._p(s), self._p(wo), self._p(so),
                                          self._p(fo), self._p(order), self._stream()), "sb_es_select")
        return wo, so, fo, order

    def es_reset_sigmas(self, seed, generation, initial_sigma, s):
        self._check(self.lib.sb_es_reset_sigmas(self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(generation), s.shape[0], s.shape[1],
                                                float(initial_sigma), self._p(s), self._stream()), "sb_es_reset_sigmas")

    def es_inject_diversity(self, seed, generation, tau, tau_prime, min_sigma, initial_sigma, w, s, chosen=None):
        self._check(self.lib.sb_es_inject_diversity(self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(generation), w.shape[0], w.shape[1], float(tau),
                                                    float(tau_prime), float(min_sigma), float(initial_sigma), self._p(w), self._p(s),
                                                    self._p(chosen), self._stream()), "sb_es_inject_diversity")

    def legal_mask(self, states, out=None):
        n = states.shape[0]
        masks = out if out is not None else torch.empty((n, MASK_WORDS), dtype=torch.int32, device=self.device)
        self._check(self.lib.sb_legal_mask(self.h, n, self._p(states), self._p(masks), self._stream()), "sb_legal_mask")
        return masks

    def step(self, states, actions, reward=None, done=None, err=None, next_masks=None):
        n = states.shape[0]
        actions = self._dev(actions, torch.uint8)
        reward = reward if reward is not None else torch.empty(n, dtype=torch.int8, device=self.device)
        done = done if done is not None else torch.empty(n, dtype=torch.uint8, device=self.device)
        err = err if err is not None else torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(self.lib.sb_step(self.h, n, self._p(states), self._p(actions), self._p(reward), self._p(done),
                                     self._p(err), self._p(next_masks), self._stream()), "sb_step")
        return reward, done, err

    def observe(self, states):
        n = states.shape[0]
        obs = torch.empty((n, 27, 5, 4), dtype=torch.int32, device=self.device)
        err = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(self.lib.sb_observe(self.h, n, self._p(states), self._p(obs), self._p(err), self._stream()), "sb_observe")
        return obs, err

    def features(self, states):
        n = states.shape[0]
        f = torch.empty((n, 10), dtype=torch.float64, device=self.device)
        err = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(self.lib.sb_features(self.h, n, self._p(states), self._p(f), self._p(err), self._stream()), "sb_features")
        return f, err

    def select_action(self, states, weights, want_scores=False):
        n = states.shape[0]
        weights = self._dev(weights, torch.float64)
        assert weights.shape == (n, 10)
        actions = torch.empty(n, dtype=torch.uint8, device=self.device)
        scores = torch.empty((n, N_ACTIONS), dtype=torch.float64, device=self.device) if want_scores else None
        self._check(self.lib.sb_select_action(self.h, n, self._p(states), self._p(weights), self._p(actions),
                                              self._p(scores), self._stream()), "sb_select_action")
        return actions, scores

    def expert_action(self, states):
        """Stormbound.expert_action per game; advances each state's random-stream draw counter in place."""
        n = states.shape[0]
        actions = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(self.lib.sb_expert_action(self.h, n, self._p(states), self._p(actions), self._stream()), "sb_expert_action")
        return actions

    def rollout_random(self, states, max_steps=400, chain=None):
        n = states.shape[0]
        steps = torch.empty(n, dtype=torch.int32, device=self.device)
        self._check(self.lib.sb_rollout_random(self.h, n, self._p(states), max_steps, self._p(steps), self._p(chain),
                                               self._stream()), "sb_rollout_random")
        return steps

    def rollout_heuristic(self, states, w_first, w_second, idx_first=None, idx_second=None, max_steps=400):
        """Whole heuristic games; w_first / w_second = None hands that seat to the scripted expert opponent."""
        n = states.shape[0]
        if w_first is None and w_second is None:
            raise ValueError("at least one seat needs a weight table (expert-vs-expert games: expert_action + step)")
        w_first = None if w_first is None else self._dev(w_first, torch.float64)
        w_second = None if w_second is None else self._dev(w_second, torch.float64)
        for w, idx in ((w_first, idx_first), (w_second, idx_second)):  # the kernels index these tables unchecked
            if w is not None:
                assert w.dim() == 2 and w.shape[1] == 10, "weight tables are f64[P, 10] (SB_N_FEATURES)"
                if idx is None:
                    assert w.shape[0] >= n
                else:
                    self._dev(idx, torch.int32)
                    assert idx.numel() == n
        result = torch.empty(n, dtype=torch.int8, device=self.device)
        steps = torch.empty(n, dtype=torch.int32, device=self.device)
        self._check(self.lib.sb_rollout_heuristic(self.h, n, self._p(states), self._p(w_first), self._p(w_second),
                                                  self._p(idx_first), self._p(idx_second), max_steps, self._p(result),
                                                  self._p(steps), self._stream()), "sb_rollout_heuristic")
        return result, steps

    # ---- batched auto-resetting environment (sb_env_reset / sb_env_step)
    def _env_args(self, n, decks, factions, opponent, seat, w_opp, idx_opp):
        if decks is None:
            decks, factions = self._default_deck_tensors()
        decks = self._dev(decks, torch.uint8)
        shared = 1 if decks.dim() == 2 else 0
        if factions is None:
            factions = torch.zeros((2,) if shared else (n, 2), dtype=torch.uint8, device=self.device)
        assert decks.shape[-2] == 2 and (shared or decks.shape[0] == n), "decks are u8[2,k] (shared) or u8[n,2,k]"
        factions = self._dev(factions, torch.uint8)
        assert factions.shape == ((2,) if shared else (n, 2)), "factions are u8[2] with shared decks, else u8[n,2]"
        if seat is not None:
            self._dev(seat, torch.uint8)
            assert seat.numel() == n
        if w_opp is not None:  # the kernel indexes the table unchecked
            self._dev(w_opp, torch.float64)
            assert w_opp.dim() == 2 and w_opp.shape[1] == 10, "weight tables are f64[P, 10] (SB_N_FEATURES)"
            if idx_opp is None:
                assert w_opp.shape[0] >= n
            else:
                self._dev(idx_opp, torch.int32)
                assert idx_opp.numel() == n
        return decks, decks.shape[-1], shared, factions

    def _default_deck_tensors(self):
        if self._default_decks is None:
            self._default_decks = (torch.tensor([deck_indices(d) for d in DEFAULT_DECKS], dtype=torch.uint8, device=self.device),
                                   torch.tensor(DEFAULT_FACTIONS, dtype=torch.uint8, device=self.device))
        return self._default_decks

    def _env_outputs(self, n, out, names):
        out = dict(out or {})
        shapes = {"states": ((n, STATE_BYTES), torch.uint8), "obs": ((n, 27, 5, 4), torch.int32), "masks": ((n, MASK_WORDS), torch.int32),
                  "obs_err": ((n,), torch.uint8), "result": ((n,), torch.int8), "length": ((n,), torch.int32),
                  "final_states": ((n, STATE_BYTES), torch.uint8)}
        for k in names:
            shape, dtype = shapes[k]
            if k not in out:
                out[k] = torch.empty(shape, dtype=dtype, device=self.device)
            elif out[k] is not None:
                self._dev(out[k], dtype)
                assert tuple(out[k].shape) == shape, (k, tuple(out[k].shape), shape)
        return out

    def env_reset(self, seeds, opponent=0, seat=None, w_opp=None, idx_opp=None, max_steps=400, decks=None, factions=None, out=None):
        """sb_env_reset: deal games from seeds i64[n] and let the opponent (0 none, 1 random, 2 expert, 3 heuristic with
        w_opp f64[P,10] / idx_opp i32[n]) play until the learner (seat u8[n], 0 FIRST / 1 SECOND) is to move.
        out: dict of preallocated buffers (states, obs, masks, obs_err; None skips a nullable output).  Returns that dict."""
        seeds = self._dev(seeds, torch.int64)
        n = seeds.numel()
        decks, n_deck, shared, factions = self._env_args(n, decks, factions, opponent, seat, w_opp, idx_opp)
        o = self._env_outputs(n, out, ("states", "obs", "masks", "obs_err"))
        self._check(self.lib.sb_env_reset(self.h, n, self._p(seeds), self._p(decks), n_deck, shared, self._p(factions), int(opponent),
                                          self._p(seat), self._p(w_opp), self._p(idx_opp), int(max_steps), self._p(o["states"]),
                                          self._p(o["obs"]), self._p(o["masks"]), self._p(o["obs_err"]), self._stream()), "sb_env_reset")
        return o

    def env_step(self, states, actions, opponent=0, seat=None, w_opp=None, idx_opp=None, max_steps=400, decks=None, factions=None,
                 out=None):
        """sb_env_step on states u8[n,512] in place with actions u8[n]: check, apply, opponent, auto-reset, observe.
        out: dict of preallocated buffers (result, length, final_states, obs, masks, obs_err; None skips a nullable output).
        Returns that dict."""
        states = self._dev(states, torch.uint8)
        assert states.dim() == 2 and states.shape[1] == STATE_BYTES, "states are u8[n, 512]"
        n = states.shape[0]
        actions = self._dev(actions, torch.uint8)
        assert actions.numel() == n
        decks, n_deck, shared, factions = self._env_args(n, decks, factions, opponent, seat, w_opp, idx_opp)
        o = self._env_outputs(n, out, ("result", "length", "final_states", "obs", "masks", "obs_err"))
        self._check(self.lib.sb_env_step(self.h, n, self._p(states), self._p(actions), self._p(decks), n_deck, shared, self._p(factions),
                                         int(opponent), self._p(seat), self._p(w_opp), self._p(idx_opp), int(max_steps), self._p(o["result"]),
                                         self._p(o["length"]), self._p(o["final_states"]), self._p(o["obs"]), self._p(o["masks"]),
                                         self._p(o["obs_err"]), self._stream()), "sb_env_step")
        return o

    # ---- batched tree search (sb_search_begin / sb_search_simulate / sb_search_end)
    def search_workspace_bytes(self, n, max_nodes):
        return search_workspace_bytes(n, max_nodes)

    def _search_outputs(self, n, out, names):
        out = dict(out or {})
        shapes = {"states": ((n, STATE_BYTES), torch.uint8), "obs": ((n, 27, 5, 4), torch.int32), "masks": ((n, MASK_WORDS), torch.int32),
                  "obs_err": ((n,), torch.uint8), "to_move": ((n,), torch.uint8), "kind": ((n,), torch.uint8),
                  "visits": ((n, N_ACTIONS), torch.int32), "q": ((n, N_ACTIONS), torch.float64), "root_value": ((n,), torch.float64),
                  "action": ((n,), torch.int32), "policy": ((n, N_ACTIONS), torch.float32)}
        for k in names:
            shape, dtype = shapes[k]
            if k not in out:
                out[k] = torch.empty(shape, dtype=dtype, device=self.device)
            elif out[k] is not None:
                self._dev(out[k], dtype)
                assert tuple(out[k].shape) == shape, (k, tuple(out[k].shape), shape)
        return out

    def _search_eval(self, n, prior, value):
        self._dev(prior, torch.float32)
        self._dev(value, torch.float32)
        assert tuple(prior.shape) == (n, N_ACTIONS) and tuple(value.shape) == (n,), "prior is f32[n,156], value f32[n]"

    def search_begin(self, ws, roots, max_nodes, max_steps=400, out=None):
        """sb_search_begin: root records u8[n,512] -> node 0 of n trees in the workspace ws (u8 tensor of at least
        search_workspace_bytes(n, max_nodes) bytes).  out: dict of preallocated leaf buffers (states, obs, masks, obs_err,
        to_move, kind; None skips a nullable output).  Returns that dict: the roots as the first leaves to evaluate."""
        self._dev(ws, torch.uint8)
        roots = self._dev(roots, torch.uint8)
        assert roots.dim() == 2 and roots.shape[1] == STATE_BYTES, "roots are u8[n, 512]"
        n = roots.shape[0]
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_search_begin(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(roots), int(max_steps),
                                             self._p(o["states"]), self._p(o["obs"]), self._p(o["masks"]), self._p(o["obs_err"]),
                                             self._p(o["to_move"]), self._p(o["kind"]), self._stream()), "sb_search_begin")
        return o

    def search_simulate(self, ws, n, max_nodes, prior, value, c_puct=1.25, fpu=0.0, out=None):
        """sb_search_simulate: back up the pending leaves with prior f32[n,156] / value f32[n] (the seat to move's view), then
        select, expand and emit the next leaves into out (as search_begin).  Returns that dict."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_search_simulate(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                                float(c_puct), float(fpu), self._p(o["states"]), self._p(o["obs"]), self._p(o["masks"]),
                                                self._p(o["obs_err"]), self._p(o["to_move"]), self._p(o["kind"]), self._stream()),
                    "sb_search_simulate")
        return o

    def search_end(self, ws, n, max_nodes, prior, value, out=None):
        """sb_search_end: back up the last pending leaves, then read out the roots into out: visits i32[n,156], q f64[n,156]
        (NaN where unvisited) and root_value f64[n], both for the seat to move at the root.  Returns that dict."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        o = self._search_outputs(n, out, ("visits", "q", "root_value"))
        self._check(self.lib.sb_search_end(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                           self._p(o["visits"]), self._p(o["q"]), self._p(o["root_value"]), self._stream()), "sb_search_end")
        return o

    # ---- information-set tree search (sb_ismcts_begin / sb_ismcts_simulate / sb_ismcts_end)
    def ismcts_workspace_bytes(self, n, max_nodes):
        return ismcts_workspace_bytes(n, max_nodes)

    def _worlds(self, det):
        det = self._dev(det, torch.uint8)
        assert det.dim() == 2 and det.shape[1] == STATE_BYTES, "worlds are u8[n, 512]"
        return det

    def ismcts_begin(self, ws, det, max_nodes, max_steps=400, out=None):
        """sb_ismcts_begin: node 0 of n information-set trees in ws (u8 tensor of at least ismcts_workspace_bytes(n, max_nodes)
        bytes) from det u8[n,512], the first world of each root (a determinization of it for its own local_order).  out: dict
        of preallocated leaf buffers (as search_begin).  Returns that dict: the worlds' roots as the first leaves."""
        self._dev(ws, torch.uint8)
        det = self._worlds(det)
        n = det.shape[0]
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_ismcts_begin(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(det), int(max_steps),
                                             self._p(o["states"]), self._p(o["obs"]), self._p(o["masks"]), self._p(o["obs_err"]),
                                             self._p(o["to_move"]), self._p(o["kind"]), self._stream()), "sb_ismcts_begin")
        return o

    def ismcts_simulate(self, ws, det, max_nodes, prior, value, c_puct=1.25, fpu=0.0, out=None):
        """sb_ismcts_simulate: back up the pending leaves with prior f32[n,156] / value f32[n] (the seat to move's view), then
        walk each tree through this call's world det u8[n,512] and emit the next leaves into out (as search_begin)."""
        self._dev(ws, torch.uint8)
        det = self._worlds(det)
        n = det.shape[0]
        self._search_eval(n, prior, value)
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_ismcts_simulate(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(det), self._p(prior),
                                                self._p(value), float(c_puct), float(fpu), self._p(o["states"]), self._p(o["obs"]),
                                                self._p(o["masks"]), self._p(o["obs_err"]), self._p(o["to_move"]), self._p(o["kind"]),
                                                self._stream()), "sb_ismcts_simulate")
        return o

    def ismcts_end(self, ws, n, max_nodes, prior, value, out=None):
        """sb_ismcts_end: back up the last pending leaves, then read out the roots by their action ids into out: visits
        i32[n,156], q f64[n,156] (NaN where unvisited or not the representative of its move code) and root_value f64[n]."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        o = self._search_outputs(n, out, ("visits", "q", "root_value"))
        self._check(self.lib.sb_ismcts_end(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                           self._p(o["visits"]), self._p(o["q"]), self._p(o["root_value"]), self._stream()), "sb_ismcts_end")
        return o

    # ---- Gumbel search over both trees (sb_search_simulate_gumbel / sb_search_end_gumbel, sb_ismcts_*_gumbel)
    def _gumbel(self, n, gumbel):
        self._dev(gumbel, torch.float32)
        assert tuple(gumbel.shape) == (n, N_ACTIONS), "gumbel is f32[n,156]"

    def search_simulate_gumbel(self, ws, n, max_nodes, prior, value, gumbel, sim, num_simulations, max_considered=16,
                               c_visit=50.0, c_scale=0.1, out=None):
        """sb_search_simulate_gumbel: as search_simulate, selecting with the Gumbel rule (DESIGN.md 8.9): call sim = 1..S of
        a search of num_simulations = S calls, gumbel f32[n,156] the search's Gumbel noise (the same for every call)."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        self._gumbel(n, gumbel)
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_search_simulate_gumbel(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                                       self._p(gumbel), int(sim), int(num_simulations), int(max_considered), float(c_visit),
                                                       float(c_scale), self._p(o["states"]), self._p(o["obs"]), self._p(o["masks"]),
                                                       self._p(o["obs_err"]), self._p(o["to_move"]), self._p(o["kind"]), self._stream()),
                    "sb_search_simulate_gumbel")
        return o

    def search_end_gumbel(self, ws, n, max_nodes, prior, value, gumbel, c_visit=50.0, c_scale=0.1, out=None):
        """sb_search_end_gumbel: search_end's read-out plus action i32[n] (255 without root visits) and the improved policy
        f32[n,156] (0 outside the legal set).  Returns the dict (action, policy, visits, q, root_value)."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        self._gumbel(n, gumbel)
        o = self._search_outputs(n, out, ("action", "policy", "visits", "q", "root_value"))
        self._check(self.lib.sb_search_end_gumbel(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                                  self._p(gumbel), float(c_visit), float(c_scale), self._p(o["action"]), self._p(o["policy"]),
                                                  self._p(o["visits"]), self._p(o["q"]), self._p(o["root_value"]), self._stream()),
                    "sb_search_end_gumbel")
        return o

    def ismcts_simulate_gumbel(self, ws, det, max_nodes, prior, value, gumbel, sim, num_simulations, max_considered=16,
                               c_visit=50.0, c_scale=0.1, out=None):
        """sb_ismcts_simulate_gumbel: as ismcts_simulate (this call's world det u8[n,512]), selecting with the Gumbel rule."""
        self._dev(ws, torch.uint8)
        det = self._worlds(det)
        n = det.shape[0]
        self._search_eval(n, prior, value)
        self._gumbel(n, gumbel)
        o = self._search_outputs(n, out, ("states", "obs", "masks", "obs_err", "to_move", "kind"))
        self._check(self.lib.sb_ismcts_simulate_gumbel(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(det), self._p(prior),
                                                       self._p(value), self._p(gumbel), int(sim), int(num_simulations), int(max_considered),
                                                       float(c_visit), float(c_scale), self._p(o["states"]), self._p(o["obs"]),
                                                       self._p(o["masks"]), self._p(o["obs_err"]), self._p(o["to_move"]), self._p(o["kind"]),
                                                       self._stream()), "sb_ismcts_simulate_gumbel")
        return o

    def ismcts_end_gumbel(self, ws, n, max_nodes, prior, value, gumbel, c_visit=50.0, c_scale=0.1, out=None):
        """sb_ismcts_end_gumbel: ismcts_end's read-out plus action i32[n] and the improved policy f32[n,156], by the root's
        action ids (an id that repeats a lower id's card reads 0)."""
        self._dev(ws, torch.uint8)
        self._search_eval(n, prior, value)
        self._gumbel(n, gumbel)
        o = self._search_outputs(n, out, ("action", "policy", "visits", "q", "root_value"))
        self._check(self.lib.sb_ismcts_end_gumbel(self.h, n, int(max_nodes), self._p(ws), ws.numel(), self._p(prior), self._p(value),
                                                  self._p(gumbel), float(c_visit), float(c_scale), self._p(o["action"]), self._p(o["policy"]),
                                                  self._p(o["visits"]), self._p(o["q"]), self._p(o["root_value"]), self._stream()),
                    "sb_ismcts_end_gumbel")
        return o

    # ---- determinization for sampled search (sb_determinize)
    def determinize(self, states, keys, observer=None, out=None):
        """sb_determinize: states u8[n,512] with what the observer cannot see resampled (the other seat's hand / deck
        assignment of its cards, and the Philox key <- keys i64[n]); observer u8[n] or None (each record's local_order,
        non-zero = SECOND).  out: u8[n,512] (a new tensor when None; may be states itself).  Returns out."""
        states = self._dev(states, torch.uint8)
        assert states.dim() == 2 and states.shape[1] == STATE_BYTES, "states are u8[n, 512]"
        n = states.shape[0]
        keys = self._dev(keys.view(torch.int64) if keys.dtype == torch.uint64 else keys, torch.int64)
        assert tuple(keys.shape) == (n,), "keys are i64[n]"
        if observer is not None:
            observer = self._dev(observer, torch.uint8)
            assert tuple(observer.shape) == (n,), "observer is u8[n]"
        out = out if out is not None else self.empty_states(n)
        self._dev(out, torch.uint8)
        assert tuple(out.shape) == (n, STATE_BYTES), "out is u8[n, 512]"
        self._check(self.lib.sb_determinize(self.h, n, self._p(states), self._p(observer), self._p(keys), self._p(out),
                                            self._stream()), "sb_determinize")
        return out

    def accumulate_fitness(self, result, idx_first, counts):
        n = result.shape[0]
        self._check(self.lib.sb_accumulate_fitness(self.h, n, self._p(result), self._p(idx_first), self._p(counts),
                                                   self._stream()), "sb_accumulate_fitness")
        return counts

    def count_aborted(self, states, result, out=None):
        """i32[2] += {aborted like the reference would (err 1..4), aborted by a limit of this engine (err 5..7)}"""
        out = out if out is not None else torch.zeros(2, dtype=torch.int32, device=self.device)
        self._check(self.lib.sb_count_aborted(self.h, result.shape[0], self._p(states), self._p(result), self._p(out), self._stream()),
                    "sb_count_aborted")
        return out

    SCHEDULES = {"round_robin": 0, "versus": 1, "solo": 2}

    def eval_schedule(self, mode, n_ind, n_total, games_per_pair, base_seed, generation, game_lo, n):
        """sb_eval_schedule: (idx_first i32[n], idx_second i32[n], seeds i64[n]) of the games game_lo .. game_lo + n - 1"""
        i1 = torch.empty(n, dtype=torch.int32, device=self.device)
        i2 = torch.empty(n, dtype=torch.int32, device=self.device)
        seeds = torch.empty(n, dtype=torch.int64, device=self.device)
        self._check(self.lib.sb_eval_schedule(self.h, self.SCHEDULES[mode], n_ind, n_total, games_per_pair, int(base_seed) & 0xFFFFFFFFFFFFFFFF,
                                              int(generation), int(game_lo), n, self._p(i1), self._p(i2), self._p(seeds), self._stream()),
                    "sb_eval_schedule")
        return i1, i2, seeds

    def eval_population(self, mode, n_ind, weights, games_per_pair, base_seed, generation, game_lo, game_hi, max_steps=400,
                        counts=None, aborted=None, chunk_games=0, decks=None, factions=None):
        """sb_eval_population: counts i32[n_ind,3] += {wins, draws, losses}, aborted i32[2] += ...; asynchronous.  Every game is
        dealt the same deck pair: decks u8[2, n_deck] with factions u8[2], or the default decks when decks is None."""
        weights = self._dev(weights, torch.float64)
        assert weights.dim() == 2 and weights.shape[1] == 10 and weights.shape[0] >= n_ind, "weight tables are f64[P, 10] (SB_N_FEATURES)"
        if decks is None:
            assert factions is None, "factions go with decks"
            if self._default_decks is None:
                self._default_decks = (torch.tensor([deck_indices(d) for d in DEFAULT_DECKS], dtype=torch.uint8, device=self.device),
                                       torch.tensor(DEFAULT_FACTIONS, dtype=torch.uint8, device=self.device))
            decks, factions = self._default_decks
        decks, factions = self._dev(decks, torch.uint8), self._dev(factions, torch.uint8)
        assert decks.dim() == 2 and decks.shape[0] == 2 and tuple(factions.shape) == (2,), "one deck pair u8[2, n_deck], factions u8[2]"
        counts = counts if counts is not None else torch.zeros((n_ind, 3), dtype=torch.int32, device=self.device)
        aborted = aborted if aborted is not None else torch.zeros(2, dtype=torch.int32, device=self.device)
        self._dev(counts, torch.int32)
        assert counts.numel() >= 3 * n_ind
        self._check(self.lib.sb_eval_population(self.h, self.SCHEDULES[mode], n_ind, weights.shape[0], games_per_pair,
                                                int(base_seed) & 0xFFFFFFFFFFFFFFFF, int(generation), int(game_lo), int(game_hi), self._p(weights),
                                                self._p(decks), decks.shape[-1], self._p(factions), max_steps, int(chunk_games), self._p(counts),
                                                self._p(aborted), self._stream()), "sb_eval_population")
        return counts, aborted

    # ------------------------------------------------------------------ host-buffer (e2e) entry points
    def step_host(self, states_np, actions_np, want_masks=True):
        """numpy in, numpy out; H2D + kernel + D2H inside the call (sb_step_host)."""
        n = states_np.shape[0]
        reward = np.empty(n, dtype=np.int8)
        done = np.empty(n, dtype=np.uint8)
        err = np.empty(n, dtype=np.uint8)
        masks = np.empty((n, MASK_WORDS), dtype=np.uint32) if want_masks else None
        self._check(self.lib.sb_step_host(self.h, n, states_np.ctypes.data, actions_np.ctypes.data, reward.ctypes.data,
                                          done.ctypes.data, err.ctypes.data, masks.ctypes.data if want_masks else None),
                    "sb_step_host")
        return reward, done, err, masks

    def rollout_random_host(self, seeds_np, decks_np=None, factions_np=None, max_steps=400, want_states=True, want_chain=False,
                            out_states=None, out_steps=None):
        """Host-buffer variant (sb_rollout_random_host).  out_states / out_steps: caller-owned result buffers, e.g. pinned."""
        n = seeds_np.shape[0]
        if decks_np is None:
            decks_np = np.array([deck_indices(d) for d in DEFAULT_DECKS], dtype=np.uint8)
            factions_np = np.array(DEFAULT_FACTIONS, dtype=np.uint8)
        seeds_np = np.ascontiguousarray(seeds_np, dtype=np.uint64)
        states = (out_states if out_states is not None else np.empty((n, STATE_BYTES), dtype=np.uint8)) if want_states else None
        steps = out_steps if out_steps is not None else np.empty(n, dtype=np.int32)
        assert steps.dtype == np.int32 and steps.shape == (n,) and (states is None or (states.dtype == np.uint8 and states.shape == (n, STATE_BYTES)))
        chain = np.zeros(n, dtype=np.uint64) if want_chain else None
        self._check(self.lib.sb_rollout_random_host(self.h, n, seeds_np.ctypes.data, decks_np.ctypes.data, decks_np.shape[-1],
                                                    factions_np.ctypes.data, max_steps,
                                                    states.ctypes.data if want_states else None, steps.ctypes.data,
                                                    chain.ctypes.data if want_chain else None), "sb_rollout_random_host")
        return states, steps, chain


def search_workspace_bytes(n, max_nodes):
    """sb_search_workspace_bytes: bytes of the search workspace of n trees of max_nodes nodes (host only, no GPU needed)."""
    b = int(_lib.load().sb_search_workspace_bytes(int(n), int(max_nodes)))
    if n < 0 or max_nodes < 1 or (n > 0 and b == 0):
        raise ValueError("no search workspace for n=%d, max_nodes=%d (n >= 0, max_nodes 1..2^24)" % (n, max_nodes))
    return b


def ismcts_workspace_bytes(n, max_nodes):
    """sb_ismcts_workspace_bytes: bytes of the information-set search workspace of n trees of max_nodes nodes (host only)."""
    b = int(_lib.load().sb_ismcts_workspace_bytes(int(n), int(max_nodes)))
    if n < 0 or max_nodes < 1 or (n > 0 and b == 0):
        raise ValueError("no ISMCTS workspace for n=%d, max_nodes=%d (n >= 0, max_nodes 1..2^24)" % (n, max_nodes))
    return b


_engines = {}


def get_engine(device=None):
    """One engine per device; None = the caller's current CUDA device (LOCAL_RANK under torchrun once the launcher has
    called torch.cuda.set_device), never a hard-wired device 0."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        lr = os.environ.get("LOCAL_RANK")
        if device == 0 and lr is not None and torch.cuda.is_available():  # torchrun rank that never called set_device
            device = int(lr) % torch.cuda.device_count()
    if isinstance(device, torch.device):
        device = device.index or 0
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
