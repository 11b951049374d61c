"""GPU-resident replay memory: the reference's ``src/replaybuffer.py`` for a whole population at once.

``ReplayRings`` holds one ring per agent (ring id = m*P + p) in a single HBM tensor
``data[capacity, M, P, 10]``; the fused environment step writes slot ``ring_count % capacity`` of every
ring in one sweep, ``sample_indices`` draws ``batch`` uniform indices per ring with Philox (bit-exact vs
oracle/philox_np.py) and ``gather`` pulls the 40-byte records.  ``ReplayBuffer`` is the per-agent drop-in
with the reference's constructor and ``add`` / ``sample`` / ``buffer_counter`` surface
(replaybuffer.py:5-63).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .environment import DeviceClock


class ReplayRings:
    def __init__(self, capacity: int, M: int, P: int, batch_size: int = 64, *, seed: int = 1, ring_id_base: int = 0,
                 clock: Optional[DeviceClock] = None, device=None, runs=None):
        """runs: an environment.RunTable; ring m*P + p is then keyed like ring m*Pr + p mod Pr of run p // Pr (seed and
        ring_id_base are unused)."""
        if capacity <= 0 or batch_size <= 0 or batch_size % 4:
            raise ValueError("capacity must be > 0 and batch_size a positive multiple of 4")
        self.lib = _lib.load()
        _lib.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.capacity, self.M, self.P, self.batch_size = int(capacity), int(M), int(P), int(batch_size)
        self.n_rings = self.M * self.P
        self.seed, self.ring_id_base = int(seed), int(ring_id_base)
        if runs is not None and (runs.P != self.P or self.ring_id_base != 0):
            raise ValueError(f"a run table of {runs.S} x {runs.Pr} platoons needs P = {runs.P} and ring_id_base = 0")
        self.runs = runs
        self.data = torch.empty(self.capacity, self.M, self.P, _lib.RING_RECORD_FLOATS, dtype=torch.float32, device=self.device)
        self.clock = clock if clock is not None else DeviceClock(self.device)
        self.idx = self.s = self.a = self.r = self.s2 = None      # sample buffers: allocated on first use

    def _alloc_sample_buffers(self):
        if self.idx is None:
            n = self.n_rings * self.batch_size
            self.idx = torch.zeros(self.n_rings, self.batch_size, dtype=torch.int64, device=self.device)
            self.s = torch.zeros(n, 4, dtype=torch.float32, device=self.device)
            self.a = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.r = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.s2 = torch.zeros(n, 4, dtype=torch.float32, device=self.device)

    def add(self, s, a, r, s2, advance_clock=True):
        """Stand-alone ReplayBuffer.add for all rings: s, s2 [4][M][P]; a, r [M][P] (native layout)."""
        _lib.check(self.lib.avd_replay_add(_lib.ptr(self.data), self.capacity, self.M, self.P, self.clock.ptr, _lib.ptr(s),
                                           _lib.ptr(a), _lib.ptr(r), _lib.ptr(s2), _lib.current_stream()))
        if advance_clock:
            self.clock.advance(ring=1)

    def fill_synthetic(self, seed=12345):
        _lib.check(self.lib.avd_replay_fill_synthetic(_lib.ptr(self.data), self.capacity, self.M, self.P, seed,
                                                      _lib.current_stream()))
        self.clock.set(ring_count=self.capacity)

    def sample_indices(self):
        self._alloc_sample_buffers()
        if self.runs is not None:
            _lib.check(self.lib.avd_replay_sample_indices_runs(_lib.ptr(self.idx), self.n_rings, self.batch_size, self.capacity, self.runs.ptr,
                                                               self.clock.ptr, _lib.current_stream()))
            return self.idx
        _lib.check(self.lib.avd_replay_sample_indices(_lib.ptr(self.idx), self.n_rings, self.ring_id_base, self.batch_size,
                                                      self.capacity, self.seed, self.clock.ptr, _lib.current_stream()))
        return self.idx

    def gather(self, idx=None):
        self._alloc_sample_buffers()
        idx = self.idx if idx is None else idx
        _lib.check(self.lib.avd_replay_gather(_lib.ptr(self.data), self.capacity, self.M, self.P, _lib.ptr(idx),
                                              self.batch_size, _lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.r),
                                              _lib.ptr(self.s2), _lib.current_stream()))
        return self.s, self.a, self.r, self.s2

    def sample(self, advance_clock=True, keep_indices=False):
        """ReplayBuffer.sample for every ring in one launch (avd_replay_sample: index draw + gathers fused, identical to
        sample_indices() + gather()); keep_indices also writes the draws to self.idx."""
        self._alloc_sample_buffers()
        idx = _lib.ptr(self.idx) if keep_indices else None
        if self.runs is not None:
            _lib.check(self.lib.avd_replay_sample_runs(_lib.ptr(self.data), self.capacity, self.M, self.P, self.batch_size, self.runs.ptr,
                                                       self.clock.ptr, idx, _lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.r),
                                                       _lib.ptr(self.s2), _lib.current_stream()))
        else:
            _lib.check(self.lib.avd_replay_sample(_lib.ptr(self.data), self.capacity, self.M, self.P, self.ring_id_base, self.batch_size,
                                                  self.seed, self.clock.ptr, idx, _lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.r),
                                                  _lib.ptr(self.s2), _lib.current_stream()))
        if advance_clock:
            self.clock.advance(update=1)
        return self.s, self.a, self.r, self.s2


class ReplayBuffer:
    """Per-agent drop-in (one ring).  Returns CUDA float32 tensors where the reference returns TF tensors."""

    def __init__(self, buffer_capacity=100000, batch_size=64, num_states=None, num_actions=None, platoon_size=None, *,
                 seed: int = 1, ring_id: int = 0):
        if num_states is None or num_states > 4 or (num_actions or 1) != 1:
            raise NotImplementedError("rings hold up to 4 state words and 1 action per agent (decentralized framework)")
        self.buffer_capacity, self.batch_size = buffer_capacity, batch_size
        self.num_states, self.num_actions = num_states, num_actions or 1
        self.buffer_counter = 0
        self._rings = ReplayRings(buffer_capacity, 1, 1, batch_size, seed=seed, ring_id_base=ring_id)
        dev = self._rings.device
        self._s = torch.zeros(4, 1, 1, device=dev)
        self._s2 = torch.zeros(4, 1, 1, device=dev)
        self._a = torch.zeros(1, 1, device=dev)
        self._r = torch.zeros(1, 1, device=dev)

    def add(self, obs_tuple):
        s, a, r, s2 = obs_tuple
        ns = self.num_states
        self._s.zero_(); self._s2.zero_()
        self._s[:ns, 0, 0] = torch.as_tensor(np.asarray(s, dtype=np.float32).reshape(-1)[:ns])
        self._s2[:ns, 0, 0] = torch.as_tensor(np.asarray(s2, dtype=np.float32).reshape(-1)[:ns])
        self._a[0, 0] = float(np.asarray(a).reshape(-1)[0])
        self._r[0, 0] = float(np.asarray(r).reshape(-1)[0])
        self._rings.add(self._s, self._a, self._r, self._s2)
        self.buffer_counter += 1

    def sample(self, indices=None):
        """(state, action, reward, next_state) batches.  ``indices`` injects the reference's draw
        (np.random.choice) for parity runs; otherwise Philox indices are drawn on the device."""
        if self.buffer_counter == 0:
            raise ValueError("a must be greater than 0 unless no samples are taken")   # np.random.choice(0, n)
        if indices is None:
            self._rings.sample_indices()
            self._rings.clock.advance(update=1)
            idx = None
        else:
            idx = torch.as_tensor(np.asarray(indices, dtype=np.int64).reshape(1, -1), device=self._rings.device)
            if idx.shape[1] != self.batch_size or int(idx.max()) >= min(self.buffer_counter, self.buffer_capacity) or int(idx.min()) < 0:
                raise ValueError("injected indices out of range")
        s, a, r, s2 = self._rings.gather(idx)
        ns = self.num_states
        return s[:, :ns].clone(), a.reshape(-1, 1).clone(), r.reshape(-1, 1).clone(), s2[:, :ns].clone()
