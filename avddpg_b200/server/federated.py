"""Federated averaging -- the reference's ``src/server/federated.py`` + the FRL glue of
``workers/trainer.py:361-456`` -- on the GPU, with NCCL for the cross-GPU exchange.

``Server`` is the drop-in: ``get_avg_params`` / ``get_weighted_avg_params`` over nested lists
``system_params[system][member][layer]`` (federated.py:18-122), each layer reduced by one kernel launch.

``FederatedAggregator`` is what the batched trainer uses: the actor/critic gradients (or weights) of a
``DDPGPopulation`` are reduced over the members of each system on this GPU (``avd_fed_reduce``), exchanged
with ONE ``all_reduce(sum)`` over NVLink on a flat fp32 buffer ``[systems x (actor ‖ critic ‖ sum_w)]`` when a
process group spans several GPUs, scaled by 1/P or 1/sum(w), and written back to every member
(``avd_fed_broadcast``), after which each member applies Adam / Polyak (gradients mode, trainer.py:400-431) or
takes the averaged weights for online AND target nets (weights mode, trainer.py:433-456).

Systems: interfrl = follower index m averaged over platoons (trainer.py:338-339, 419-421) -- the one
cross-GPU exchange, since platoons are sharded over ranks; intrafrl = platoon averaged over its followers
(trainer.py:341-342, 423-425) -- purely local.  Agent index a = m*G + g.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np
import torch

from .. import _lib


def _as_cuda(x):
    if torch.is_tensor(x):
        return x.detach().to("cuda", torch.float32)
    return torch.as_tensor(np.asarray(x, dtype=np.float32), device="cuda")


class Server:
    def __init__(self, name, debug_enabled=False):
        self.name, self.debug = name, debug_enabled
        self.lib = _lib.load()
        _lib.require_device()

    def _reduce(self, members, scale):
        """members: list of X same-shaped layer tensors -> scale * sum (one avd_fed_reduce launch)."""
        shape = tuple(np.shape(members[0]))
        stack = torch.stack([_as_cuda(m).reshape(-1) for m in members]).contiguous()
        x, n = stack.shape
        out = torch.empty(n, dtype=torch.float32, device="cuda")
        sc = torch.tensor([scale], dtype=torch.float32, device="cuda")
        _lib.check(self.lib.avd_fed_reduce(_lib.ptr(out), n, _lib.ptr(stack), n, 1, x, 0, 1, None, _lib.ptr(sc), n,
                                           _lib.current_stream()))
        return out.reshape(shape)

    def get_avg_params(self, system_params: list):
        """[[mean over members of layer l for l in layers] for each system]  (federated.py:47-63)."""
        out = []
        for members in system_params:
            n_layers = len(members[0])
            out.append([self._reduce([mem[l] for mem in members], 1.0 / len(members)) for l in range(n_layers)])
        return out

    def get_weighted_avg_params(self, system_params: list, weight_sums):
        """Members arrive pre-multiplied by their weights; result = float32(1/sum_w) * sum  (federated.py:99-118)."""
        out = []
        for members, wsum in zip(system_params, weight_sums):
            n_layers = len(members[0])
            scale = float(np.float32(1 / float(wsum)))
            out.append([self._reduce([mem[l] for mem in members], scale) for l in range(n_layers)])
        return out


def exchange_and_scale(buf: torch.Tensor, process_group=None, n: Optional[int] = None) -> torch.Tensor:
    """buf[systems, n+1]: local (weighted) SUMS with the local member count / weight sum in the last column.
    One all_reduce(sum) over the group (NCCL on GPUs, gloo in the CPU tests), then the division that turns the
    sums into the mean (federated.py:62) or the weighted mean (federated.py:110).  In place."""
    n = buf.shape[1] - 1 if n is None else int(n)      # divisor column (the row pitch may be padded beyond n + 1)
    if process_group is not None:
        import torch.distributed as dist
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=process_group)
    if buf.is_cuda:
        _lib.check(_lib.load().avd_fed_finalize(_lib.ptr(buf), buf.shape[1], buf.shape[0], n, _lib.current_stream()))
    else:   # host tensors: only the gloo unit test of the exchange logic
        buf[:, :n] *= (1.0 / buf[:, n]).unsqueeze(1)
    return buf


class PeerExchange:
    """NVLink-native transport of the interfrl exchange (csrc/avd_peer.cu): a symmetric, peer-mapped buffer per rank
    (torch.distributed._symmetric_memory) holding two alternating halves of partial sums plus the epoch flags; ONE kernel per
    round signals the peers, waits for them, reads the sum over ranks -- reduced inside the NVSwitch through the NVLS multicast
    mapping when the fabric provides one, otherwise with peer loads -- and either writes the means locally (`exchange`) or
    consumes them on the spot (Adam + Polyak of every local member, `FederatedAggregator.aggregate_gradients`).  The epoch of the
    barrier is a counter in device memory (`ctrl`), so rounds captured into a CUDA graph replay correctly.  Collective: every rank
    of the group must construct it (rendezvous) and issue the same sequence of rounds."""
    FLAG_BYTES = 256

    def __init__(self, process_group, n_systems: int, max_pitch: int, device, allow_multicast: bool = True):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.lib = _lib.load()
        self.half_bytes = (n_systems * max_pitch * 4 + 255) // 256 * 256
        nbytes = self.FLAG_BYTES + 2 * self.half_bytes
        self.raw = symm.empty(nbytes, dtype=torch.uint8, device=device)
        self.raw.zero_()
        torch.cuda.synchronize(device)
        self.hdl = symm.rendezvous(self.raw, process_group.group_name)
        self.comm = _lib.PeerComm()
        self.comm.rank, self.comm.world = self.hdl.rank, self.hdl.world_size
        if self.hdl.world_size > _lib.AVD_MAX_PEERS:
            raise ValueError(f"at most {_lib.AVD_MAX_PEERS} ranks")
        for r, ptr in enumerate(self.hdl.buffer_ptrs):
            self.comm.peer_base[r] = int(ptr)
        self.comm.multicast_base = int(getattr(self.hdl, "multicast_ptr", 0) or 0) if allow_multicast else 0
        self.nvls = self.comm.multicast_base != 0
        self.ctrl = torch.zeros(4, dtype=torch.int32, device=device)      # [0] completed rounds (device-resident epoch), [1] CTA ticket,
                                                                           # [2] 1 + rank of a peer that missed a round's barrier (0: healthy)
        dist.barrier(group=process_group)        # every rank has zeroed its flags before the first signal can arrive
        self.round = 0                           # host count: only its PARITY (which half) goes into launch arguments

    def data_offset(self) -> int:
        return self.FLAG_BYTES + (self.round & 1) * self.half_bytes

    def check(self):
        """Raise if a round's cross-rank barrier timed out (synchronises the device: call it at episode / checkpoint boundaries).
        The kernels give up after AVD_PEER_TIMEOUT_MS instead of spinning forever when a peer never issues the round."""
        missing = int(self.ctrl[2].item())
        if missing:
            raise RuntimeError(f"federated exchange: rank {missing - 1} did not reach the barrier of a round within the time limit "
                               f"(rank {self.comm.rank} of {self.comm.world}); the averaged values of that round are invalid")

    def half(self, n_systems: int, pitch: int) -> torch.Tensor:
        """This round's [n_systems, pitch] float32 view of the local symmetric buffer (fill it, then exchange)."""
        off = self.data_offset()
        return self.raw[off:off + n_systems * pitch * 4].view(torch.float32).view(n_systems, pitch)

    def exchange(self, out: torch.Tensor, n: int):
        """out[s, :n] = sum over ranks of half[s, :n] / sum over ranks of half[s, n];  out[s, n] = that divisor."""
        S, pitch = out.shape
        _lib.check(self.lib.avd_fed_exchange_peer(C.byref(self.comm), 0, self.data_offset(), _lib.ptr(self.ctrl), _lib.ptr(out), pitch, S, n,
                                                  _lib.current_stream()))
        self.round += 1
        return out


def shard_platoons(num_platoons: int, rank: int, world: int):
    """Contiguous platoon range of a rank (SURVEY.md §8e): [lo, hi)."""
    base, rem = divmod(num_platoons, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class FederatedAggregator:
    def __init__(self, population, conf, process_group=None, world_size: Optional[int] = None,
                 reference_weights_quirk: bool = True, transport: str = "auto", runs: int = 1):
        """population: DDPGPopulation (A = G*M agents of THIS rank).  process_group: a torch.distributed group
        (NCCL on GPUs) or None for single-process.  reference_weights_quirk: weights mode applies system 0's
        average to every agent, as workers/trainer.py:442-456 does (`[...][0]`).  transport: "peer" = the NVLink-native
        one-kernel exchange over symmetric memory (NVLS in-switch reduction when available; "p2p" forces plain peer loads),
        "nccl" = all_reduce + finalize,
        "auto" = peer when the group spans several CUDA ranks and symmetric memory can be set up ON EVERY RANK, else nccl.
        runs: the population's groups are `runs` independent runs of G / runs groups (DDPGPopulation seeds); interfrl then averages
        each follower over the groups of its own run.  A population with per-run overrides (DDPGPopulation.hp) applies every round
        with each agent's own learning rates and tau."""
        self.pop, self.conf, self.pg = population, conf, process_group
        self.lib = _lib.load()
        if conf.fed_method not in ("interfrl", "intrafrl"):
            raise ValueError(f"fed_method {conf.fed_method!r} is not a federated method")
        self.inter = conf.fed_method == "interfrl"
        self.quirk = reference_weights_quirk
        self.world = 1
        if process_group is not None or (world_size or 1) > 1:
            import torch.distributed as dist
            self.world = dist.get_world_size(process_group)
        G, M = population.G, population.M
        self.runs = int(runs)
        if self.runs > 1 and conf.aggregation_method == conf.weights:
            raise NotImplementedError("weights-mode FRL over several runs: its reference quirk broadcasts system 0 to every agent, "
                                      "which would have to be per run")
        # member row of (system s, member x) = s*stride_s + x*stride_x in the [A, n] banks (a = m*G + g).  interfrl over runs: system
        # (m, run) = m*runs + run has the run's Gr groups as members, row (m*runs + run)*Gr + g' = m*G + run*Gr + g'.
        if self.inter:
            Gr = G // self.runs
            self.n_systems, self.n_members, self.stride_s, self.stride_x = M * self.runs, Gr, Gr, 1
        else:
            self.n_systems, self.n_members, self.stride_s, self.stride_x = G, M, 1, G
        dev = population.device
        self._bufs = {}
        self.device = dev
        self.apply_mask = None
        if (not self.inter) and getattr(conf, "intra_directional_averaging", False):
            mask = torch.ones(G * M, dtype=torch.uint8, device=dev)
            mask[:G] = 0            # follower m = 0 ("leader is king", trainer.py:417-418, 450-451)
            self.apply_mask = mask
        self.rounds = 0
        self.peer = None
        self.transport = "nccl" if (self.inter and self.world > 1) else "local"
        self.fallback_reason = None
        if transport not in ("auto", "peer", "p2p", "nccl"):
            raise ValueError("transport must be auto, peer, p2p or nccl")
        if transport != "nccl" and self.inter and self.world > 1 and dev.type == "cuda":
            self._setup_peer(process_group, transport, dev)
        self.ctrl = torch.zeros(4, dtype=torch.int32, device=dev) if dev.type == "cuda" else None     # single-rank rounds of the fused consumer
        self.wsum = torch.zeros(self.n_systems, dtype=torch.float32, device=dev)
        self.last_weight_sums = None         # [systems] divisors of the last round (sum of the FedAvg weights over ALL members), or None
        self._apply_io = None

    def _setup_peer(self, process_group, transport, dev):
        """Symmetric-memory set-up, agreed COLLECTIVELY: a rank that failed locally must not call all_reduce while the others spin
        in the peer kernel, so every rank contributes a success flag and all take the peer transport only if all succeeded."""
        import torch.distributed as dist
        pop = self.pop
        max_pitch = (pop.actor.total + pop.critic.total + 1 + 3) // 4 * 4
        peer, err = None, None
        try:
            peer = PeerExchange(process_group, self.n_systems, max_pitch, dev, allow_multicast=transport != "p2p")
        except (RuntimeError, ValueError, ImportError, AttributeError, NotImplementedError) as e:      # what symm.empty / rendezvous raise
            err = e
        ok = torch.tensor([1 if peer is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=process_group)
        if int(ok.item()) == 1:
            self.peer = peer
            self.transport = "peer/nvls" if peer.nvls else "peer/p2p"
            return
        self.fallback_reason = repr(err) if err is not None else "symmetric memory unavailable on another rank"
        if transport in ("peer", "p2p"):
            raise RuntimeError(f"peer transport requested but not available on every rank: {self.fallback_reason}")
        import warnings
        warnings.warn(f"FederatedAggregator: falling back to the NCCL transport ({self.fallback_reason})")

    @property
    def graph_safe(self) -> bool:
        """Rounds may be captured into a CUDA graph: the peer kernels keep their epoch on the device; single-rank rounds have no
        exchange at all.  (The NCCL transport goes through torch.distributed, which this package does not capture.)"""
        return self.world == 1 or self.peer is not None or not self.inter

    def _buffer(self, na, nc):
        key = (na, nc)
        if key not in self._bufs:
            pitch = (na + nc + 1 + 3) // 4 * 4        # rows start 16-byte aligned (vector / multimem loads of the peer exchange)
            self._bufs[key] = torch.zeros(self.n_systems, pitch, dtype=torch.float32, device=self.device)
        return self._bufs[key]

    def _weights(self, weights):
        if weights is None:
            return None
        return torch.as_tensor(weights, dtype=torch.float32, device=self.device).reshape(self.n_systems, self.n_members).contiguous()

    def _use_peer(self):
        return self.peer is not None and self.inter and self.world > 1

    def _reduce(self, a_src, na, c_src, nc, a_pitch, c_pitch, weights):
        """Local (weighted) sums of both banks + the divisor column, one launch; with the peer transport they go straight into this
        round's half of the symmetric buffer.  -> (tensor [systems, pitch] holding the partial sums, pitch)"""
        S, X = self.n_systems, self.n_members
        buf = self._buffer(na, nc)
        pitch = buf.shape[1]
        dst = self.peer.half(S, pitch) if self._use_peer() else buf
        w = self._weights(weights)
        _lib.check(self.lib.avd_fed_reduce2(_lib.ptr(dst), pitch, _lib.ptr(a_src), a_pitch, na, _lib.ptr(c_src), c_pitch, nc, S, X,
                                            self.stride_s, self.stride_x, _lib.ptr(w), _lib.current_stream()))
        return dst, pitch

    def _reduce_exchange(self, a_src, na, c_src, nc, a_pitch, c_pitch, weights):
        """-> buffer [systems, pitch]: columns [0, na+nc) the (weighted) means of actor / critic vectors, column na+nc the divisor."""
        buf = self._buffer(na, nc)
        self._reduce(a_src, na, c_src, nc, a_pitch, c_pitch, weights)
        if self._use_peer():
            self.peer.exchange(buf, na + nc)
        else:
            exchange_and_scale(buf, self.pg if (self.inter and self.world > 1) else None, n=na + nc)
        self.last_weight_sums = buf[:, na + nc]
        self.rounds += 1
        return buf

    def aggregate_gradients(self, weights=None, apply: bool = True, write_back: bool = True, apply_mask=None):
        """train_all_models_federated_gradients (trainer.py:400-431): average actor/critic gradients per system, then every member
        applies them with its own Adam and soft-updates its targets.  On CUDA with `apply` this is TWO launches: avd_fed_reduce2 and
        the fused consumer avd_fed_apply_gradients (barrier -> in-switch reduction -> division -> Adam -> Polyak -> step counters);
        `write_back` also stores the averaged gradients into every member's .grad row (what the unfused path leaves there).
        The NCCL transport, `apply=False` and host tensors take reduce -> all_reduce -> finalize -> broadcast (-> Adam / Polyak).
        apply_mask: [A] uint8, the agents that take this round (default: self.apply_mask); the others keep weights and gradients."""
        pop = self.pop
        mask = self.apply_mask if apply_mask is None else apply_mask
        na, nc = pop.actor.n_train, pop.critic.n_train
        fused = apply and self.device.type == "cuda" and (self._use_peer() or not (self.inter and self.world > 1))
        if fused:
            part, pitch = self._reduce(pop.actor.grad, na, pop.critic.grad, nc, na, nc, weights)
            self._apply_fused(part, pitch, write_back, mask)
            self.last_weight_sums = self.wsum
            self.rounds += 1
            return None
        buf = self._reduce_exchange(pop.actor.grad, na, pop.critic.grad, nc, na, nc, weights)
        _lib.check(self.lib.avd_fed_broadcast2(_lib.ptr(pop.actor.grad), na, na, _lib.ptr(pop.critic.grad), nc, nc, _lib.ptr(buf), buf.shape[1],
                                               self.n_systems, self.n_members, self.stride_s, self.stride_x, _lib.ptr(mask),
                                               _lib.current_stream()))
        if apply:
            pop.apply_gradients_and_soft_update(mask)
        return buf

    def _apply_fused(self, part, pitch, write_back, mask):
        pop, conf = self.pop, self.conf
        if self._apply_io is None:
            io = _lib.FedApplyIO()
            a, c = pop.actor, pop.critic
            io.n_systems, io.n_members, io.member_stride_s, io.member_stride_x, io.A = self.n_systems, self.n_members, self.stride_s, self.stride_x, pop.A
            io.actor, io.t_actor, io.actor_m, io.actor_v, io.actor_step = a.flat.data_ptr(), pop.t_actor.flat.data_ptr(), a.m.data_ptr(), a.v.data_ptr(), a.step.data_ptr()
            io.critic, io.t_critic, io.critic_m, io.critic_v, io.critic_step = c.flat.data_ptr(), pop.t_critic.flat.data_ptr(), c.m.data_ptr(), c.v.data_ptr(), c.step.data_ptr()
            io.actor_total, io.actor_train, io.critic_total, io.critic_train = a.total, a.n_train, c.total, c.n_train
            io.wsum_out = self.wsum.data_ptr()
            io.agent_hp = None if pop.hp is None else pop.hp.data_ptr()      # per-run learning rates and tau (DDPGPopulation overrides)
            io.actor_lr, io.critic_lr, io.beta1, io.beta2, io.eps, io.tau = float(conf.actor_lr), float(conf.critic_lr), 0.9, 0.999, 1e-7, float(conf.tau)
            self._apply_io = io
        io = self._apply_io
        io.pitch = pitch
        io.apply_mask = None if mask is None else mask.data_ptr()
        io.actor_grad_out = pop.actor.grad.data_ptr() if write_back else None
        io.critic_grad_out = pop.critic.grad.data_ptr() if write_back else None
        if self._use_peer():
            io.comm, io.flag_offset, io.data_offset = self.peer.comm, 0, self.peer.data_offset()
            io.local_sums, io.ctrl = None, self.peer.ctrl.data_ptr()
        else:
            io.comm.rank, io.comm.world = 0, 1
            io.flag_offset, io.data_offset, io.local_sums, io.ctrl = 0, 0, part.data_ptr(), self.ctrl.data_ptr()
        _lib.check(self.lib.avd_fed_apply_gradients(C.byref(io), _lib.current_stream()))
        if self._use_peer():
            self.peer.round += 1

    def check_health(self):
        """Raise if a cross-rank round timed out on this rank (PeerExchange.check; synchronises the device).  No-op for the NCCL and
        single-rank transports, whose failures surface through torch.distributed / CUDA errors."""
        if self.peer is not None:
            self.peer.check()

    def aggregate_weights(self, weights=None):
        """train_all_models_federated_weights (trainer.py:433-456): average `.weights` (incl. BN statistics) and
        set them on the online AND target nets of every member."""
        pop = self.pop
        na, nc = pop.actor.total, pop.critic.total
        buf = self._reduce_exchange(pop.actor.flat, na, pop.critic.flat, nc, na, nc, weights)
        st = _lib.current_stream()
        for a_bank, c_bank in ((pop.actor, pop.critic), (pop.t_actor, pop.t_critic)):      # online AND target nets (trainer.py:448-456)
            if self.quirk:   # every agent receives system 0's average
                _lib.check(self.lib.avd_fed_broadcast2(_lib.ptr(a_bank.flat), na, na, _lib.ptr(c_bank.flat), nc, nc, _lib.ptr(buf), buf.shape[1],
                                                       1, pop.A, 0, 1, _lib.ptr(self.apply_mask), st))
            else:
                _lib.check(self.lib.avd_fed_broadcast2(_lib.ptr(a_bank.flat), na, na, _lib.ptr(c_bank.flat), nc, nc, _lib.ptr(buf), buf.shape[1],
                                                       self.n_systems, self.n_members, self.stride_s, self.stride_x,
                                                       _lib.ptr(self.apply_mask), st))
        return buf
