"""Actor / critic parameter containers -- the GPU counterpart of the reference's ``agent/model.py``.

The reference builds Keras functional models (model.py:4-38 actor, 41-85 critic).  Here a network is a flat
fp32 vector in HBM (layout in include/avddpg_b200.h, trainable tensors first) and all arithmetic happens in
the CUDA kernels; ``NetBank`` holds the vectors of a whole population of agents ``[A, total]`` and hands out
zero-copy views in the Keras orders (`.weights`, `.trainable_variables`).

``get_actor`` / ``get_critic`` keep the reference's signatures and return single-agent objects with the
surface workers/trainer.py uses: ``__call__``, ``.weights``, ``.trainable_variables``, ``.get_weights()``,
``.set_weights()``, ``.save()``.  Bit-exact TensorFlow initial weights cannot be reproduced without TF
(seeded tf.random_uniform_initializer), so initial weights are drawn from the same distributions with a torch
generator and can be injected with ``set_weights`` (SURVEY.md §3.3).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional

import numpy as np
import torch

from . import _lib

# tensor name -> shape builder; orders follow agent/model.py's layer order (see oracle/ddpg_np.py)
ACTOR_FLAT = ["W1", "b1", "g1", "be1", "W2", "b2", "g2", "be2", "W3", "b3", "mu1", "var1", "mu2", "var2"]
ACTOR_WEIGHTS = ["W1", "b1", "g1", "be1", "mu1", "var1", "W2", "b2", "g2", "be2", "mu2", "var2", "W3", "b3"]
ACTOR_TRAINABLE = ["W1", "b1", "g1", "be1", "W2", "b2", "g2", "be2", "W3", "b3"]
CRITIC_FLAT = ["Ws", "bs", "Wa", "ba", "gs", "bes", "ga", "bea", "W2", "b2", "g2", "be2", "W3", "b3",
               "mus", "vars", "mua", "vara", "mu2", "var2"]
CRITIC_WEIGHTS = ["Ws", "bs", "Wa", "ba", "gs", "bes", "mus", "vars", "ga", "bea", "mua", "vara",
                  "W2", "b2", "g2", "be2", "mu2", "var2", "W3", "b3"]
CRITIC_TRAINABLE = ["Ws", "bs", "Wa", "ba", "gs", "bes", "ga", "bea", "W2", "b2", "g2", "be2", "W3", "b3"]


def make_dims(num_states=4, layer1=256, act_layer=48, layer2=128) -> _lib.NetDims:
    return _lib.NetDims(int(num_states), int(layer1), int(act_layer), int(layer2))


def dims_from_config(conf, num_states=4) -> _lib.NetDims:
    if conf.actor_layer1_size != conf.critic_layer1_size or conf.actor_layer2_size != conf.critic_layer2_size:
        raise NotImplementedError("kernels assume actor and critic share layer1/layer2 widths (reference defaults)")
    return make_dims(num_states, conf.actor_layer1_size, conf.critic_act_layer_size, conf.actor_layer2_size)


def tensor_shapes(kind: str, d: _lib.NetDims):
    if kind == "actor":
        return {"W1": (d.ns, d.l1), "b1": (d.l1,), "g1": (d.l1,), "be1": (d.l1,), "mu1": (d.l1,), "var1": (d.l1,),
                "W2": (d.l1, d.l2), "b2": (d.l2,), "g2": (d.l2,), "be2": (d.l2,), "mu2": (d.l2,), "var2": (d.l2,),
                "W3": (d.l2, 1), "b3": (1,)}
    return {"Ws": (d.ns, d.l1), "bs": (d.l1,), "Wa": (1, d.la), "ba": (d.la,),
            "gs": (d.l1,), "bes": (d.l1,), "mus": (d.l1,), "vars": (d.l1,),
            "ga": (d.la,), "bea": (d.la,), "mua": (d.la,), "vara": (d.la,),
            "W2": (d.l1 + d.la, d.l2), "b2": (d.l2,), "g2": (d.l2,), "be2": (d.l2,), "mu2": (d.l2,), "var2": (d.l2,),
            "W3": (d.l2, 1), "b3": (1,)}


def layout(kind: str, d: _lib.NetDims):
    """-> (offsets dict name -> (offset, shape), n_trainable, total); cross-checked against the C library."""
    flat = ACTOR_FLAT if kind == "actor" else CRITIC_FLAT
    train = ACTOR_TRAINABLE if kind == "actor" else CRITIC_TRAINABLE
    shapes = tensor_shapes(kind, d)
    off, p, n_train = {}, 0, None
    for i, name in enumerate(flat):
        if i == len(train):
            n_train = p
        off[name] = (p, shapes[name])
        p += int(np.prod(shapes[name]))
    counts = (C.c_int64 * 4)()
    _lib.check(_lib.load().avd_ddpg_param_counts(C.byref(d), counts))
    want = (counts[0], counts[1]) if kind == "actor" else (counts[2], counts[3])
    if (n_train, p) != tuple(want):
        raise _lib.AvdError(f"{kind} layout mismatch between Python {(n_train, p)} and C {tuple(want)}")
    return off, n_train, p


class NetBank:
    """Flat parameters of one network kind for A agents: ``flat[A, total]`` (+ optional Adam state)."""

    def __init__(self, kind: str, dims: _lib.NetDims, num_agents: int, device, with_optimizer: bool = False):
        assert kind in ("actor", "critic")
        self.kind, self.dims, self.A = kind, dims, int(num_agents)
        self.offsets, self.n_train, self.total = layout(kind, dims)
        self.flat = torch.zeros(self.A, self.total, dtype=torch.float32, device=device)
        self.weight_names = ACTOR_WEIGHTS if kind == "actor" else CRITIC_WEIGHTS
        self.trainable_names = ACTOR_TRAINABLE if kind == "actor" else CRITIC_TRAINABLE
        self.grad = self.m = self.v = self.step = None
        if with_optimizer:
            self.grad = torch.zeros(self.A, self.n_train, dtype=torch.float32, device=device)
            self.m = torch.zeros_like(self.grad)
            self.v = torch.zeros_like(self.grad)
            self.step = torch.zeros(self.A, dtype=torch.int32, device=device)

    def view(self, name: str, agent: Optional[int] = None, source: Optional[torch.Tensor] = None):
        off, shape = self.offsets[name]
        src = self.flat if source is None else source
        n = int(np.prod(shape))
        if agent is None:
            return src[:, off: off + n].view(src.shape[0], *shape)
        return src[agent, off: off + n].view(*shape)

    def weights(self, agent: int) -> List[torch.Tensor]:
        """Keras ``model.weights`` order (views)."""
        return [self.view(n, agent) for n in self.weight_names]

    def trainable(self, agent: int) -> List[torch.Tensor]:
        return [self.view(n, agent) for n in self.trainable_names]

    def grads(self, agent: int) -> List[torch.Tensor]:
        """Gradients in ``trainable_variables`` order (views into the flat gradient vector)."""
        return [self.view(n, agent, self.grad) for n in self.trainable_names]

    def init_reference(self, generator: torch.Generator):
        """Initialisers of agent/model.py:19-25 / 53-60; every agent starts from agent 0's weights
        (workers/trainer.py:121-131)."""
        d = self.dims

        def uni(shape, bound):
            return (torch.rand(shape, generator=generator, dtype=torch.float32) * 2 - 1) * bound

        vals = {}
        if self.kind == "actor":
            vals["W1"] = uni((d.ns, d.l1), 1 / math.sqrt(d.l1))
            vals["W2"] = uni((d.l1, d.l2), 1 / math.sqrt(d.l2))
            vals["W3"] = uni((d.l2, 1), 3e-3)
            ones = ["g1", "var1", "g2", "var2"]
        else:
            vals["Ws"] = uni((d.ns, d.l1), 1 / math.sqrt(d.l1))
            vals["Wa"] = uni((1, d.la), 1 / math.sqrt(d.l2))       # model.py:70 uses the layer-2 bound
            vals["W2"] = uni((d.l1 + d.la, d.l2), 1 / math.sqrt(d.l2))
            vals["W3"] = uni((d.l2, 1), 3e-4)
            ones = ["gs", "vars", "ga", "vara", "g2", "var2"]
        self.flat.zero_()
        for name, v in vals.items():
            self.view(name).copy_(v.to(self.flat.device).unsqueeze(0).expand(self.A, *v.shape))
        for name in ones:
            self.view(name).fill_(1.0)

    def set_weights(self, agent: Optional[int], arrays):
        """Keras ``set_weights`` (list in `.weights` order); agent=None sets every agent."""
        if len(arrays) != len(self.weight_names):
            raise ValueError(f"expected {len(self.weight_names)} arrays, got {len(arrays)}")
        for name, arr in zip(self.weight_names, arrays):
            t = torch.as_tensor(np.asarray(arr.detach().cpu() if torch.is_tensor(arr) else arr, dtype=np.float32))
            shape = self.offsets[name][1]
            if tuple(t.shape) != tuple(shape):
                raise ValueError(f"{name}: shape {tuple(t.shape)} does not match {tuple(shape)}")
            dst = self.view(name, agent)
            t = t.to(self.flat.device)
            dst.copy_(t if agent is not None else t.unsqueeze(0).expand_as(dst))

    def get_weights(self, agent: int):
        return [w.detach().cpu().numpy().copy() for w in self.weights(agent)]

    def load_named(self, agent: Optional[int], named: dict):
        """Set tensors by name (oracle/ddpg_np.py naming); agent=None sets every agent."""
        for name, arr in named.items():
            t = torch.as_tensor(np.asarray(arr, dtype=np.float32)).reshape(self.offsets[name][1]).to(self.flat.device)
            dst = self.view(name, agent)
            dst.copy_(t if agent is not None else t.unsqueeze(0).expand_as(dst))


# ------------------------------------------------------------------------------------------ drop-in models
class _Model:
    """Single-agent model object with the Keras surface the reference trainer touches."""

    def __init__(self, kind, dims, high_bound=None, device=None, seed=None):
        _lib.require_device()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.bank = NetBank(kind, dims, 1, device)
        gen = torch.Generator().manual_seed(0 if seed is None else int(seed))
        self.bank.init_reference(gen)
        self.high_bound = high_bound
        self._ws = None

    @property
    def weights(self):
        return self.bank.weights(0)

    @property
    def trainable_variables(self):
        return self.bank.trainable(0)

    def get_weights(self):
        return self.bank.get_weights(0)

    def set_weights(self, arrays):
        self.bank.set_weights(0, arrays)

    def save(self, path):
        """The reference writes Keras .h5 (trainer.py:584); h5py is not part of this stack, so the same
        tensors go to an .npz with Keras `.weights` names/order (N3 in SURVEY.md §8f tracks .h5 export)."""
        np.savez(path if str(path).endswith(".npz") else str(path) + ".npz",
                 **{f"{i:02d}_{n}": w for i, (n, w) in enumerate(zip(self.bank.weight_names, self.get_weights()))})

    def _workspace(self, rows, critic):
        need = _lib.load().avd_forward_workspace_bytes(C.byref(self.bank.dims), 1, rows, int(critic), 0)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.bank.flat.device)
        return self._ws


class Actor(_Model):
    def __call__(self, state, training=False):
        s = torch.as_tensor(np.asarray(state, dtype=np.float32) if not torch.is_tensor(state) else state,
                            dtype=torch.float32, device=self.bank.flat.device).reshape(-1, self.bank.dims.ns).contiguous()
        d, n = self.bank.dims, s.shape[0]
        out = torch.empty(n, 1, dtype=torch.float32, device=s.device)
        ws = self._workspace(n, critic=False)
        _lib.check(_lib.load().avd_actor_forward(C.byref(d), 1, n, _lib.ptr(self.bank.flat), _lib.ptr(s), d.ns, 1,
                                                 float(self.high_bound), _lib.ptr(out), _lib.ptr(ws), ws.numel(), 0,
                                                 _lib.current_stream()))
        return out


class Critic(_Model):
    def __call__(self, inputs, training=False):
        state, action = inputs
        dev = self.bank.flat.device
        d = self.bank.dims
        s = torch.as_tensor(np.asarray(state, dtype=np.float32) if not torch.is_tensor(state) else state,
                            dtype=torch.float32, device=dev).reshape(-1, d.ns).contiguous()
        a = torch.as_tensor(np.asarray(action, dtype=np.float32) if not torch.is_tensor(action) else action,
                            dtype=torch.float32, device=dev).reshape(-1).contiguous()
        n = s.shape[0]
        q = torch.empty(n, 1, dtype=torch.float32, device=dev)
        ws = self._workspace(n, critic=True)
        _lib.check(_lib.load().avd_critic_forward(C.byref(d), 1, n, _lib.ptr(self.bank.flat), _lib.ptr(s), _lib.ptr(a),
                                                  _lib.ptr(q), _lib.ptr(ws), ws.numel(), 0, _lib.current_stream()))
        return q


def get_actor(num_states, num_actions, high_bound, seed_int=None, hidd_mult=1, layer1_size=400, layer2_size=300):
    """agent/model.py:4-38 signature.  num_actions must be 1 and hidd_mult 1 (decentralized framework)."""
    if num_actions != 1 or hidd_mult != 1:
        raise NotImplementedError("centralized framework (num_actions>1 / hidd_mult!=1) is outside the hot-path scope")
    return Actor("actor", make_dims(num_states, layer1_size, 48, layer2_size), high_bound, seed=seed_int)


def get_critic(num_states, num_actions, hidd_mult=1, seed_int=None, layer1_size=400, layer2_size=300, action_layer_size=64):
    """agent/model.py:41-85 signature."""
    if num_actions != 1 or hidd_mult != 1:
        raise NotImplementedError("centralized framework (num_actions>1 / hidd_mult!=1) is outside the hot-path scope")
    return Critic("critic", make_dims(num_states, layer1_size, action_layer_size, layer2_size), seed=seed_int)
