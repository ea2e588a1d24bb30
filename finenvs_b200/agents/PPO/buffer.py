"""Buffer — drop-in for the reference's PPO rollout storage, finenvs/agents/PPO/buffer.py:8-152.

Same constructor and methods (`store`, `size`, `prepare_training_data`, `get_batches`,
`get_mini_batch_indices`, `clear`, the `container` dict), so `PPOAgent` runs unchanged with
`agent.buffer = Buffer(num_mini_batches, gamma, device_id)`.  What differs is the storage:

* the reference re-grows every tensor with `torch.cat(..., dim=1)` on each store (buffer.py:51-56):
  O(T^2) bytes per rollout, (N, t, W, 5) f64 for the observations.  Here every key lives in ONE
  pre-allocated TIME-MAJOR tensor (capacity, N, ...): a store is a copy into slot t, and with
  `bind_env(env)` not even that — the env's step kernel writes each observation straight into the slot
  the agent will store it in (zero-copy hand-off; only the first observation after `clear()` is copied).
* `compute_returns_and_advantages` (buffer.py:80-100), a Python loop of ~6 torch ops per time step, is ONE
  launch of `fe_returns_advantages` (csrc/fe_rollout.cu) with the reference's dtype promotion.
* after `prepare_training_data` the flattened sample order is time-major (sample = t * N + env) where the
  reference's is env-major (env * T + t).  Every key uses the same order and `get_batches()` always
  shuffles (buffer.py:111-127), so training sees the same distribution of mini-batches.

Observations as handles (`bind_env(env, lazy=True)`, single-asset envs).  An observation is fully described by the
12-byte handle (row0 i64, posfeat): obs[j, 0:4] = logret[row0 + j], obs[j, 4] = posfeat.  In this mode `states` is
stored as two time-major tensors, row0 (capacity + 1, N) i64 and posfeat (capacity + 1, N) in the observation dtype,
instead of (capacity + 1, N, W, 5) values: 1 Mi envs x 64 steps at W = 60 take 0.8 GB (f32) instead of 82 GB.  The env
still returns dense observations to the policy; `store()` accepts exactly those tensors (it records the handle the env
already wrote into its slot; any other tensor raises ValueError, since a tensor cannot be turned back into a handle).
After `prepare_training_data`, `container["states"]` is a `LazyStates`, and `shuffle()` permutes the handles, not the
observations.  The reference's trainer (finenvs/agents/PPO/PPO_agent.py) consumes a rollout as

    batch = buffer.get_batches()                    # shuffled; {"states", "actions", "log_probs", "advantages", "returns"}
    for indices in buffer.get_mini_batch_indices():  # one 1-D int64 tensor of sample numbers per mini-batch
        states = batch["states"][indices, :]        # LazyStates: one fe_gather_obs launch -> a new dense tensor

`LazyStates` has `shape` ((T*N, W, 5), or (T*N, W*5) for flat_obs envs), `dtype`, `device` and `len()`; indexing by a
1-D integer tensor, a slice, `(index, :)` or `(index, ...)` returns a new dense tensor gathered by ONE launch of
`fe_gather_obs` (TMA gather4 while the series' observation-layout table stays in L2), and `materialize()` returns every
sample.  Index values must lie in [0, len) (negative indices are not wrapped).

There is no CPU path: the tensors must live on a CUDA device.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import weakref

import numpy as np
import torch

from ... import _lib
from ...base_object import BaseObject
from ...device_utils import require_cuda_device

_KEYS = ("states", "actions", "rewards", "dones", "log_probs", "values")


class LazyStates:
    """The flattened `states` of a rollout kept as handles (bind_env(env, lazy=True)); see the module docstring."""

    def __init__(self, env, row0: torch.Tensor, posfeat: torch.Tensor):
        self.env, self.row0, self.posfeat = env, row0, posfeat
        W, F = env.num_intervals, env.num_obs
        M = row0.numel()
        self.shape = torch.Size((M, W * F) if env.flat_obs else (M, W, F))
        self.dtype = env.obs_dtype
        self.device = row0.device

    def __len__(self) -> int:
        return self.shape[0]

    def _gather(self, row0: torch.Tensor, posfeat: torch.Tensor, index: Optional[torch.Tensor], count: int) -> torch.Tensor:
        out = torch.empty((count, *self.shape[1:]), dtype=self.dtype, device=self.device)
        self.env.gather_obs(row0, posfeat, index, out)
        return out

    def materialize(self) -> torch.Tensor:
        """Every sample as one dense tensor."""
        return self._gather(self.row0, self.posfeat, None, len(self))

    def select(self, index: torch.Tensor) -> "LazyStates":
        """The handles of samples `index`, in that order (no observation is built)."""
        return LazyStates(self.env, self.row0[index], self.posfeat[index])

    def __getitem__(self, key) -> torch.Tensor:
        if isinstance(key, tuple):
            rest = key[1] if len(key) == 2 else None
            if not (rest is Ellipsis or (isinstance(rest, slice) and rest == slice(None))):
                raise IndexError("LazyStates takes (index, :) or (index, ...) as a tuple index")
            key = key[0]
        if isinstance(key, slice):
            start, stop, step = key.indices(len(self))
            if step == 1:   # a contiguous range of handles: no index tensor needed
                stop = max(start, stop)
                return self._gather(self.row0[start:stop], self.posfeat[start:stop], None, stop - start)
            key = torch.arange(start, stop, step, device=self.device)
        if torch.is_tensor(key) and key.dim() == 1 and not key.is_floating_point() and key.dtype != torch.bool:
            index = key.to(device=self.device, dtype=torch.int64).contiguous()
            return self._gather(self.row0, self.posfeat, index, index.numel())
        raise IndexError("LazyStates is indexed by a 1-D integer tensor, a slice, (index, :) or (index, ...)")


class Buffer(BaseObject):
    def __init__(self, num_mini_batches: int = 16, gamma: float = 0.99, device_id: int = 0, *, capacity: int = 64):
        """Reference arguments: buffer.py:9-12.  `capacity` = time steps pre-allocated per rollout (the reference
        example trains every 64 steps, PPO_LSTM_training_SPY.py:12); it doubles on overflow."""
        self.num_mini_batches = num_mini_batches
        self.gamma = gamma
        self.device = require_cuda_device(device_id)
        self._dev = torch.device(self.device)
        self._L = _lib.lib()
        self.capacity = int(capacity)
        self._store: Dict[str, Optional[torch.Tensor]] = {k: None for k in _KEYS}
        self._t = 0                  # time steps stored in the current rollout
        self._env = None
        self._held_slot = None       # states slot holding the observation the agent has in hand (None: not in storage)
        self._states_flat = None     # states storage as one flat tensor: slot k = [k * stride, k * stride + numel)
        self._slot_stride = 0
        self._lazy = False           # bind_env(env, lazy=True): states are kept as handles
        self._row0 = None            # lazy: (capacity + 1, N) i64 handle slots
        self._posfeat = None         # lazy: (capacity + 1, N) position features, observation dtype
        self._handed = []            # lazy: [(slot, weak reference to the tensor the env returned)] for the last two
        self.container: Dict[str, Optional[torch.Tensor]] = {k: None for k in (*_KEYS, "advantages", "returns")}
        self.batch_keys = ["states", "actions", "log_probs", "advantages", "returns"]

    # ------------------------------------------------------------------ zero-copy observation hand-off
    def bind_env(self, env, lazy: bool = False) -> None:
        """Let `env` (finenvs_b200 TimeSeriesEnv) write its observations directly into this buffer's `states`
        storage: reset()/step() then return views of the slot the agent stores next.  May be called at any point
        of the loop (before or after the first reset(), or between rollouts): an observation the agent already holds
        is simply copied in by the store() that follows.

        lazy=True (single-asset envs; NotImplementedError otherwise): the buffer keeps each observation's 12-byte handle
        instead (module docstring).  Bind before the reset() whose observation is stored first: store() only accepts
        observations the bound env returned."""
        if lazy != self._lazy:
            if self._t != 0:
                raise ValueError("bind_env cannot switch between dense and handle storage inside a rollout")
            self._store["states"] = self._states_flat = self._row0 = self._posfeat = None
        if lazy:
            env._bind_handle_ring(self)
        else:
            env._obs_ring, env._handle_ring = self, None
        self._lazy = lazy
        self._env = env
        self._held_slot = None
        self._handed = []

    def next_obs_slot(self, shape, dtype, for_reset: bool = False) -> torch.Tensor:
        """Called by the bound env instead of torch.empty.  Slot protocol (the loop of
        examples/time_series/PPO_LSTM_training_SPY.py:22-30 is `agent.step -> env.step -> agent.store`):

        * reset(): the observation becomes the one the agent holds and stores NEXT -> slot `_t`;
        * step(): the agent still holds the previous observation, which store() puts in slot `_t` (a no-op when it
          already lives there) -> the new one goes to slot `_t + 1`, where it will be "next" after that store().

        A slot that holds the agent's current observation is never handed out again (after clear() the held observation
        sits in the old slot T; a second step() without a store() in between would ask for the same slot twice): those
        calls get the next free slot or a plain tensor, and store() copies.  capacity + 1 slots exist: after T stores
        the observation of step T is live in slot T."""
        self._states_storage(tuple(shape), dtype)
        k = self._t if for_reset else self._t + 1
        if not for_reset and self._held_slot is not None and k == self._held_slot:
            k += 1
            if k == self._t:        # cannot happen (k >= _t + 2), kept as an invariant
                raise AssertionError("observation slot would alias the slot being stored")
        while k >= self._num_slots():
            self._grow()
        self._held_slot = k
        return self._state_slot(k)

    def next_handle_slot(self, num_envs: int, dtype, for_reset: bool = False):
        """next_obs_slot() for an env bound with lazy=True: the (row0, posfeat) views of the handle slot the env writes
        next, chosen by the same protocol."""
        self._handle_storage(num_envs, dtype)
        k = self._t if for_reset else self._t + 1
        if not for_reset and self._held_slot is not None and k == self._held_slot:
            k += 1
        while k >= self.capacity + 1:
            self._grow()
        self._held_slot = k
        return self._row0[k], self._posfeat[k]

    def hand_out(self, obs: torch.Tensor) -> None:
        """The bound env returns `obs`, built from the handle slot next_handle_slot() gave it last."""
        self._handed = [*self._handed[-1:], (self._held_slot, weakref.ref(obs))]

    def _handle_slot_of(self, states: torch.Tensor) -> Optional[int]:
        for slot, ref in reversed(self._handed):
            obs = ref()
            if obs is not None and (obs is states or (obs.data_ptr() == states.data_ptr() and obs.shape == states.shape
                                                      and obs.dtype == states.dtype)):
                return slot
        return None

    def _handle_storage(self, num_envs: int, dtype) -> None:
        if self._row0 is not None and self._row0.shape[1] == num_envs and self._posfeat.dtype == dtype:
            return
        if self._t != 0 and self._row0 is not None:
            raise ValueError("'states' changed shape/dtype inside a rollout")
        self._row0 = torch.empty((self.capacity + 1, num_envs), dtype=torch.int64, device=self._dev)
        self._posfeat = torch.empty((self.capacity + 1, num_envs), dtype=dtype, device=self._dev)
        self._held_slot = None
        self._handed = []

    def _store_handles(self, states: torch.Tensor) -> None:
        slot = self._handle_slot_of(states)
        if slot is None:
            raise ValueError("with bind_env(env, lazy=True) store() takes the observations the bound env returned: the "
                             "buffer keeps their handles, and a tensor cannot be turned back into a handle")
        while self._t + 1 >= self.capacity + 1:       # slot _t for this observation, slot _t + 1 for the one in flight
            self._grow()
        if slot != self._t:
            if self._held_slot == self._t:
                raise RuntimeError("Buffer.store(states) would overwrite the observation the bound env returned last; "
                                   "store the observations in the order they were returned")
            self._row0[self._t].copy_(self._row0[slot])
            self._posfeat[self._t].copy_(self._posfeat[slot])

    # ------------------------------------------------------------------ storage
    def _num_slots(self) -> int:
        return 0 if self._states_flat is None else self._states_flat.numel() // self._slot_stride

    def _states_storage(self, shape, dtype) -> None:
        """(capacity + 1) observation slots whose starts are 16-byte aligned whatever N, W and dtype are (the step
        kernels store observations with 16-byte bulk / vector stores): the per-slot stride is padded up."""
        if self._states_flat is not None and self._states_shape == shape and self._states_flat.dtype == dtype:
            return
        if self._t != 0 and self._states_flat is not None:
            raise ValueError("'states' changed shape/dtype inside a rollout")
        numel = 1
        for d in shape:
            numel *= int(d)
        per16 = 16 // torch.empty((), dtype=dtype).element_size()
        self._slot_stride = max(per16, (numel + per16 - 1) // per16 * per16)
        self._states_shape, self._states_numel = tuple(shape), numel
        self._states_flat = torch.empty((self.capacity + 1) * self._slot_stride, dtype=dtype, device=self._dev)
        self._store["states"] = self._states_view(self.capacity + 1)
        self._held_slot = None

    def _state_slot(self, k: int) -> torch.Tensor:
        o = k * self._slot_stride
        return self._states_flat[o: o + self._states_numel].view(self._states_shape)

    def _states_view(self, T: int) -> torch.Tensor:
        """(T, *shape) view of the first T slots (contiguous when the stride needed no padding)."""
        inner = torch.empty(self._states_shape, device="meta").stride()
        return torch.as_strided(self._states_flat, (T, *self._states_shape), (self._slot_stride, *inner))

    def _alloc(self, key: str, like: torch.Tensor) -> torch.Tensor:
        if key == "states":
            self._states_flat = None
            self._states_storage(tuple(like.shape), like.dtype)
            return self._store["states"]
        self._store[key] = torch.empty((self.capacity, *like.shape), dtype=like.dtype, device=self._dev)
        return self._store[key]

    def _grow(self) -> None:
        self.capacity *= 2
        if self._row0 is not None:  # handles: same slot numbers in the larger storage
            for name in ("_row0", "_posfeat"):
                old = getattr(self, name)
                new = torch.empty((self.capacity + 1, old.shape[1]), dtype=old.dtype, device=self._dev)
                new[: old.shape[0]].copy_(old)
                setattr(self, name, new)
        else:
            self._held_slot = None  # an observation in hand stays valid in the OLD storage; no new slot aliases it
        for key, old in self._store.items():
            if old is None:
                continue
            if key == "states":
                flat = torch.empty((self.capacity + 1) * self._slot_stride, dtype=old.dtype, device=self._dev)
                flat[: self._states_flat.numel()].copy_(self._states_flat)
                self._states_flat = flat
                self._store["states"] = self._states_view(self.capacity + 1)
                continue
            new = torch.empty((self.capacity, *old.shape[1:]), dtype=old.dtype, device=self._dev)
            new[: old.shape[0]].copy_(old)
            self._store[key] = new

    def force_2D(self, tensor: torch.Tensor) -> torch.Tensor:
        """buffer.py:58-63 without the time axis (it is the leading storage axis here): (N,) -> (N, 1)."""
        return tensor.unsqueeze(-1) if tensor.dim() < 2 else tensor

    def store_tensor(self, key: str, tensor: torch.Tensor) -> None:
        """buffer.py:51-56: append one time step of `key`."""
        if key == "states" and self._lazy:
            return self._store_handles(tensor)
        tensor = self.force_2D(tensor)
        if key == "states":
            return self._store_states(tensor)
        st = self._store[key]
        if st is None:
            st = self._alloc(key, tensor)
        elif st.shape[1:] != tensor.shape or st.dtype != tensor.dtype:
            if self._t != 0:
                raise ValueError(f"'{key}' changed shape/dtype inside a rollout: {tuple(tensor.shape)} {tensor.dtype} "
                                 f"vs {tuple(st.shape[1:])} {st.dtype}")
            st = self._alloc(key, tensor)
        if self._t >= self.capacity:
            self._grow()
            st = self._store[key]
        slot = st[self._t]
        if tensor.data_ptr() != slot.data_ptr():      # the bound env already wrote it in place otherwise
            slot.copy_(tensor)

    def _store_states(self, tensor: torch.Tensor) -> None:
        self._states_storage(tuple(tensor.shape), tensor.dtype)
        while self._t + 1 >= self._num_slots():      # slot _t for this observation, slot _t + 1 for the one in flight
            self._grow()
        slot = self._state_slot(self._t)
        if tensor.data_ptr() != slot.data_ptr():      # the bound env already wrote it in place otherwise
            if self._held_slot == self._t:
                # the slot being stored into was handed out for a LATER observation that the caller still holds
                # (store() called with something other than the observation in hand): keep that one intact
                raise RuntimeError("Buffer.store(states) would overwrite the observation the bound env returned last; "
                                   "store the observations in the order they were returned")
            slot.copy_(tensor)

    def store(self, states: torch.Tensor, actions: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor,
              log_probs: torch.Tensor, values: torch.Tensor) -> None:
        """buffer.py:33-49."""
        self.store_tensor("states", states)
        self.store_tensor("actions", actions)
        self.store_tensor("rewards", rewards)
        self.store_tensor("dones", dones)
        self.store_tensor("log_probs", log_probs)
        self.store_tensor("values", values)
        self._t += 1

    def size(self) -> int:
        """buffer.py:65-74: samples held = envs x steps."""
        d = self._store["dones"]
        if d is None or self._t == 0:
            return 0
        return d.shape[1] * self._t

    # ------------------------------------------------------------------ training data
    def prepare_training_data(self, current_state_values: torch.Tensor) -> None:
        """buffer.py:76-78."""
        self.compute_returns_and_advantages(current_state_values)
        self.reshape()

    def compute_returns_and_advantages(self, last_values: torch.Tensor) -> None:
        """buffer.py:80-100 as one kernel launch over the time-major rollout."""
        T = self._t
        if T == 0:
            raise RuntimeError("the buffer is empty")
        rewards, dones, values = (self._store[k][:T] for k in ("rewards", "dones", "values"))
        N = rewards.shape[1]
        if rewards.shape[2:] != (1,) or values.shape[2:] != (1,) or dones.shape[2:] != (1,):
            raise ValueError("rewards, dones and values must be one number per env and step")
        if rewards.dtype not in (torch.float32, torch.float64):
            raise TypeError("rewards must be float32 or float64")
        if dones.dtype != torch.int32:
            dones = dones.to(torch.int32)
        values = values if values.dtype == torch.float32 else values.float()
        last = last_values.detach().to(device=self._dev, dtype=torch.float32).reshape(-1).contiguous()
        if last.numel() != N:
            raise ValueError(f"last_values must hold one value per env ({N})")
        returns = torch.empty((T, N, 1), dtype=torch.float32, device=self._dev)
        advantages = torch.empty((T, N, 1), dtype=torch.float32, device=self._dev)
        _lib.check(
            self._L.fe_returns_advantages(rewards.data_ptr(), int(rewards.dtype == torch.float64), dones.data_ptr(),
                                          values.data_ptr(), last.data_ptr(), N, T, float(self.gamma),
                                          returns.data_ptr(), advantages.data_ptr(),
                                          torch.cuda.current_stream(self._dev).cuda_stream),
            "fe_returns_advantages",
        )
        self.container["returns"] = returns
        self.container["advantages"] = advantages

    def reshape(self) -> None:
        """buffer.py:102-109: flatten (steps, envs, ...) -> (steps * envs, ...); views, no copies."""
        T = self._t
        for key in _KEYS:
            if key == "states" and self._lazy:
                self.container[key] = LazyStates(self._env, self._row0[:T].reshape(-1), self._posfeat[:T].reshape(-1))
                continue
            st = self._states_view(T) if key == "states" else self._store[key][:T]
            self.container[key] = st.reshape(T * st.shape[1], *st.shape[2:])   # a copy only if the slot stride is padded
        for key in ("returns", "advantages"):
            t = self.container[key]
            self.container[key] = t.reshape(t.shape[0] * t.shape[1], *t.shape[2:])

    def get_batches(self) -> Dict[str, torch.Tensor]:
        """buffer.py:111-116."""
        self.shuffle()
        return {key: self.container[key] for key in self.batch_keys}

    def shuffle(self) -> None:
        """buffer.py:118-127: one permutation applied to every key (to the handles for LazyStates)."""
        with torch.no_grad():
            random_indices = torch.randperm(self.size(), device=self._dev, requires_grad=False)
            for key, tensor in self.container.items():
                self.container[key] = (tensor.select(random_indices) if isinstance(tensor, LazyStates)
                                       else torch.index_select(tensor, 0, random_indices))

    def get_mini_batch_indices(self) -> List[torch.Tensor]:
        """buffer.py:129-148: contiguous index ranges of the (already shuffled) flattened samples."""
        buffer_size = self.size()
        num_mini_batches = self.num_mini_batches
        mini_batch_size = int(np.floor(buffer_size / num_mini_batches))
        if mini_batch_size * num_mini_batches != buffer_size:
            print(f"WARNING: buffer size {buffer_size} does not divide evenly into {num_mini_batches} mini-batches!")
        return [torch.arange(i * mini_batch_size, (i + 1) * mini_batch_size, dtype=torch.long, device=self._dev)
                for i in range(num_mini_batches)]

    def clear(self) -> None:
        """buffer.py:150-152.  The storage is kept for the next rollout.  The observation the agent still holds stays
        where it is (slot T of the finished rollout): the first store() of the next rollout copies it into slot 0 and
        next_obs_slot() never hands that slot out while it is held."""
        for key in self.container.keys():
            self.container[key] = None
        self._t = 0
