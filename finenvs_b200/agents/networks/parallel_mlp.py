"""ParallelMLP — drop-in for the reference's finenvs/agents/networks/parallel_mlp.py:9-275 that scales to
millions of envs per GPU.

Same constructor, attributes (`weight_layers`, `bias_layers`, Adam moments) and methods (`forward`,
`perturb_parameters`, `reconstruct_perturbations`, `update_parameters`, `get_l2_norm`, `adam_update`), so the
reference's `EvoAgent` logic runs unchanged on top of it.  What differs is the storage and the kernels
(csrc/fe_es.cu):

* the reference materialises one perturbed copy of every layer per env (`perturbed_weights`: N x in x out f32,
  :114-155).  Here a mirrored pair shares one UNIT perturbation eps ~ N(0,1) stored as fp16 in a packed
  layout (`fe_es_perturb`), env p evaluates theta + sigma*eps[p], env p + T/2 evaluates theta - sigma*eps[p];
* `forward` is one launch of `fe_es_forward` for the whole population — also straight from the env's lazy
  observation handles (TimeSeriesEnv.step_lazy), in which case no observation tensor exists at all;
* `update_parameters` reduces eps with `fe_es_gradient` (+ an NCCL all-reduce of the parameter-sized sum when
  the population is sharded over GPUs) and then applies the reference's Adam step op for op (:220-275).

Only tanh activations (the reference's defaults, :19-20) are implemented.  There is no CPU path.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist
import torch.nn as nn

from ... import _lib
from ...base_object import BaseObject
from ...device_utils import require_cuda_device


class ParallelMLP(BaseObject):
    def __init__(
        self,
        num_envs: int,
        num_eval_envs: int,
        shape: tuple,
        learning_rate: float = 0.01,
        noise_std_dev: float = 0.02,
        l2_coefficient: float = 0.005,
        layer_activation=nn.Tanh,
        output_activation=nn.Tanh,
        device_id: int = 0,
        *,
        seed: Optional[int] = None,
        pair_id_base: int = 0,
        total_pairs: Optional[int] = None,
        env_id_base: int = 0,
        action_noise_std: float = 0.01,
        group=None,
    ):
        """Reference arguments: :11-22.  Extensions (keyword-only): `seed` keys the perturbation / action-noise
        streams (default torch.initial_seed()); `pair_id_base`, `total_pairs`, `env_id_base`, `group` describe this
        object as a shard of a larger population (one process per GPU): perturbations are keyed by GLOBAL pair id and
        the gradient is summed over `group` and averaged over `total_pairs`."""
        self.device = require_cuda_device(device_id)
        self._dev = torch.device(self.device)
        num_training_envs = num_envs - num_eval_envs
        assert (num_training_envs) % 2 == 0 and (num_training_envs) > 0, (
            f"The number of training environments ({num_envs} - {num_eval_envs}) "
            + "must be positive and even for mirrored sampling."
        )
        if layer_activation is not nn.Tanh or output_activation is not nn.Tanh:
            raise NotImplementedError("finenvs_b200's ParallelMLP implements the reference's default tanh activations only")
        if not (2 <= len(shape) <= _lib.FE_ES_MAX_LAYERS + 1):
            raise ValueError(f"shape must have 2..{_lib.FE_ES_MAX_LAYERS + 1} entries")
        self.num_envs = num_envs
        self.num_training_envs = num_training_envs
        self.num_eval_envs = num_eval_envs
        self.num_pairs = num_training_envs // 2
        self.shape = tuple(int(d) for d in shape)
        self.learning_rate = learning_rate
        self.noise_std_dev = noise_std_dev
        self.l2_coefficient = l2_coefficient
        self.action_noise_std = action_noise_std
        self.seed = int(torch.initial_seed() if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
        self.pair_id_base = int(pair_id_base)
        self.total_pairs = int(self.num_pairs if total_pairs is None else total_pairs)
        self.env_id_base = int(env_id_base)
        self.group = group
        self.weight_layers: List[torch.Tensor] = []
        self.bias_layers: List[torch.Tensor] = []
        self.activation_functions: List[nn.Module] = []
        self.create_layers(layer_activation, output_activation)
        self.set_adam_parameters()
        # ---- packed layout (include/finenvs_b200.h) ----
        self._L = _lib.lib()
        self._net = _lib.FeEsNet(len(self.shape) - 1, (_lib.C.c_int32 * (_lib.FE_ES_MAX_LAYERS + 1))(*self.shape))
        self._pnet = _lib.C.byref(self._net)
        self.params_padded = int(self._L.fe_es_params_padded(self._pnet))
        self._widx, self._bidx = [], []
        off = 0
        for i in range(len(self.shape) - 1):
            n_in, n_out = self.shape[i], self.shape[i + 1]
            o = torch.arange(n_out, device=self._dev)
            j = torch.arange(n_in + 1, device=self._dev)
            idx = off + ((o // 8)[None, :] * (n_in + 1) + j[:, None]) * 8 + (o % 8)[None, :]     # (in + 1, out)
            self._widx.append(idx[:n_in].contiguous())
            self._bidx.append(idx[n_in:].contiguous())
            off += ((n_out + 7) // 8) * (n_in + 1) * 8
        assert off == self.params_padded
        self._theta = torch.zeros(self.params_padded, dtype=torch.float32, device=self._dev)
        self._theta_dirty = True
        self._eps = torch.empty((self.num_pairs, self.params_padded), dtype=torch.float16, device=self._dev)
        self._grad = torch.empty(self.params_padded, dtype=torch.float32, device=self._dev)
        self._scratch = torch.empty(int(self._L.fe_es_gradient_scratch(self._pnet, self.num_pairs)), dtype=torch.float32,
                                    device=self._dev)
        self.generation = 0
        self.forward_calls = 0
        self.perturbed = False

    # ------------------------------------------------------------------ reference :44-82 (unchanged)
    def create_layers(self, layer_activation: type, output_activation: type) -> None:
        for i, current_size in enumerate(self.shape):
            if i == len(self.shape) - 1:
                break
            next_size = self.shape[i + 1]
            weight_layer = torch.normal(0, np.sqrt(2 / current_size), (current_size, next_size), device=self.device)
            bias_layer = torch.normal(0, np.sqrt(2 / current_size), (1, next_size), device=self.device)
            self.weight_layers.append(weight_layer)
            self.bias_layers.append(bias_layer)
            final_activation = i == len(self.shape) - 2
            self.activation_functions.append(output_activation() if final_activation else layer_activation())

    def set_adam_parameters(self) -> None:
        self.adam_timestep = 0
        self.beta_1 = 0.9
        self.beta_2 = 0.999
        self.first_moment_weights = [torch.zeros_like(w) for w in self.weight_layers]
        self.first_moment_biases = [torch.zeros_like(b) for b in self.bias_layers]
        self.second_moment_weights = [torch.zeros_like(w) for w in self.weight_layers]
        self.second_moment_biases = [torch.zeros_like(b) for b in self.bias_layers]

    # ------------------------------------------------------------------ packing
    def _stream(self) -> int:
        return torch.cuda.current_stream(self._dev).cuda_stream

    def pack(self, weights: List[torch.Tensor], biases: List[torch.Tensor], out: torch.Tensor) -> torch.Tensor:
        """Reference-layout layers ((in,out) weights, (1,out) biases) -> packed vector (padding stays 0)."""
        for w, b, wi, bi in zip(weights, biases, self._widx, self._bidx):
            out[wi.reshape(-1)] = w.reshape(-1).to(out.dtype)
            out[bi.reshape(-1)] = b.reshape(-1).to(out.dtype)
        return out

    def unpack(self, packed: torch.Tensor) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        """Packed (..., P_pad) -> lists of (..., in, out) weights and (..., 1, out) biases."""
        return [packed[..., wi] for wi in self._widx], [packed[..., bi] for bi in self._bidx]

    def theta_packed(self) -> torch.Tensor:
        if self._theta_dirty:
            self.pack(self.weight_layers, self.bias_layers, self._theta)
            self._theta_dirty = False
        return self._theta

    def perturbations(self) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        """The stored UNIT perturbations in reference layout: (pairs, in, out) / (pairs, 1, out) f32 per layer.
        Env p < T/2 runs with layer + noise_std_dev * eps[p], env p + T/2 with layer - noise_std_dev * eps[p]."""
        return self.unpack(self._eps.float())

    def set_perturbations(self, eps_w: List[torch.Tensor], eps_b: List[torch.Tensor]) -> None:
        """Install caller-supplied unit perturbations (reference layout, see perturbations()); they are rounded to the
        fp16 storage.  For tests and for reproducing a run of the reference."""
        buf = torch.zeros((self.num_pairs, self.params_padded), dtype=torch.float32, device=self._dev)
        for w, b, wi, bi in zip(eps_w, eps_b, self._widx, self._bidx):
            buf[:, wi.reshape(-1)] = w.to(self._dev, torch.float32).reshape(self.num_pairs, -1)
            buf[:, bi.reshape(-1)] = b.to(self._dev, torch.float32).reshape(self.num_pairs, -1)
        self._eps.copy_(buf)
        self.perturbed = True

    # ------------------------------------------------------------------ forward (:84-109)
    def check_inputs(self, inputs) -> None:
        num_observations = self.shape[0]
        if tuple(inputs.shape) != (self.num_envs, num_observations):
            raise Exception(f"inputs to ParallelMLP must have shape {(self.num_envs, num_observations)}")

    def forward(self, inputs) -> torch.Tensor:
        """inputs: (num_envs, num_observations) float32 tensor, or a LazyObs handle from TimeSeriesEnv.step_lazy."""
        if not self.perturbed:
            raise RuntimeError("call perturb_parameters() first (the reference's forward reads perturbed_weights)")
        self.check_inputs(inputs)
        self.forward_calls += 1
        actions = torch.empty((self.num_envs, self.shape[-1]), dtype=torch.float32, device=self._dev)
        lazy = not torch.is_tensor(inputs)
        if lazy:
            obs_ptr, logret, row0, pf, W = None, inputs.logret, inputs.row0, inputs.posfeat, inputs.window
            if logret.dtype != torch.float32 or pf.dtype != torch.float32:
                raise TypeError("lazy observations must come from a float32 env")
            args = (None, logret.data_ptr(), row0.data_ptr(), pf.data_ptr(), W)
        else:
            if inputs.dtype != torch.float32 or not inputs.is_contiguous() or inputs.device != self._dev:
                inputs = inputs.to(device=self._dev, dtype=torch.float32).contiguous()
            args = (inputs.data_ptr(), None, None, None, 0)
        _lib.check(
            self._L.fe_es_forward(self._pnet, self.theta_packed().data_ptr(), self._eps.data_ptr(), float(self.noise_std_dev),
                                  self.num_envs, self.num_eval_envs, *args, float(self.action_noise_std), self.seed,
                                  self.forward_calls, self.env_id_base, actions.data_ptr(), self._dev.index, self._stream()),
            "fe_es_forward",
        )
        return actions

    def forward_kernel_name(self, lazy: bool = True, obs_aligned: bool = True) -> str:
        """Which fe_es_forward kernel `forward` launches for this network (and its launch shape); host-only.
        `obs_aligned`: a dense input starts on a 16-byte boundary (freshly allocated tensors do)."""
        return self._L.fe_es_forward_kernel_name(self._pnet, int(lazy), int(obs_aligned)).decode()

    # ------------------------------------------------------------------ perturbations (:112-174)
    def perturb_parameters(self) -> None:
        """:112-155 — new mirrored perturbations for every pair (a new `generation` of the keyed stream)."""
        self.generation += 1
        _lib.check(self._L.fe_es_perturb(self._pnet, self.seed, self.generation, self.pair_id_base, self.num_pairs,
                                         self._eps.data_ptr(), self._stream()), "fe_es_perturb")
        self.perturbed = True

    def reconstruct_perturbations(self) -> None:
        """:157-174 — nothing to do: the perturbations are stored as such, never added to the base parameters."""

    # ------------------------------------------------------------------ update (:176-275)
    def update_parameters(self, fitnesses: torch.Tensor) -> None:
        self.adam_timestep += 1
        half = self.num_training_envs // 2
        diffed = (fitnesses[0:half] - fitnesses[half: self.num_training_envs]).to(torch.float32).contiguous()
        _lib.check(self._L.fe_es_gradient(self._pnet, self._eps.data_ptr(), diffed.data_ptr(), self.num_pairs,
                                          self._scratch.data_ptr(), self._grad.data_ptr(), self._stream()), "fe_es_gradient")
        grad = self._grad
        if dist.is_initialized() and dist.get_world_size(self.group) > 1:
            dist.all_reduce(grad, op=dist.ReduceOp.SUM, group=self.group)
        # :204-207 mean over pairs of diff * (sigma*eps), divided by sigma == mean of diff * eps
        grad_w, grad_b = self.unpack(grad / float(self.total_pairs))
        for idx, (weight_layer, bias_layer) in enumerate(zip(self.weight_layers, self.bias_layers)):
            mean_weight_grad = grad_w[idx] - self.l2_coefficient * weight_layer   # :208
            mean_bias_grad = grad_b[idx] - self.l2_coefficient * bias_layer       # :209
            self.adam_update((weight_layer, bias_layer), (mean_weight_grad, mean_bias_grad), idx)
        self._theta_dirty = True
        self.perturbed = False   # :217-218 perturbed_weights = []

    def get_l2_norm(self) -> float:
        l2_norm = 0
        for weight_layer, bias_layer in zip(self.weight_layers, self.bias_layers):
            l2_norm += weight_layer.square().sum() + bias_layer.square().sum()
        return l2_norm.sqrt().item()

    def adam_update(self, layers: Tuple[torch.Tensor], grads: Tuple[torch.Tensor], idx: int) -> None:
        """:230-275, op for op."""
        assert len(layers) == 2, "layers passed to adam_update must be of the form (weight_layer, bias_layer)"
        assert len(grads) == 2, "grads passed to adam_update must be of the form (weight_grad, bias_grad)"
        t, alpha, beta_1, beta_2 = self.adam_timestep, self.learning_rate, self.beta_1, self.beta_2
        weight_layer, bias_layer = layers
        mean_weight_grad, mean_bias_grad = grads
        self.first_moment_weights[idx] = beta_1 * self.first_moment_weights[idx] + (1 - beta_1) * mean_weight_grad
        self.first_moment_biases[idx] = beta_1 * self.first_moment_biases[idx] + (1 - beta_1) * mean_bias_grad
        self.second_moment_weights[idx] = beta_2 * self.second_moment_weights[idx] + (1 - beta_2) * torch.square(mean_weight_grad)
        self.second_moment_biases[idx] = beta_2 * self.second_moment_biases[idx] + (1 - beta_2) * torch.square(mean_bias_grad)
        alpha_t = np.sqrt(1 - beta_2**t) / (1 - beta_1**t) * alpha
        weight_grad = alpha_t * torch.div(self.first_moment_weights[idx], torch.sqrt(self.second_moment_weights[idx]) + 10**-8)
        bias_grad = alpha_t * torch.div(self.first_moment_biases[idx], torch.sqrt(self.second_moment_biases[idx]) + 10**-8)
        weight_layer.add_(weight_grad)
        bias_layer.add_(bias_grad)
