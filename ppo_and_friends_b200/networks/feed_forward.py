"""
Actor / critic feed-forward networks as views into ONE flat device buffer per policy.

Mirrors the structure the reference builds with torch.nn (networks/ppo_networks/feed_forward.py:14-86,
networks/utils.py:53-80, 114-191, networks/actor_critic/wrappers.py:10-82): Linear(in,h) -> act ->
[Linear(h,h) -> act] x (depth-1) -> Linear(h,out); orthogonal init with gain sqrt(2), output gain
0.01 (actor) / 1.0 (critic), zero biases; the Gaussian actor owns `distribution.log_std`.
state_dict() keys are the reference's (`sequential_net.0.*`, `sequential_net.2.{0,2,..}.*`,
`sequential_net.3.*`, `distribution.log_std`), so reference checkpoints load and vice versa.

The flat layout [actor | critic] (params, grads, Adam m, Adam v share it) is what the CUDA step and
the NCCL all-reduce operate on: one gradient all-reduce per minibatch instead of one per tensor.
"""
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

from .. import _lib, ops

_ACT_NAMES = {nn.ReLU: "relu", nn.LeakyReLU: "leaky_relu", nn.Tanh: "tanh", nn.Identity: "identity", nn.ELU: "elu",
              nn.CELU: "elu", nn.SELU: "selu", nn.Sigmoid: "sigmoid", nn.Softplus: "softplus", nn.SiLU: "silu",
              nn.Mish: "mish"}
_SUPPORTED = ("ReLU, LeakyReLU(0.01), Tanh, ELU(alpha=1), CELU(alpha=1), SELU, Sigmoid, Softplus(beta=1, threshold=20), "
              "SiLU, GELU('none' or 'tanh'), Mish")


def activation_name(activation):
    """Map a torch activation instance (the reference passes module instances) or a string.  The kernels carry no
    activation parameter, so a module whose parameter differs from the one value they implement is refused."""
    if isinstance(activation, str):
        if activation not in _lib.ACT_IDS:
            raise ValueError(f"unsupported activation {activation}")
        return activation
    if isinstance(activation, nn.GELU):
        if activation.approximate not in ("none", "tanh"):
            raise ValueError(f"GELU approximate={activation.approximate!r} is not supported (supported: 'none', 'tanh')")
        return "gelu" if activation.approximate == "none" else "gelu_tanh"
    for cls, name in _ACT_NAMES.items():
        if isinstance(activation, cls):
            if cls is nn.LeakyReLU and abs(activation.negative_slope - 0.01) > 1e-12:
                raise ValueError("LeakyReLU slope other than 0.01 is not supported by the CUDA path")
            if cls in (nn.ELU, nn.CELU) and activation.alpha != 1.0:
                raise ValueError(f"{cls.__name__} alpha={activation.alpha} is not supported by the CUDA path "
                                 "(supported: alpha=1.0)")
            if cls is nn.Softplus and (activation.beta != 1.0 or activation.threshold != 20.0):
                raise ValueError(f"Softplus beta={activation.beta}, threshold={activation.threshold} is not supported "
                                 "by the CUDA path (supported: beta=1.0, threshold=20.0)")
            return name
    raise ValueError(f"unsupported activation {activation!r} (supported: {_SUPPORTED})")


def hidden_sizes(hidden_size, hidden_depth):
    """networks/utils.py:140-158."""
    if not isinstance(hidden_size, list):
        if (hidden_size == 0) != (hidden_depth == 0):
            raise ValueError("if either hidden_size or hidden_depth is 0, both must be 0")
        return [hidden_size] * hidden_depth
    return list(hidden_size)


def layer_key_stems(n_hidden):
    if n_hidden == 0:
        return ["sequential_net.0"]
    return (["sequential_net.0"] + [f"sequential_net.2.{2 * i}" for i in range(n_hidden - 1)]
            + ["sequential_net.3"])


def reference_init(dims, out_gain):
    """Host-side initialisation in the reference's construction order (so a given torch seed
    yields the same weights): nn.Linear's own reset, then orthogonal_/constant_ (networks/utils.py:53-80)."""
    layers = []
    n = len(dims) - 1
    for l in range(n):
        lin = nn.Linear(dims[l], dims[l + 1])
        gain = np.sqrt(2) if (l + 1 < n or out_gain is None) else out_gain
        nn.init.orthogonal_(lin.weight, gain)
        nn.init.constant_(lin.bias, 0.0)
        layers.append((lin.weight.detach().clone(), lin.bias.detach().clone()))
    return layers


class FlatNetwork:
    """One MLP living at [base, base + total) of the policy's flat buffers."""

    def __init__(self, name, dims, activation, log_std_dim=0):
        self.name = name
        self.dims = [int(d) for d in dims]
        self.activation = activation_name(activation)
        self.desc = _lib.MlpDesc.make(self.dims, self.activation)
        self.log_std_dim = int(log_std_dim)
        self.offsets, self.total = _lib.param_layout(self.desc, self.log_std_dim)
        self.stems = layer_key_stems(len(self.dims) - 2)
        self.base = 0
        self.owner = None

    def bind(self, owner, base):
        self.owner, self.base = owner, base

    def _views(self, flat):
        out = OrderedDict()
        n = len(self.dims) - 1
        for l in range(n):
            w0 = self.base + self.offsets[2 * l]
            b0 = self.base + self.offsets[2 * l + 1]
            out[self.stems[l] + ".weight"] = flat[w0:w0 + self.dims[l] * self.dims[l + 1]].view(self.dims[l + 1], self.dims[l])
            out[self.stems[l] + ".bias"] = flat[b0:b0 + self.dims[l + 1]]
        if self.log_std_dim:
            s0 = self.base + self.offsets[2 * n]
            out["distribution.log_std"] = flat[s0:s0 + self.log_std_dim]
        return out

    def state_dict(self):
        return self._views(self.owner.flat_params)

    def grad_dict(self):
        return self._views(self.owner.flat_grads)

    def adam_dicts(self):
        return self._views(self.owner.adam_m), self._views(self.owner.adam_v)

    def parameters(self):
        return list(self.state_dict().values())

    def load_state_dict(self, sd):
        mine = self.state_dict()
        missing = [k for k in mine if k not in sd]
        if missing:
            raise KeyError(f"{self.name}: missing keys {missing}")
        with torch.no_grad():
            for k, v in mine.items():
                v.copy_(torch.as_tensor(np.asarray(sd[k].detach().cpu() if torch.is_tensor(sd[k]) else sd[k]),
                                        dtype=torch.float32).reshape(v.shape))

    @property
    def flat(self):
        return self.owner.flat_params[self.base:self.base + self.total]

    def __call__(self, obs, softmax_out=False):
        """Forward through the CUDA MLP kernels; obs: [n, in] fp32 (numpy or tensor)."""
        x = obs if torch.is_tensor(obs) else torch.as_tensor(np.ascontiguousarray(obs))
        x = x.to(device=self.owner.device, dtype=torch.float32).reshape(x.shape[0], -1).contiguous()
        return ops.mlp_forward(self.desc, self.flat, x, softmax_out=softmax_out)

    def save(self, path, rank=0):
        import os
        torch.save(OrderedDict((k, v.detach().cpu().clone()) for k, v in self.state_dict().items()),
                   os.path.join(path, "{}_{}.model".format(self.name, rank)))

    def load(self, path, rank=0):
        import os
        f = os.path.join(path, "{}_{}.model".format(self.name, rank))
        if not os.path.exists(f):
            f = os.path.join(path, "{}_0.model".format(self.name))
        self.load_state_dict(torch.load(f))


class PolicyNetworks:
    """Flat [actor | critic] parameter / gradient / Adam buffers of one policy."""

    def __init__(self, device, actor_dims, critic_dims, actor_activation, critic_activation, gaussian, act_dim,
                 std_offset=0.5, init=True):
        self.device = torch.device(device)
        self.actor = FlatNetwork("actor", actor_dims, actor_activation, act_dim if gaussian else 0)
        self.critic = FlatNetwork("critic", critic_dims, critic_activation, 0)
        self.n_actor, self.n_critic = self.actor.total, self.critic.total
        n = self.n_actor + self.n_critic
        self.flat_params = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.flat_grads = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.adam_m = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.adam_v = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.adam_step = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.actor.bind(self, 0)
        self.critic.bind(self, self.n_actor)
        if init:
            # actor first, then critic: the reference's construction order (ppo_policy.py:433-446)
            a_layers = reference_init(actor_dims, 0.01)
            c_layers = reference_init(critic_dims, 1.0)
            sd = OrderedDict()
            for stem, (w, b) in zip(self.actor.stems, a_layers):
                sd[stem + ".weight"], sd[stem + ".bias"] = w, b
            if gaussian:
                sd["distribution.log_std"] = torch.full((act_dim,), -float(std_offset))
            self.actor.load_state_dict(sd)
            sd = OrderedDict()
            for stem, (w, b) in zip(self.critic.stems, c_layers):
                sd[stem + ".weight"], sd[stem + ".bias"] = w, b
            self.critic.load_state_dict(sd)


class _AdamView:
    """
    torch.optim.Adam's surface as the trainer and the checkpoints use it (`param_groups[i]['lr']`, `state_dict()`,
    `load_state_dict()`), over the flat device buffers of one network.  The state dict has torch's layout
    (`state[i] = {step, exp_avg, exp_avg_sq}` in `named_parameters()` order, one param group), so files written by the
    reference's `torch.save(self.actor_optim.state_dict(), ...)` (policies/ppo_policy.py:1228-1247) load here and the
    files written here load into a real `torch.optim.Adam`.
    """

    def __init__(self, lr, net=None):
        self.net = net
        self.param_groups = [dict(lr=lr, betas=(0.9, 0.999), eps=1e-5)]

    def state_dict(self):
        m, v = self.net.adam_dicts()
        step = float(self.net.owner.adam_step.item())
        state = {}
        if step > 0:                                   # torch creates the per-parameter state at the first step
            for i, k in enumerate(m):
                state[i] = dict(step=torch.tensor(step, dtype=torch.float32), exp_avg=m[k].detach().cpu().clone(),
                                exp_avg_sq=v[k].detach().cpu().clone())
        g = self.param_groups[0]
        group = dict(lr=g["lr"], betas=tuple(g["betas"]), eps=g["eps"], weight_decay=0, amsgrad=False, maximize=False,
                     foreach=None, capturable=False, differentiable=False, fused=None, decoupled_weight_decay=False,
                     params=list(range(len(m))))
        return dict(state=state, param_groups=[group])

    def load_state_dict(self, sd):
        m, v = self.net.adam_dicts()
        keys = list(m.keys())
        state = sd.get("state", {})
        steps = set()
        with torch.no_grad():
            for i, k in enumerate(keys):
                st = state.get(i, state.get(str(i)))
                if st is None:
                    m[k].zero_(); v[k].zero_()
                    continue
                m[k].copy_(torch.as_tensor(st["exp_avg"]).to(m[k].device, torch.float32).reshape(m[k].shape))
                v[k].copy_(torch.as_tensor(st["exp_avg_sq"]).to(v[k].device, torch.float32).reshape(v[k].shape))
                steps.add(int(round(float(st["step"]))))
        if len(steps) > 1:
            raise ValueError(f"{self.net.name}: parameters with different Adam step counts {sorted(steps)} cannot be "
                             "represented (the fused optimizer keeps one step counter)")
        step = steps.pop() if steps else 0
        owner = self.net.owner
        if getattr(owner, "_loaded_adam_step", None) not in (None, step):
            raise ValueError("actor and critic optimizers were saved at different step counts "
                             f"({owner._loaded_adam_step} vs {step}); the fused optimizer keeps one step counter")
        owner._loaded_adam_step = step
        owner.adam_step.fill_(step)
        groups = sd.get("param_groups") or [{}]
        for key in ("lr", "betas", "eps"):
            if key in groups[0]:
                self.param_groups[0][key] = groups[0][key]
