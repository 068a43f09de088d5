"""
Hidden activations beyond ReLU / LeakyReLU(0.01) / Tanh: ELU (and CELU at alpha = 1), SELU, Sigmoid, Softplus, SiLU,
GELU (exact and tanh), Mish, through the module map, the C ABI, the forward-only GEMMs, both minibatch-step engines,
rollout sampling and checkpoints.  The expected values come from torch itself: its activation modules in float64 for
the forward, the float32 torch-CPU oracle (oracle/update.py, with these modules entered into its ACTIVATIONS table by
a fixture) for the update, and torch.distributions for sampling.

Bounds, with u = 2^-24 (the unit roundoff of float32):
  epilogue sweep   [1, H, H] nets make the pre-activation exactly z (FFMA: one FMA of 1 * z + 0, then an identity
                   layer whose sums are exact).  Each activation is a short float32 expression of at most ~6 roundings
                   and accurate libm calls (expf, expm1f, log1pf, erff, tanhf: <= 2 ulp each), written as torch's CUDA
                   kernels write it.  A relative error r in an intermediate reaches y through the activation's
                   condition number, so |y - ref| <= 8u (|y| + |z| m(z)), where m(z) is the sum of the absolute values
                   of the terms of act'(z) (terms that cancel in act'(z) do not cancel in the error).  GELU (both
                   forms) adds 1 + f with f = erf or tanh near -1: f's 2-ulp error is absolute there, <= 2^-23, and
                   0.5 z multiplies it: + 4u min(|z|, 8) for z < 0 (below z = -8 the float32 1 + f is exactly 0 and
                   |ref| < 1e-14).  Results below 2^-126 may flush or lose digits: + 2^-126.  tcgen05 adds the hi/lo
                   split of z and of h, 2^-22 (|y| + |z| m(z)), as test_forward_optim_kernels does.  The tensor-core
                   split cannot carry +-Inf or NaN (lo = x - hi), so non-finite z runs on FFMA only, each in its own
                   [1, 1, 1] net, and must give exactly torch's Inf or NaN.
  depth            the GEMM bound of test_forward_optim_kernels per layer plus the propagated input error; after an
                   activation e <- L e + the sweep bound at the pre-activation, L the activation's Lipschitz constant.
  update           status scalars and every parameter within the 1e-4 |ref| + 1e-6 of test_wide_heads.  lr follows
                   test_wide_heads._update_vs_oracle: 3e-4 for Discrete; 3e-5 for Box, whose log-probs in the tens
                   make Adam turn float32 gradient differences of small elements into a sizeable share of an lr step.
  gradients        the first minibatch's actor and critic gradients against the oracle run in float64, per tensor
                   within 1e-4 of its largest element, or 4 times the float32 oracle's own error where that is larger
                   (test_first_minibatch_gradients says where).
  sampling         Discrete: device and oracle probabilities differ by the forward rounding (~1e-6 relative), so a
                   row may sample differently only when its two largest p / q (q the Exp(1) draws) lie within 1e-4
                   relative; such rows are counted and at most 1 % of them may occur.  Box: raw actions within 1e-5.
"""
import ctypes as C
import glob
import math
import os
import shutil
import subprocess
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from helpers import run_device_rollout
from oracle import update as oracle_update
from oracle.update import OracleMLP, OracleUpdater

U = 2.0 ** -24
TINY = 2.0 ** -126

# name -> (torch module factory, float64/float32 torch function, Lipschitz constant)
NEW = OrderedDict([
    ("elu", (nn.ELU, F.elu, 1.0)),
    ("selu", (nn.SELU, F.selu, 1.0507009873554805 * 1.6732632423543772)),
    ("sigmoid", (nn.Sigmoid, torch.sigmoid, 0.25)),
    ("softplus", (nn.Softplus, F.softplus, 1.0)),
    ("silu", (nn.SiLU, F.silu, 1.1)),
    ("gelu", (nn.GELU, F.gelu, 1.13)),
    ("gelu_tanh", (lambda: nn.GELU(approximate="tanh"), lambda x: F.gelu(x, approximate="tanh"), 1.13)),
    ("mish", (nn.Mish, F.mish, 1.09)),
])
IDS = {"elu": 4, "selu": 5, "sigmoid": 6, "softplus": 7, "silu": 8, "gelu": 9, "gelu_tanh": 10, "mish": 11}
FROM_OUTPUT = ["elu", "selu", "sigmoid", "softplus"]
STORED = ["silu", "gelu", "gelu_tanh", "mish"]


@pytest.fixture(autouse=True)
def oracle_activations(monkeypatch):
    """The oracle's activation table, extended by the modules under test (the oracle file itself stays as it is)."""
    for name, (_, fn, _) in NEW.items():
        monkeypatch.setitem(oracle_update.ACTIVATIONS, name, fn)


# ---- float64 references -------------------------------------------------------------------------------------------
def ref64(z, name):
    return NEW[name][1](torch.as_tensor(np.asarray(z, np.float64))).numpy()


def deriv_terms64(z, name):
    """m(z): the sum of |terms| of act'(z) in float64 (module docstring)."""
    x = np.asarray(z, np.float64)
    with np.errstate(all="ignore"):
        if name == "elu":
            return np.where(x > 0, 1.0, np.exp(np.minimum(x, 0)))
        if name == "selu":
            return np.where(x > 0, 1.0507009873554805, 1.0507009873554805 * 1.6732632423543772 * np.exp(np.minimum(x, 0)))
        s = 1.0 / (1.0 + np.exp(-x))
        if name == "sigmoid":
            return s * (1 - s)
        if name == "softplus":
            return s
        if name == "silu":
            return s + np.abs(x) * s * (1 - s)
        if name == "gelu":
            return 0.5 * (1 + np.vectorize(math.erf)(x / math.sqrt(2))) + np.abs(x) * np.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
        if name == "gelu_tanh":
            b = math.sqrt(2 / math.pi)
            t = np.tanh(b * (x + 0.044715 * x ** 3))
            return 0.5 * (1 + t) + 0.5 * np.abs(x) * (1 - t * t) * b * (1 + 3 * 0.044715 * x * x)
        sp = np.logaddexp(0, x)
        t = np.tanh(sp)
        return np.abs(t) + np.abs(x) * s * (1 - t * t)


def act_bound(z, name, backend="ffma"):
    x = np.asarray(z, np.float64)
    y = ref64(x, name)
    with np.errstate(all="ignore"):
        scale = np.abs(y) + np.abs(x) * deriv_terms64(x, name)
        b = 8 * U * scale + TINY
        if name in ("gelu", "gelu_tanh"):
            b = b + np.where(x < 0, 4 * U * np.minimum(np.abs(x), 8.0), 0.0)
        if backend == "tcgen05":
            b = b + 2.0 ** -22 * scale
    return b


Z_MAG = (0.0, 1e-30, 1e-3, 1.0, 5.0, 20.0, 21.0, 88.0, 104.0, 1e30)
Z_FINITE = np.array([s * z for z in Z_MAG for s in (1.0, -1.0)], dtype=np.float32)
Z_SPECIAL = np.array([np.inf, -np.inf, np.nan], dtype=np.float32)


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_modules_map_to_their_ids_and_parameterised_variants_are_refused():
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.networks.feed_forward import activation_name
    accepted = [(nn.ELU(), "elu"), (nn.ELU(alpha=1.0), "elu"), (nn.CELU(), "elu"), (nn.SELU(), "selu"),
                (nn.Sigmoid(), "sigmoid"), (nn.Softplus(), "softplus"), (nn.Softplus(beta=1, threshold=20), "softplus"),
                (nn.SiLU(), "silu"), (nn.GELU(), "gelu"), (nn.GELU(approximate="tanh"), "gelu_tanh"),
                (nn.Mish(), "mish"), (nn.ReLU(), "relu"), (nn.LeakyReLU(), "leaky_relu"), (nn.Tanh(), "tanh")]
    for mod, name in accepted:
        assert activation_name(mod) == name, mod
        assert _lib.MlpDesc.make([3, 4, 2], activation_name(mod)).activation == _lib.ACT_IDS[name]
    for name, i in IDS.items():
        assert _lib.ACT_IDS[name] == i
    refused = [(nn.ELU(alpha=0.5), "alpha"), (nn.CELU(alpha=2.0), "alpha"), (nn.Softplus(beta=2), "beta"),
               (nn.Softplus(threshold=10), "threshold"), (nn.LeakyReLU(0.2), "slope"), (nn.Hardtanh(), "unsupported"),
               (nn.ReLU6(), "unsupported"), (nn.Softsign(), "unsupported")]
    for mod, word in refused:
        with pytest.raises(ValueError, match=word):
            activation_name(mod)


def test_act_ids_match_the_c_header(tmp_path):
    from ppo_and_friends_b200 import _lib
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = list(_lib.ACT_IDS)
    src = tmp_path / "acts.c"
    src.write_text('#include <stdio.h>\n#include "ppoaf_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("%d\\n", (int)PPOAF_ACT_{n.upper()});\n' for n in names)
                   + '  printf("%d\\n", (int)PPOAF_ACT_COUNT);\n  return 0;\n}\n')
    exe = tmp_path / "acts"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got[:-1] == [_lib.ACT_IDS[n] for n in names]
    assert got[-1] == len(names) == max(_lib.ACT_IDS.values()) + 1


def _lib_loaded():
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.build import build
    build()
    return _lib, _lib.load()


def test_unknown_activation_id_is_refused():
    _lib, lib = _lib_loaded()
    for act in (12, 99, -1):
        desc = _lib.MlpDesc.make([3, 4, 2], act)
        assert lib.ppoaf_mlp_forward(C.byref(desc), None, None, None, 1, 0, None, None, 0, None) != 0
        assert f"unknown activation id {act}" in lib.ppoaf_last_error().decode()
        cfg = _c4_cfg(act)
        assert lib.ppoaf_ppo_minibatch_grads(C.byref(cfg), C.byref(_lib.UpdateBufs()), None) != 0
        assert f"unknown activation id {act}" in lib.ppoaf_last_error().decode()
    desc = _lib.MlpDesc.make([3, 4, 2], 11)
    assert lib.ppoaf_param_layout(C.byref(desc), 0, None) > 0


def _c4_cfg(act):
    from ppo_and_friends_b200 import _lib
    cfg = _lib.UpdateCfg()
    cfg.actor = _lib.MlpDesc.make([376, 256, 256, 256, 17], act)
    cfg.critic = _lib.MlpDesc.make([376, 256, 256, 256, 1], act)
    cfg.head, cfg.act_dim, cfg.world_size, cfg.min_std = _lib.HEAD_GAUSSIAN_TANH, 17, 1, 0.01
    return cfg


def test_one_launch_engine_takes_the_derivative_from_output_ids_only():
    _lib, lib = _lib_loaded()
    assert lib.ppoaf_ppo_fused_supported(C.byref(_c4_cfg(3))) == 1                    # Tanh: the control
    for name in FROM_OUTPUT:
        assert lib.ppoaf_ppo_fused_supported(C.byref(_c4_cfg(IDS[name]))) == 1, name
    for name in STORED:
        assert lib.ppoaf_ppo_fused_supported(C.byref(_c4_cfg(IDS[name]))) == 0, name
        assert "activation needs a stored derivative" in lib.ppoaf_last_error().decode()


def test_stored_derivative_buffers_leave_other_workspaces_alone():
    """Only ids 8-11 grow the update's workspace: by one [B, hidden] buffer per hidden layer of each network."""
    _lib, lib = _lib_loaded()
    lib.ppoaf_update_workspace_bytes.restype = C.c_size_t
    B = 512
    base = lib.ppoaf_update_workspace_bytes(C.byref(_c4_cfg(3)), B)
    for name in FROM_OUTPUT + ["relu", "leaky_relu"]:
        assert lib.ppoaf_update_workspace_bytes(C.byref(_c4_cfg(_lib.ACT_IDS[name])), B) == base, name
    for name in STORED:
        assert lib.ppoaf_update_workspace_bytes(C.byref(_c4_cfg(IDS[name])), B) == base + 6 * B * 256 * 4, name


def test_sweep_bound_covers_float32_torch():
    """(CPU) the sweep bound holds for torch's own float32 CPU kernels at every finite z."""
    for name in NEW:
        ref = ref64(Z_FINITE, name)
        got = NEW[name][1](torch.from_numpy(Z_FINITE)).double().numpy()
        err = np.abs(got - ref)
        assert (err <= act_bound(Z_FINITE, name)).all(), (name, Z_FINITE[err > act_bound(Z_FINITE, name)])


# ---- GPU: forward -------------------------------------------------------------------------------------------------
def _net(dims, act, layers):
    from ppo_and_friends_b200 import _lib
    desc = _lib.MlpDesc.make(dims, act)
    offs, total = _lib.param_layout(desc)
    flat = torch.zeros(total)
    for l, (W, b) in enumerate(layers):
        flat[offs[2 * l]:offs[2 * l] + W.size] = torch.from_numpy(W.reshape(-1))
        flat[offs[2 * l + 1]:offs[2 * l + 1] + b.size] = torch.from_numpy(b)
    return desc, flat.cuda()


def _forward(backend, desc, params, x):
    from ppo_and_friends_b200 import ops
    ops.set_gemm_backend(backend)
    try:
        y = ops.mlp_forward(desc, params, x)
        torch.cuda.synchronize()
    finally:
        ops.set_gemm_backend("ffma")
    return y.cpu().numpy().astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["ffma", "tcgen05"])
@pytest.mark.parametrize("name", list(NEW))
def test_epilogue_sweep(backend, name):
    """[1, H, H] nets: layer 1 makes the pre-activation exactly z, layer 2 is the identity with zero bias."""
    H = Z_FINITE.size
    layers = [(Z_FINITE.reshape(H, 1).copy(), np.zeros(H, np.float32)), (np.eye(H, dtype=np.float32), np.zeros(H, np.float32))]
    desc, params = _net([1, H, H], name, layers)
    y = _forward(backend, desc, params, torch.ones(5, 1, device="cuda"))
    z = Z_FINITE.astype(np.float64)
    ref, bound = ref64(z, name), act_bound(z, name, backend)
    err = np.abs(y - ref)
    assert (err <= bound).all(), [(float(z[j]), float(y[0, j]), float(ref[j])) for j in np.nonzero((err > bound).any(0))[0]]
    print(f"{name} {backend}: worst err / bound {float(np.max(err / bound)):.3f}")
    if backend == "ffma":
        for zs in Z_SPECIAL:                                     # one [1, 1, 1] net each: no 0 * Inf in the identity layer
            desc, params = _net([1, 1, 1], name, [(np.array([[zs]], np.float32), np.zeros(1, np.float32)),
                                                  (np.ones((1, 1), np.float32), np.zeros(1, np.float32))])
            got = _forward("ffma", desc, params, torch.ones(3, 1, device="cuda"))
            want = float(np.float32(ref64(np.array([zs], np.float64), name)[0]))   # e.g. SELU(-Inf) = -float(lambda alpha)
            if math.isnan(want):
                assert np.isnan(got).all(), (name, zs, got)
            else:
                assert (got == want).all(), (name, zs, got, want)


DEPTH_DIMS = [[24, 96, 40, 7], [33, 130, 64, 65, 9]]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["ffma", "tcgen05"])
@pytest.mark.parametrize("name", list(NEW))
@pytest.mark.parametrize("dims", DEPTH_DIMS, ids=lambda d: "x".join(map(str, d)))
def test_random_nets_vs_float64(backend, name, dims):
    from test_forward_optim_kernels import gemm_bound
    rng = np.random.default_rng(len(dims) * 100 + IDS[name])
    layers = [((rng.standard_normal((dims[l + 1], dims[l])) * 1.5 / np.sqrt(dims[l])).astype(np.float32),
               (rng.standard_normal(dims[l + 1]) * 0.3).astype(np.float32)) for l in range(len(dims) - 1)]
    x = rng.standard_normal((300, dims[0])).astype(np.float32)
    desc, params = _net(dims, name, layers)
    y = _forward(backend, desc, params, torch.from_numpy(x).cuda())
    h, e = x.astype(np.float64), np.zeros((300, dims[0]))
    for l, (W, b) in enumerate(layers):
        W64, b64 = np.abs(W.astype(np.float64)), np.abs(b.astype(np.float64))
        pre = h @ W.astype(np.float64).T + b.astype(np.float64)
        e = gemm_bound(backend, dims[l], (np.abs(h) + e) @ W64.T + b64) + e @ W64.T
        if l + 1 < len(layers):
            h = ref64(pre, name)
            e = NEW[name][2] * e + act_bound(pre, name, backend)
        else:
            h = pre
    err = np.abs(y - h)
    assert (err <= e).all(), f"max err/bound {np.max(err / e):.3f}"
    print(f"{name} {backend} {dims}: worst err / bound {float(np.max(err / e)):.3f}")


# ---- GPU: the update ----------------------------------------------------------------------------------------------
def _rollout(n_actions, box_dim, seed):
    from ppo_and_friends_b200.synthetic import make_rollout
    return make_rollout(seed=seed, T=32, E=16, obs_dim=12, act_dim=box_dim or 2, n_discrete=n_actions,
                        max_ts_per_ep=12, obs_scale=False)


def _policy(ro, name, hidden, **policy_kw):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.spaces import Box, Discrete
    space = Discrete(ro.n_discrete) if ro.n_discrete else Box(-1.0, 1.0, (ro.act_dim,))
    pol = PPOPolicy("pol", space, Box(-np.inf, np.inf, (ro.obs_dim,)), Box(-np.inf, np.inf, (ro.critic_obs_dim,)),
                    envs_per_proc=ro.E,
                    actor_kw_args=dict(activation=NEW[name][0](), hidden_size=hidden, hidden_depth=3),
                    critic_kw_args=dict(activation=NEW[name][0](), hidden_size=hidden, hidden_depth=3), **policy_kw)
    for a in ro.agents:
        pol.register_agent(a)
    pol.agent_ids = np.array(ro.agents)
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device("cuda"))
    return pol


def _fill_old_outputs(pol, ro):
    with torch.no_grad():
        for a in ro.agents:
            obs = ro.obs[a].reshape(ro.T * ro.E, -1)
            cobs = ro.critic_obs[a].reshape(ro.T * ro.E, -1)
            values, lp, _ = pol.evaluate(cobs, obs, ro.raw_actions[a].reshape(ro.T * ro.E, -1))
            ro.log_probs[a] = lp.cpu().numpy().reshape(ro.T, ro.E)
            ro.values[a] = values.cpu().numpy().reshape(ro.T, ro.E)


def _host(ds):
    return {k: getattr(ds, k).cpu().numpy().copy() for k in (
        "critic_observations", "observations", "raw_actions", "advantages", "log_probs", "rewards_to_go", "values")}


SPACES = {"Discrete(5)": (5, 0), "Box(17)": (0, 17)}
SHAPES = {"h256-fused-heads": dict(hidden=256), "h512-chain": dict(hidden=512),
          "h64-vf-clip": dict(hidden=64, vf_clip=0.5, use_huber_loss=True)}


def _update_vs_oracle(name, space, shape, engine, use_graphs, monkeypatch):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    monkeypatch.setenv("PPOAF_STEP", engine)
    monkeypatch.setenv("PPOAF_NO_GRAPH", "0" if use_graphs else "1")
    n_actions, box_dim = SPACES[space]
    kw = dict(SHAPES[shape])
    hidden = kw.pop("hidden")
    lr = 3e-4 if n_actions else 3e-5
    ro = _rollout(n_actions, box_dim, seed=17 + IDS[name])
    torch.manual_seed(5)
    pol = _policy(ro, name, hidden, lr=lr, **kw)
    _fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    host = _host(ds)
    oracle = OracleUpdater({n: v.cpu().numpy() for n, v in pol.actor.state_dict().items()},
                           {n: v.cpu().numpy() for n, v in pol.critic.state_dict().items()}, name, bool(n_actions),
                           lr=lr, vf_clip=kw.get("vf_clip"), use_huber_loss=kw.get("use_huber_loss", False))
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    torch.manual_seed(11)
    ppo_batch_train(state, _Loader(ds, 128), "pol")
    st = oracle.batch_train([host], [pol._engine._perm_dev.cpu().numpy()], 128)
    sd = state.status_dict["pol"]
    keys = ("actor loss", "critic loss", "kl avg", "weighted entropy")
    got, ref = np.array([sd[k] for k in keys]), np.array([st[k] for k in keys])
    # test_wide_heads' bound: the actor loss and KL carry a few 2^-24 |log-prob| of float32 rounding
    bound = 1e-4 * np.maximum(np.abs(ref), 1e-3) + np.array([1, 0, 1, 0]) * 2.0 ** -21 * float(np.abs(host["log_probs"]).mean())
    assert bool((np.abs(got - ref) <= bound).all()), (got, ref, bound)
    ref_state = oracle.state()
    for net, obj in (("actor", pol.actor), ("critic", pol.critic)):
        for k, v in obj.state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref_state[f"{net}/param/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
    np.testing.assert_allclose(ds.values.cpu().numpy(), host["values"], rtol=1e-4, atol=1e-5)
    return pol


def _fusable(name, shape):
    return shape == "h256-fused-heads" and name in FROM_OUTPUT


@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False], ids=["graphs", "no-graphs"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("space", list(SPACES))
@pytest.mark.parametrize("name", list(NEW))
def test_update_vs_oracle_chain(name, space, shape, use_graphs, monkeypatch):
    """The launch chain: fused head layers (h256), the 10-launch chain (h512, value clipping)."""
    pol = _update_vs_oracle(name, space, shape, "chain", use_graphs, monkeypatch)
    assert not pol._engine.fused


@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False], ids=["graphs", "no-graphs"])
@pytest.mark.parametrize("space", list(SPACES))
@pytest.mark.parametrize("name", FROM_OUTPUT)
def test_update_vs_oracle_one_launch_engine(name, space, use_graphs, monkeypatch):
    pol = _update_vs_oracle(name, space, "h256-fused-heads", "fused", use_graphs, monkeypatch)
    assert pol._engine.fused


@pytest.mark.gpu
@pytest.mark.parametrize("space", list(SPACES))
@pytest.mark.parametrize("name", STORED)
def test_one_launch_request_runs_the_chain_for_stored_derivatives(name, space, monkeypatch):
    chain = _update_vs_oracle(name, space, "h256-fused-heads", "chain", True, monkeypatch)
    fused = _update_vs_oracle(name, space, "h256-fused-heads", "fused", True, monkeypatch)
    assert not fused._engine.fused
    assert torch.equal(chain.nets.flat_params, fused.nets.flat_params)


class _FirstGradients(OracleUpdater):
    """OracleUpdater that keeps the actor and critic gradients of its first minibatch (before clipping).  in_float64:
    the same minibatch with the parameters and dataset in float64; it records the gradients and takes no step."""

    def __init__(self, actor_params, critic_params, activation, in_float64=False):
        super().__init__(actor_params, critic_params, activation, True)
        self.in_float64 = in_float64
        if in_float64:
            for mlp in (self.actor, self.critic):
                mlp.p = {k: v.detach().double().requires_grad_() for k, v in mlp.p.items()}

    def _clip_and_step(self, which, params, grads_override=None):
        if not hasattr(self, "first_" + which):
            setattr(self, "first_" + which, [g.clone() for g in (grads_override or [q.grad for q in params])])
        if not self.in_float64:
            super()._clip_and_step(which, params, grads_override)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["h256-fused-heads", "h512-chain"])
@pytest.mark.parametrize("name", list(NEW))
def test_first_minibatch_gradients(name, shape, monkeypatch):
    """One minibatch of all 512 rows: every actor and critic gradient tensor against the oracle's autograd.  At h256
    the heads' dX comes from the loss kernel, at h512 from a backward-x GEMM; both multiply by act'(z).

    Each tensor's error is taken against the oracle in float64, as a share of its largest element: at most 1e-4, or
    4 times the float32 oracle's own error where that is larger.  Orthogonal init with gain sqrt(2) makes some nets
    ill-conditioned in float32: with SELU at 512 wide, float32 torch's hidden-layer weight gradients are 2e-3 to 9e-3
    of their largest element away from float64, so no float32 summation order meets 1e-4 there."""
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    monkeypatch.setenv("PPOAF_STEP", "chain")
    ro = _rollout(5, 0, seed=29 + IDS[name])
    torch.manual_seed(5)
    pol = _policy(ro, name, SHAPES[shape]["hidden"])
    _fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    host = _host(ds)
    params = ({n: v.cpu().numpy() for n, v in pol.actor.state_dict().items()},
              {n: v.cpu().numpy() for n, v in pol.critic.state_dict().items()})
    n = len(ds)
    torch.manual_seed(11)
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=n, epochs_per_iter=1), _Loader(ds, n), "pol")
    perm = pol._engine._perm_dev.cpu().numpy()
    o32 = _FirstGradients(*params, name)
    o32.batch_train([host], [perm], n)
    o64 = _FirstGradients(*params, name, in_float64=True)
    o64.batch_train([{k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in host.items()}], [perm], n)
    worst = 0.0
    for net, refs32, refs64 in ((pol.actor, o32.first_actor, o64.first_actor),
                                (pol.critic, o32.first_critic, o64.first_critic)):
        got = net.grad_dict()
        assert len(got) == len(refs32) == len(refs64)
        for (k, g), r32, r64 in zip(got.items(), refs32, refs64):
            g = g.detach().cpu().double()
            r32, r64 = r32.detach().double().reshape(g.shape), r64.detach().double().reshape(g.shape)
            scale = float(r64.abs().max())
            err, err32 = float((g - r64).abs().max()) / scale, float((r32 - r64).abs().max()) / scale
            assert err <= max(1e-4, 4 * err32), (net.name, k, err, err32)
            worst = max(worst, err)
    print(f"{name} {shape}: worst gradient error / largest element {worst:.2e}")


# ---- GPU: rollout and checkpoints ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("space", list(SPACES))
@pytest.mark.parametrize("name", list(NEW))
def test_rollout_actions_match_torch_distributions(name, space):
    from torch.distributions import Categorical
    n_actions, box_dim = SPACES[space]
    ro = _rollout(n_actions, box_dim, seed=41 + IDS[name])
    ro_obs = ro.obs[ro.agents[0]][0]
    torch.manual_seed(4)
    pol = _policy(ro, name, 64)
    oracle = OracleMLP({k: v.cpu().numpy() for k, v in pol.actor.state_dict().items() if k != "distribution.log_std"},
                       name)
    with torch.no_grad():
        pred = oracle.forward(torch.as_tensor(ro_obs))
    torch.manual_seed(123)
    raw, act, lp = pol.get_rollout_actions(ro_obs)
    torch.manual_seed(123)
    if n_actions:
        probs = torch.softmax(pred, -1)
        want = Categorical(probs=probs).sample().numpy()
        torch.manual_seed(123)
        q = torch.empty(probs.shape).exponential_(1).double()
        v = probs.double() / q
        top = torch.topk(v, 2, dim=1).values
        exempt = ((top[:, 0] - top[:, 1]) <= 1e-4 * top[:, 0]).numpy()
        act = np.asarray(act).reshape(-1)
        assert np.array_equal(act[~exempt], want[~exempt])
        assert exempt.sum() <= max(1, len(want) // 100)
    else:
        from oracle.update import gaussian_std
        std = gaussian_std(pol.actor.state_dict()["distribution.log_std"].cpu(), pol.min_std)
        want = torch.empty(pred.shape).normal_(0, 1).mul_(std).add_(pred)
        np.testing.assert_allclose(raw, want.numpy(), rtol=1e-5, atol=1e-5)


class _Reference(nn.Module):
    """The reference FeedForwardNetwork's Sequential layout (networks/utils.py:160-183), depth 3."""

    def __init__(self, dims, module):
        super().__init__()
        self.sequential_net = nn.Sequential(nn.Linear(dims[0], dims[1]), module(),
                                            nn.Sequential(nn.Linear(dims[1], dims[2]), module(),
                                                          nn.Linear(dims[2], dims[3]), module()),
                                            nn.Linear(dims[3], dims[4]))

    def forward(self, x):
        return self.sequential_net(x)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NEW))
def test_checkpoint_round_trip_and_reference_layout(name, tmp_path):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    ro = _rollout(0, 17, seed=53 + IDS[name])
    torch.manual_seed(2)
    pol = _policy(ro, name, 32)
    ds = run_device_rollout(pol, ro)
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1), _Loader(ds, 128), "pol")
    pol.save(str(tmp_path))
    files = glob.glob(os.path.join(str(tmp_path), "**", "actor_0.model"), recursive=True)
    assert len(files) == 1
    sd = torch.load(files[0])
    ref = _Reference(pol.actor.dims, NEW[name][0])
    ref.load_state_dict({k: v for k, v in sd.items() if k != "distribution.log_std"}, strict=True)
    obs = torch.as_tensor(ro.obs[ro.agents[0]][0])
    with torch.no_grad():
        want = ref(obs)
    got = pol.actor(obs.cuda()).cpu()
    np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=1e-5, atol=1e-6)
    torch.manual_seed(3)
    fresh = _policy(ro, name, 32)
    assert not torch.equal(fresh.nets.flat_params, pol.nets.flat_params)
    fresh.load(str(tmp_path))
    for k in ("flat_params", "adam_m", "adam_v", "adam_step"):
        assert torch.equal(getattr(fresh.nets, k), getattr(pol.nets, k)), k
    assert int(fresh.nets.adam_step.item()) > 0
