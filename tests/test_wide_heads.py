"""
Discrete and Box action spaces wider than 64 actor outputs: the wide Categorical and Gaussian-tanh kernels through the C
ABI, the update (against the float32 torch-CPU oracle), rollout sampling, inference and checkpoints.

Discrete(n <= 64) keeps the one-section multi-categorical route; Discrete(65 .. 65536) and Box(65 .. 4096 flattened dims)
take the wide kernels.  The expected values come from oracle/update.py (softmax + Categorical(probs), the Gaussian-tanh
log-prob) and torch.distributions, which have no width limit.
"""
import ctypes as C

import numpy as np
import pytest
import torch
from torch.distributions import Categorical

from helpers import make_policy, run_device_rollout
from oracle.update import OracleUpdater, categorical_from_probs, gaussian_std, gaussian_tanh_log_prob
from ppo_and_friends_b200.spaces import Box, Discrete, MultiBinary, MultiDiscrete


# ----------------------------------------------------------------------------------------- CPU
def _policy(action_space):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    return PPOPolicy("pol", action_space, Box(-1, 1, (4,)), Box(-1, 1, (4,)), envs_per_proc=2)


def test_policy_accepts_and_refuses_wide_spaces():
    from ppo_and_friends_b200 import _lib
    for n in (65, 4672, 65536):
        pol = _policy(Discrete(n))
        assert (pol.action_dtype, pol.action_dim, pol.action_pred_size) == ("discrete", 1, n)
        assert pol.head == _lib.HEAD_CATEGORICAL and pol.wide_categorical
        assert not hasattr(pol, "section_ends")                       # no table wider than 64 bits is formed
    assert not _policy(Discrete(64)).wide_categorical and _policy(Discrete(64)).section_ends == 1 << 63
    for shape, d in (((65,), 65), ((8, 16), 128), ((4096,), 4096)):
        pol = _policy(Box(-1, 1, shape))
        assert (pol.action_dtype, pol.action_dim, pol.action_pred_size) == ("continuous", d, d)
        assert pol.head == _lib.HEAD_GAUSSIAN_TANH
    for bad, words in ((Discrete(65537), "65536"), (Discrete(0), "Discrete"), (Box(-1, 1, (4097,)), "4096"),
                       (Box(-1, 1, (64, 65)), "4096"), (MultiDiscrete([40, 25]), "64"), (MultiBinary(65), "64")):
        with pytest.raises(RuntimeError, match=words):
            _policy(bad)


def _cfg(head, pred, act_dim, ends=0):
    from ppo_and_friends_b200 import _lib
    cfg = _lib.UpdateCfg()
    cfg.actor = _lib.MlpDesc.make([6, 16, 16, pred], "tanh")
    cfg.critic = _lib.MlpDesc.make([6, 16, 16, 1], "tanh")
    cfg.head, cfg.act_dim = head, act_dim
    cfg.section_ends[0], cfg.section_ends[1] = ends & 0xFFFFFFFF, ends >> 32
    return cfg


def test_wide_widths_through_the_c_abi_with_required_outputs():
    """In-bound wide Categorical / Gaussian widths pass the width checks of the update and head entry points (with
    empty buffers the update calls are then refused for another reason; zero-row head calls given log_std and their
    required outputs return without launching).
    Wider rows, and Bernoulli / multi-categorical rows above 64, are refused with a message naming the width."""
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.build import build
    build()
    lib = _lib.load()
    bufs = _lib.UpdateBufs()
    msg = lambda: lib.ppoaf_last_error().decode()
    CAT, GAUSS, BERN, MULTI = (_lib.HEAD_CATEGORICAL, _lib.HEAD_GAUSSIAN_TANH, _lib.HEAD_BERNOULLI,
                               _lib.HEAD_MULTI_CATEGORICAL)
    ok = [(CAT, 65, 1), (CAT, 4672, 1), (CAT, 65536, 1), (GAUSS, 65, 65), (GAUSS, 4096, 4096)]
    bad = [(CAT, 65537, 1, 0), (GAUSS, 4097, 4097, 0), (BERN, 65, 65, 0), (MULTI, 65, 2, (1 << 63) | 1)]
    for fn in ("ppoaf_ppo_minibatch_grads", "ppoaf_ppo_fused_steps"):
        args = (C.byref(bufs), 1, None) if fn == "ppoaf_ppo_fused_steps" else (C.byref(bufs), None)
        for head, pred, act_dim in ok:
            assert getattr(lib, fn)(C.byref(_cfg(head, pred, act_dim)), *args) != 0      # refused, but later
            assert "head width" not in msg() and "output width" not in msg(), (fn, head, pred, msg())
        for head, pred, act_dim, ends in bad:
            assert getattr(lib, fn)(C.byref(_cfg(head, pred, act_dim, ends)), *args) != 0
            assert f"head width {pred}" in msg(), (fn, head, pred, msg())
    for head, pred, act_dim in ok:
        assert lib.ppoaf_ppo_fused_supported(C.byref(_cfg(head, pred, act_dim))) == 0
    fake = C.c_void_p(16)                                                        # never dereferenced: zero rows
    for head, pred, act_dim in ok:
        log_std = fake if head == GAUSS else None
        assert lib.ppoaf_head_evaluate(head, None, pred, log_std, 0.01, None, act_dim, 0, fake, None, None) == 0, msg()
        assert lib.ppoaf_head_sample(head, None, pred, log_std, 0.01, fake, None, None, act_dim, 0, fake, fake, fake,
                                     None) == 0, msg()
    for head, pred, act_dim, _ in bad[:3]:
        assert lib.ppoaf_head_evaluate(head, None, pred, None, 0.01, None, act_dim, 0, None, None, None) != 0
        assert "head width" in msg(), msg()
        assert lib.ppoaf_head_sample(head, None, pred, None, 0.01, fake, None, None, act_dim, 0, None, None, None,
                                     None) != 0
        assert "head width" in msg(), msg()


# ----------------------------------------------------------------------------------------- GPU: evaluation
@pytest.mark.gpu
@pytest.mark.parametrize("P", [65, 97, 362, 4672, 65536])
def test_categorical_evaluate_vs_oracle(P):
    """Against softmax + Categorical(probs) in float64, at the 1e-5 of the narrow tests."""
    from ppo_and_friends_b200 import _lib, ops
    torch.manual_seed(P)
    n = 64 if P == 65536 else 300
    logits = torch.randn(n, P) * 3
    logits[torch.arange(20), torch.randint(0, P, (20,))] += 60.0      # one dominant logit: the others' pn < eps
    acts = torch.randint(0, P, (n, 1))
    acts[:10, 0] = logits[:10].argmax(dim=1)                         # the dominant class: pn > 1 - eps
    # the oracle's formulas, evaluated in float64 (the float32 clamp bounds kept)
    p, lg = categorical_from_probs(torch.softmax(logits.double(), dim=-1))
    lg = torch.log(torch.clamp(p, 1.1920928955078125e-07, 1 - 1.1920928955078125e-07))
    assert bool((p[:20] < 1.2e-7).any()) and bool((p[:10].max(dim=1).values > 1 - 1.2e-7).all())
    ref_lp = lg.gather(1, acts).reshape(-1)
    ref_ent = -(p * lg).sum(dim=-1)
    assert torch.allclose(ref_lp.float(), Categorical(probs=torch.softmax(logits, -1)).log_prob(acts[:, 0]), atol=1e-5)
    lp, ent = ops.head_evaluate(_lib.HEAD_CATEGORICAL, logits.cuda(), None, acts.cuda())
    np.testing.assert_allclose(lp.cpu().numpy(), ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ent.cpu().numpy(), ref_ent.numpy(), rtol=1e-5, atol=1e-5)


def _gaussian_terms(mean, std, x):
    """Per row, the sum of |terms| of the Gaussian-tanh log-prob: two fp32 sums of these terms in different orders
    differ by a few 2^-24 of it, however much of it cancels."""
    var = std * std
    nl = torch.clamp(-((x - mean) ** 2) / (2 * var) - torch.log(std) - 0.9189385332046727, -100, 100)
    return (nl.abs() + torch.log(torch.clamp(1.0 - torch.tanh(x) ** 2, min=1e-6)).abs()).sum(dim=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [65, 200, 4096])
def test_gaussian_evaluate_vs_oracle(d):
    """Against the float32 oracle at 1e-5, plus 2^-20 of the row's sum of |terms|: rows whose large terms (min_std =
    0.01 dimensions) cancel to a small log-prob keep that much of fp32 summation-order difference."""
    from ppo_and_friends_b200 import _lib, ops
    torch.manual_seed(d)
    n = 300
    mean = torch.randn(n, d)
    log_std = torch.randn(d) * 0.5 - 0.5
    log_std[:3] = torch.tensor([-30.0, 25.0, -5.0])                   # min_std binds; softplus passes through
    std = gaussian_std(log_std)
    acts = mean + std * torch.randn(n, d) * 2
    acts[:5, :7] = 12.0                                               # tanh saturates: the 1e-6 clamp binds
    lp, ent = ops.head_evaluate(_lib.HEAD_GAUSSIAN_TANH, mean.cuda(), log_std.cuda(), acts.cuda())
    for got, ref, x in ((lp, gaussian_tanh_log_prob(mean, std, acts), acts),
                        (ent, -gaussian_tanh_log_prob(mean, std, mean), mean)):
        bound = 1e-5 + 1e-5 * ref.abs() + 2.0 ** -20 * _gaussian_terms(mean, std, x)
        err = (got.cpu() - ref).abs()
        assert bool((err <= bound).all()), (float((err / bound).max()), int((err > bound).sum()))


@pytest.mark.gpu
def test_wide_softmax_matches_torch():
    from ppo_and_friends_b200.synthetic import make_rollout
    ro = make_rollout(seed=3, T=2, E=257, obs_dim=12, n_discrete=4672, obs_scale=False)
    torch.manual_seed(1)
    pol = make_policy(ro, act="tanh", actor_hidden=64, critic_hidden=64)
    obs = torch.as_tensor(ro.obs["agent0"][0]).cuda()
    probs = pol.actor(obs, softmax_out=True).cpu()
    ref = torch.softmax(pol.actor(obs).cpu(), dim=-1)
    np.testing.assert_allclose(probs.numpy(), ref.numpy(), rtol=1e-5, atol=1e-9)


# ----------------------------------------------------------------------------------------- GPU: sampling
@pytest.mark.gpu
@pytest.mark.parametrize("P", [362, 4672])
def test_discrete_rollout_and_inference_actions(P):
    from ppo_and_friends_b200.synthetic import make_rollout
    ro = make_rollout(seed=P, T=2, E=257, obs_dim=12, n_discrete=P, obs_scale=False)
    torch.manual_seed(4)
    pol = make_policy(ro, act="leaky_relu", actor_hidden=64, critic_hidden=32)
    obs = [ro.obs["agent0"][t] for t in range(2)]
    probs = [pol.actor(torch.as_tensor(o).cuda(), softmax_out=True).cpu() for o in obs]
    torch.manual_seed(123)
    got = [pol.get_rollout_actions(o) for o in obs]
    after_got = torch.get_rng_state()
    torch.manual_seed(123)
    for (raw, act, lp), p in zip(got, probs):
        dist = Categorical(probs=p)
        ref = dist.sample()
        assert raw.dtype == np.int64 and act.shape == raw.shape == (257, 1)
        assert np.array_equal(act[:, 0], ref.numpy()) and np.array_equal(raw, act)
        assert tuple(lp.shape) == (257, 1)
        np.testing.assert_allclose(lp[:, 0].numpy(), dist.log_prob(ref).numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(after_got, torch.get_rng_state())              # exactly exponential_ of [n, P] per call
    det = pol.get_inference_actions(obs[0], True)
    assert torch.equal(det, probs[0].argmax(dim=-1))


@pytest.mark.gpu
def test_box_rollout_and_inference_actions():
    from ppo_and_friends_b200.synthetic import make_rollout
    d = 200
    ro = make_rollout(seed=9, T=2, E=257, obs_dim=12, act_dim=d, obs_scale=False)
    torch.manual_seed(5)
    pol = make_policy(ro, act="tanh", actor_hidden=64, critic_hidden=32, dist_range=2.5)
    obs = [ro.obs["agent0"][t] for t in range(2)]
    means = [pol.actor(torch.as_tensor(o).cuda()).cpu() for o in obs]
    log_std = pol.actor.state_dict()["distribution.log_std"].cpu()
    std = gaussian_std(log_std, pol.min_std)
    torch.manual_seed(77)
    got = [pol.get_rollout_actions(o) for o in obs]
    after_got = torch.get_rng_state()
    torch.manual_seed(77)
    for (raw, act, lp), mu in zip(got, means):
        ref_raw = torch.empty(257, d).normal_(0, 1).mul_(std).add_(mu)   # Normal.sample: mul_ then add_
        ref_act = (torch.tanh(ref_raw) + 1.0) / 2.0 * 5.0 - 2.5
        assert raw.shape == act.shape == (257, d) and raw.dtype == act.dtype == np.float32
        np.testing.assert_allclose(raw, ref_raw.numpy(), rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(act, ref_act.numpy(), rtol=1e-6, atol=1e-6)
        ref_lp = gaussian_tanh_log_prob(mu, std, torch.as_tensor(raw))
        np.testing.assert_allclose(lp.numpy().reshape(-1), ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(after_got, torch.get_rng_state())
    det = pol.get_inference_actions(obs[0], True)
    np.testing.assert_allclose(det.numpy(), ((torch.tanh(means[0]) + 1.0) / 2.0 * 5.0 - 2.5).numpy(), rtol=1e-6,
                               atol=1e-6)


# ----------------------------------------------------------------------------------------- GPU: the update
def _wide_rollout(n_actions, box_dim, seed):
    from ppo_and_friends_b200.synthetic import make_rollout
    return make_rollout(seed=seed, T=32, E=16, obs_dim=12, act_dim=box_dim or 2, n_discrete=n_actions,
                        max_ts_per_ep=12, obs_scale=False)


def _fill_old_outputs(pol, ro):
    """Old log-probs and values from the initial networks, so ratios start near 1."""
    with torch.no_grad():
        for a in ro.agents:
            obs = ro.obs[a].reshape(ro.T * ro.E, -1)
            cobs = ro.critic_obs[a].reshape(ro.T * ro.E, -1)
            values, lp, _ = pol.evaluate(cobs, obs, ro.raw_actions[a].reshape(ro.T * ro.E, -1))
            ro.log_probs[a] = lp.cpu().numpy().reshape(ro.T, ro.E)
            ro.values[a] = values.cpu().numpy().reshape(ro.T, ro.E)


def _update_vs_oracle(n_actions=0, box_dim=0, use_graphs=True, monkeypatch=None, lr=None, **policy_kw):
    """One epoch of 4 minibatches of 128 rows against OracleUpdater: status scalars, every parameter (log_std
    included) and dataset.values.

    Adam turns an fp32 difference in a small gradient element into a difference of up to a sizeable fraction of the
    step lr, so the parameter bound (1e-4 rel + 1e-6 abs) holds only while lr is small against it.  Discrete heads run
    at lr = 3e-4 (first-minibatch gradients within 1e-6 of their largest element, test_first_minibatch_gradients).
    Box heads have log-probs in the hundreds, their head gradients sit within 2e-5 (Box(64), the warp-per-sample
    kernel) to 4e-5 (Box(200)) of their largest element, and on a B200 the worst head weight missed the bound by 3.9x
    (Box(64)) and 4.7x (Box(200)) at lr = 3e-4 and by 1.3x / 1.6x at lr = 1e-4.  They run at lr = 3e-5: each parameter
    still moves by ~1e-4, 20 times the bound."""
    lr = lr if lr is not None else (3e-4 if n_actions else 3e-5)
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    if monkeypatch is not None:
        monkeypatch.setenv("PPOAF_NO_GRAPH", "0" if use_graphs else "1")
    ro = _wide_rollout(n_actions, box_dim, seed=61 + n_actions + box_dim)
    torch.manual_seed(5)
    pol = make_policy(ro, act="tanh", actor_hidden=64, critic_hidden=64, lr=lr, **policy_kw)
    assert pol.action_pred_size == (n_actions or box_dim)
    _fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    host = {name: getattr(ds, name).cpu().numpy().copy() for name in (
        "critic_observations", "observations", "raw_actions", "advantages", "log_probs", "rewards_to_go", "values")}
    oracle = OracleUpdater({n: v.cpu().numpy() for n, v in pol.actor.state_dict().items()},
                           {n: v.cpu().numpy() for n, v in pol.critic.state_dict().items()}, "tanh", bool(n_actions),
                           lr=lr, vf_clip=policy_kw.get("vf_clip"),
                           use_huber_loss=policy_kw.get("use_huber_loss", False))
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    torch.manual_seed(11)
    ppo_batch_train(state, _Loader(ds, 128), "pol")
    st = oracle.batch_train([host], [pol._engine._perm_dev.cpu().numpy()], 128)
    sd = state.status_dict["pol"]
    got = np.array([sd["actor loss"], sd["critic loss"], sd["kl avg"], sd["weighted entropy"]])
    ref = np.array([st["actor loss"], st["critic loss"], st["kl avg"], st["weighted entropy"]])
    # actor loss and KL are means of differences of log-probs: both sides carry a few 2^-24 |log-prob| of fp32
    # rounding in them, which exceeds the 1e-4 relative bound where |log-prob| is hundreds (wide Box heads)
    lp_scale = float(np.abs(host["log_probs"]).mean())
    bound = 1e-4 * np.maximum(np.abs(ref), 1e-3) + np.array([1, 0, 1, 0]) * 2.0 ** -21 * lp_scale
    assert bool((np.abs(got - ref) <= bound).all()), (got, ref, bound)
    ref_state = oracle.state()
    for net, obj in (("actor", pol.actor), ("critic", pol.critic)):
        for name, v in obj.state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref_state[f"{net}/param/{name}"], rtol=1e-4, atol=1e-6,
                                       err_msg=name)
    np.testing.assert_allclose(ds.values.cpu().numpy(), host["values"], rtol=1e-4, atol=1e-5)
    assert not pol._engine.fused
    return pol


@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False])
@pytest.mark.parametrize("space", ["Discrete(64)", "Discrete(65)", "Discrete(362)", "Discrete(4672)", "Box(64)",
                                   "Box(65)", "Box(200)"])
def test_update_vs_oracle(space, use_graphs, monkeypatch):
    """Discrete(64) and Box(64) run the warp-per-sample kernel: the controls at the switch to the wide kernel."""
    width = int(space[space.index("(") + 1:-1])
    _update_vs_oracle(**({"n_actions": width} if space.startswith("Discrete") else {"box_dim": width}),
                      use_graphs=use_graphs, monkeypatch=monkeypatch)


class _FirstGradients(OracleUpdater):
    """OracleUpdater that keeps the actor gradients of its first minibatch (before clipping)."""

    def _clip_and_step(self, which, params, grads_override=None):
        if which == "actor" and not hasattr(self, "first_actor_grads"):
            self.first_actor_grads = [g.clone() for g in (grads_override or [q.grad for q in params])]
        return super()._clip_and_step(which, params, grads_override)


@pytest.mark.gpu
@pytest.mark.parametrize("space", ["Discrete(362)", "Discrete(4672)", "Box(64)", "Box(65)", "Box(200)"])
def test_first_minibatch_gradients(space):
    """The actor gradients of one minibatch of all 512 rows against the oracle's autograd, per tensor within 1e-4 of
    its largest element (measured on a B200: <= 1e-6 for the Discrete heads, 2e-5 for Box(64), 4e-5 for Box(200))."""
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    width = int(space[space.index("(") + 1:-1])
    n_actions, box_dim = (width, 0) if space.startswith("Discrete") else (0, width)
    ro = _wide_rollout(n_actions, box_dim, seed=61 + width)
    torch.manual_seed(5)
    pol = make_policy(ro, act="tanh", actor_hidden=64, critic_hidden=64)
    _fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    host = {name: getattr(ds, name).cpu().numpy().copy() for name in (
        "critic_observations", "observations", "raw_actions", "advantages", "log_probs", "rewards_to_go", "values")}
    oracle = _FirstGradients({n: v.cpu().numpy() for n, v in pol.actor.state_dict().items()},
                             {n: v.cpu().numpy() for n, v in pol.critic.state_dict().items()}, "tanh", bool(n_actions))
    n = len(ds)
    torch.manual_seed(11)
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=n, epochs_per_iter=1), _Loader(ds, n), "pol")
    oracle.batch_train([host], [pol._engine._perm_dev.cpu().numpy()], n)
    got = pol.actor.grad_dict()
    names = list(pol.actor.state_dict().keys())
    assert len(names) == len(oracle.first_actor_grads)
    for name, ref in zip(names, oracle.first_actor_grads):
        g, r = got[name].detach().cpu().double(), ref.detach().double().reshape(got[name].shape)
        err = float((g - r).abs().max()) / float(r.abs().max())
        assert err < 1e-4, (name, err)


@pytest.mark.gpu
def test_update_vs_oracle_value_clip_and_huber():
    _update_vs_oracle(n_actions=362, vf_clip=0.5, use_huber_loss=True)


@pytest.mark.gpu
def test_fused_engine_request_runs_the_chain(monkeypatch):
    """PPOAF_STEP=fused cannot fuse a head wider than 24 outputs: the launch chain runs, with the same results."""
    monkeypatch.setenv("PPOAF_STEP", "chain")
    chain = _update_vs_oracle(n_actions=362)
    monkeypatch.setenv("PPOAF_STEP", "fused")
    fused = _update_vs_oracle(n_actions=362)
    assert torch.equal(chain.nets.flat_params, fused.nets.flat_params)


@pytest.mark.gpu
def test_box_checkpoint_round_trip(tmp_path):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    d = 200
    ro = _wide_rollout(0, d, seed=71)
    torch.manual_seed(2)
    pol = make_policy(ro, act="relu", actor_hidden=32, critic_hidden=32)
    ds = run_device_rollout(pol, ro)
    assert tuple(ds.raw_actions.shape) == (len(ds), d)
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1), _Loader(ds, 128), "pol")
    log_std = pol.actor.state_dict()["distribution.log_std"]
    assert tuple(log_std.shape) == (d,)
    pol.save(str(tmp_path))
    torch.manual_seed(3)
    fresh = make_policy(ro, act="relu", actor_hidden=32, critic_hidden=32)
    assert not torch.equal(fresh.nets.flat_params, pol.nets.flat_params)
    fresh.load(str(tmp_path))
    for name in ("flat_params", "adam_m", "adam_v", "adam_step"):
        assert torch.equal(getattr(fresh.nets, name), getattr(pol.nets, name)), name
    assert torch.equal(fresh.actor.state_dict()["distribution.log_std"], log_std)
    assert int(fresh.nets.adam_step.item()) > 0


@pytest.mark.gpu
def test_two_rank_box_update_matches_multirank_oracle():
    """Box(100) on 2 GPUs through the push exchange: the d(log_std) peer mirrors of the wide loss kernel."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PPOAF_MG_DISCRETE="0", PPOAF_MG_ACT_DIM="100", PPOAF_PEER="1", PPOAF_NVLS="0",
               PPOAF_MG_EXPECT="push")
    port = 29500 + (os.getpid() + 7) % 1000
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(root, "tests", "multi_gpu_wide_worker.py")], env=env, capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0 and "MULTI_GPU_CHECK PASS" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
