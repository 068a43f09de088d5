"""
MultiBinary action spaces: the Bernoulli head through the C ABI, the update (both step engines), rollout sampling,
inference, the rollout ring and checkpoints.

There is no reference golden for this head, so the expected values come from a torch-CPU restatement of
torch.distributions.Bernoulli (below): p = sigmoid(actor output), one Bernoulli(probs=p) per column, log-prob and
entropy summed over the columns, sampling a = (u < p) with u = torch.rand(n, k) from the global CPU generator.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import ACT_MODULES, rel_err, run_device_rollout
from oracle.update import OracleUpdater
from ppo_and_friends_b200.spaces import Box, MultiBinary


# ----------------------------------------------------------------------------------------- the restatement
def bernoulli_columns(logits, actions):
    """Per-column (log_prob, entropy) [n, k] of fp32 0/1 actions on the actor's logits, as torch's Bernoulli(probs)
    computes them from p = sigmoid(logits)."""
    p = torch.sigmoid(logits)
    eps = torch.finfo(p.dtype).eps
    q = torch.clamp(p, eps, 1 - eps)
    lg = torch.log(q) - torch.log1p(-q)
    ls = F.logsigmoid(lg)
    return -((1 - actions) * lg - ls), (1 - p) * lg - ls


def bernoulli_log_prob_entropy(logits, actions):
    """(log_prob [n], entropy [n]): the per-column values summed over the columns."""
    lp, ent = bernoulli_columns(logits, actions)
    return lp.sum(dim=-1), ent.sum(dim=-1)


def bernoulli_sample(probs):
    """Bernoulli(probs).sample()'s draw protocol: u = rand(n, k) from the global CPU generator, a = (u < p) as fp32.
    Returns (actions, u)."""
    u = torch.rand(probs.shape, dtype=torch.float32)
    return (u < probs).to(torch.float32), u


class BernoulliOracle(OracleUpdater):
    """OracleUpdater whose action head is the Bernoulli restatement (autograd through it; no log_std)."""

    def __init__(self, actor_params, critic_params, activation, **kw):
        super().__init__(actor_params, critic_params, activation, True, **kw)

    def evaluate(self, critic_obs, obs, raw_actions):
        values = self.critic.forward(critic_obs).squeeze()
        pred = self.actor.forward(obs)
        lp, ent = bernoulli_log_prob_entropy(pred, raw_actions.reshape(pred.shape[0], -1).to(torch.float32))
        return values, lp, ent


# ----------------------------------------------------------------------------------------- builders
def mb_rollout(seed, k, T=32, E=16, obs_dim=12, critic_obs_dim=None, max_ts_per_ep=12):
    """Synthetic rollout whose stored actions are fp32 0/1 [T, E, k]."""
    from ppo_and_friends_b200.synthetic import make_rollout
    ro = make_rollout(seed=seed, T=T, E=E, obs_dim=obs_dim, critic_obs_dim=critic_obs_dim, act_dim=k,
                      max_ts_per_ep=max_ts_per_ep, obs_scale=False)
    rng = np.random.default_rng(seed + 1)
    for a in ro.agents:
        act = rng.integers(0, 2, size=(T, E, k)).astype(np.float32)
        ro.raw_actions[a] = act
        ro.actions[a] = act.copy()
    return ro


def make_mb_policy(ro, k, act="tanh", hidden=64, depth=3, **policy_kw):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    pol = PPOPolicy("pol", MultiBinary(k), Box(-np.inf, np.inf, (ro.obs_dim,)),
                    Box(-np.inf, np.inf, (ro.critic_obs_dim,)), envs_per_proc=ro.E,
                    actor_kw_args=dict(activation=ACT_MODULES[act](), hidden_size=hidden, hidden_depth=depth),
                    critic_kw_args=dict(activation=ACT_MODULES[act](), hidden_size=hidden, hidden_depth=depth),
                    **policy_kw)
    for a in ro.agents:
        pol.register_agent(a)
    pol.agent_ids = np.array(ro.agents)
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device("cuda"))
    return pol


def fill_old_outputs(pol, ro):
    """Old log-probs and values from the initial networks, so ratios start near 1."""
    with torch.no_grad():
        for a in ro.agents:
            obs = ro.obs[a].reshape(ro.T * ro.E, -1)
            cobs = ro.critic_obs[a].reshape(ro.T * ro.E, -1)
            values, lp, _ = pol.evaluate(cobs, obs, ro.raw_actions[a].reshape(ro.T * ro.E, -1))
            ro.log_probs[a] = lp.cpu().numpy().reshape(ro.T, ro.E)
            ro.values[a] = values.cpu().numpy().reshape(ro.T, ro.E)


@pytest.fixture(params=["ffma", "fused"])
def gemm_backend(request, monkeypatch):
    """Both engines of the minibatch step: the launch chain with FFMA tiles and the persistent whole-epoch kernel
    (PPOAF_STEP=fused)."""
    from ppo_and_friends_b200 import ops
    if request.param == "fused":
        monkeypatch.setenv("PPOAF_STEP", "fused")
        yield request.param
        return
    monkeypatch.setenv("PPOAF_STEP", "chain")
    ops.set_gemm_backend(request.param)
    yield request.param
    ops.set_gemm_backend("ffma")


# ----------------------------------------------------------------------------------------- CPU
def test_restatement_equals_torch_bernoulli():
    from torch.distributions import Bernoulli
    torch.manual_seed(0)
    logits = torch.randn(500, 13) * 4
    logits[0, :4] = torch.tensor([40.0, -40.0, 17.0, -120.0])             # the clamp to [eps, 1 - eps] bites
    acts = torch.randint(0, 2, (500, 13)).to(torch.float32)
    d = Bernoulli(probs=torch.sigmoid(logits))
    lp, ent = bernoulli_columns(logits, acts)
    assert torch.equal(lp, d.log_prob(acts)) and torch.equal(ent, d.entropy())
    s_lp, s_ent = bernoulli_log_prob_entropy(logits, acts)
    assert torch.equal(s_lp, d.log_prob(acts).sum(-1)) and torch.equal(s_ent, d.entropy().sum(-1))
    for seed in (1, 2):
        torch.manual_seed(seed)
        got, _ = bernoulli_sample(d.probs)
        after_got = torch.get_rng_state()
        torch.manual_seed(seed)
        ref = d.sample()
        assert ref.dtype == torch.float32 and torch.equal(got, ref)
        assert torch.equal(after_got, torch.get_rng_state())


def _policy(action_space):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    return PPOPolicy("pol", action_space, Box(-1, 1, (4,)), Box(-1, 1, (4,)), envs_per_proc=2)


def test_policy_accepts_and_refuses_multibinary_spaces():
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.policies.ppo_policy import space_dtype_str
    assert space_dtype_str(MultiBinary(3)) == "multi-binary"
    for n in (1, 7, 64):
        pol = _policy(MultiBinary(n))
        assert (pol.action_dtype, pol.action_dim, pol.action_pred_size) == ("multi-binary", n, n)
        assert pol.head == _lib.HEAD_BERNOULLI
    for bad in (MultiBinary(65), MultiBinary([2, 3]), MultiBinary(0)):
        with pytest.raises(RuntimeError):
            _policy(bad)


def test_generate_policy_builds_a_multibinary_policy():
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.policies.utils import generate_policy
    pol = generate_policy("pol", PPOPolicy, Box(-1, 1, (5,)), Box(-1, 1, (9,)), MultiBinary(6), test_mode=False,
                          envs_per_proc=3, surr_clip=0.3)
    assert isinstance(pol, PPOPolicy) and pol.head == _lib.HEAD_BERNOULLI
    assert (pol.action_dim, pol.action_pred_size, pol.surr_clip) == (6, 6, 0.3)


def _cfg(pred, act_dim):
    from ppo_and_friends_b200 import _lib
    cfg = _lib.UpdateCfg()
    cfg.actor = _lib.MlpDesc.make([6, 16, 16, pred], "tanh")
    cfg.critic = _lib.MlpDesc.make([6, 16, 16, 1], "tanh")
    cfg.head, cfg.act_dim = _lib.HEAD_BERNOULLI, act_dim
    return cfg


def test_bernoulli_width_mismatch_is_refused_through_the_c_abi():
    """The update entry points refuse act_dim != actor output width before they touch the device; so do the
    stand-alone head entry points (which then return without launching for zero rows)."""
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.build import build
    build()
    lib = _lib.load()
    bufs = _lib.UpdateBufs()
    msg = lambda: lib.ppoaf_last_error().decode()
    for fn in ("ppoaf_ppo_minibatch_grads", "ppoaf_ppo_fused_steps"):
        args = (C.byref(bufs), 1, None) if fn == "ppoaf_ppo_fused_steps" else (C.byref(bufs), None)
        for pred, act_dim in ((7, 6), (7, 8), (7, 1)):
            assert getattr(lib, fn)(C.byref(_cfg(pred, act_dim)), *args) != 0
            assert "Bernoulli actor output width" in msg(), (fn, pred, act_dim, msg())
        assert getattr(lib, fn)(C.byref(_cfg(7, 7)), *args) != 0                 # empty buffers: refused, but later
        assert "Bernoulli" not in msg(), msg()
    fake = C.c_void_p(16)                                                        # never dereferenced: zero rows
    H = _lib.HEAD_BERNOULLI
    assert lib.ppoaf_head_evaluate(H, None, 7, None, 0.01, None, 6, 0, None, None, None) != 0
    assert "Bernoulli actor output width" in msg()
    assert lib.ppoaf_head_evaluate(H, None, 7, fake, 0.01, None, 7, 0, None, None, None) != 0
    assert "log_std" in msg()
    assert lib.ppoaf_head_evaluate(H, None, 7, None, 0.01, None, 7, 0, None, None, None) == 0
    sample = lambda pred, act_dim, log_std=None, lo=None, hi=None: lib.ppoaf_head_sample(
        H, None, pred, log_std, 0.01, fake, lo, hi, act_dim, 0, None, None, None, None)
    assert sample(7, 6) != 0 and "Bernoulli actor output width" in msg()
    assert sample(7, 7, log_std=fake) != 0 and "log_std" in msg()
    assert sample(7, 7, lo=fake, hi=fake) != 0 and "range bounds" in msg()
    assert sample(7, 7) == 0


# ----------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 5, 24, 33, 64])
def test_bernoulli_evaluate_vs_restatement(k):
    from ppo_and_friends_b200 import _lib, ops
    torch.manual_seed(k)
    n = 300
    logits = torch.randn(n, k) * 3
    # rows 0..19 saturate: |z| in [20, 120], so p < eps or p > 1 - eps (the clamp bites) and p is often exactly 0 or 1
    sat = torch.rand(20, k) * 100 + 20
    logits[:20] = torch.where(torch.rand(20, k) < 0.5, sat, -sat)
    p = torch.sigmoid(logits[:20])
    assert bool(((p == 0) | (p == 1)).any()) and bool(((p < 1.2e-7) | (p > 1 - 1.2e-7)).all())
    acts = torch.randint(0, 2, (n, k)).to(torch.float32)
    ref_lp, ref_ent = bernoulli_log_prob_entropy(logits, acts)
    lp, ent = ops.head_evaluate(_lib.HEAD_BERNOULLI, logits.cuda(), None, acts.cuda())
    np.testing.assert_allclose(lp.cpu().numpy(), ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ent.cpu().numpy(), ref_ent.numpy(), rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
def test_rollout_and_inference_actions_vs_restatement():
    k = 11
    ro = mb_rollout(21, k, T=2, E=257)
    torch.manual_seed(4)
    pol = make_mb_policy(ro, k, act="leaky_relu", hidden=32)
    obs = [ro.obs["agent0"][t] for t in range(2)]
    logits = [pol.actor(o).cpu() for o in obs]
    torch.manual_seed(123)
    got = [pol.get_rollout_actions(o) for o in obs]
    after_got = torch.get_rng_state()
    torch.manual_seed(123)
    near = 0
    for (raw, act, lp), z in zip(got, logits):
        p = torch.sigmoid(z)
        ref_a, u = bernoulli_sample(p)
        assert raw.dtype == np.float32 and act.dtype == np.float32 and raw.shape == act.shape == (257, k)
        assert np.array_equal(raw, act) and set(np.unique(act).tolist()) <= {0.0, 1.0}
        # the device's sigmoid may round differently from torch's: a draw within 1e-6 of p may flip
        close = (u - p).abs() <= 1e-6
        near += int(close.sum())
        assert np.array_equal(act[~close.numpy()], ref_a.numpy()[~close.numpy()])
        assert tuple(lp.shape) == (257,) and lp.dtype == torch.float32
        ref_lp, _ = bernoulli_log_prob_entropy(z, torch.as_tensor(act))
        np.testing.assert_allclose(lp.numpy(), ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    assert near == 0
    assert torch.equal(after_got, torch.get_rng_state())                       # the rollout drew exactly rand(n, k)
    det = pol.get_inference_actions(obs[0], True)
    assert det.dtype == torch.float32 and torch.equal(det, (torch.sigmoid(logits[0]) > 0.5).to(torch.float32))
    assert tuple(pol.get_inference_actions(obs[0], False).shape) == (257, k)


def _update_vs_oracle(k, hidden=64, use_graphs=True, monkeypatch=None, **policy_kw):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    if monkeypatch is not None:
        monkeypatch.setenv("PPOAF_NO_GRAPH", "0" if use_graphs else "1")
    ro = mb_rollout(41 + k, k)
    torch.manual_seed(5)
    pol = make_mb_policy(ro, k, act="tanh", hidden=hidden, lr=1e-3, **policy_kw)
    assert "distribution.log_std" not in pol.actor.state_dict()
    fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    assert ds.raw_actions.dtype == torch.float32 and tuple(ds.raw_actions.shape) == (len(ds), k)
    host = {name: getattr(ds, name).cpu().numpy().copy() for name in (
        "critic_observations", "observations", "raw_actions", "advantages", "log_probs", "rewards_to_go", "values")}
    oracle = BernoulliOracle({n: v.cpu().numpy() for n, v in pol.actor.state_dict().items()},
                             {n: v.cpu().numpy() for n, v in pol.critic.state_dict().items()}, "tanh",
                             lr=1e-3, vf_clip=policy_kw.get("vf_clip"),
                             use_huber_loss=policy_kw.get("use_huber_loss", False))
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    torch.manual_seed(11)
    ppo_batch_train(state, _Loader(ds, 128), "pol")
    st = oracle.batch_train([host], [pol._engine._perm_dev.cpu().numpy()], 128)
    sd = state.status_dict["pol"]
    got = np.array([sd["actor loss"], sd["critic loss"], sd["kl avg"], sd["weighted entropy"]])
    ref = np.array([st["actor loss"], st["critic loss"], st["kl avg"], st["weighted entropy"]])
    assert rel_err(got, ref, 1e-3) < 1e-4, (got, ref)
    ref_state = oracle.state()
    for net, obj in (("actor", pol.actor), ("critic", pol.critic)):
        for name, v in obj.state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref_state[f"{net}/param/{name}"], rtol=1e-4, atol=1e-6,
                                       err_msg=name)
    np.testing.assert_allclose(ds.values.cpu().numpy(), host["values"], rtol=1e-4, atol=1e-5)
    return pol


@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False])
def test_update_vs_oracle_fused_head_width(use_graphs, monkeypatch, gemm_backend):
    """14 columns: the head layers are fused into the loss (and the persistent engine runs)."""
    pol = _update_vs_oracle(14, use_graphs=use_graphs, monkeypatch=monkeypatch)
    assert pol._engine.fused == (gemm_backend == "fused")


@pytest.mark.gpu
def test_update_vs_oracle_wide_head():
    """40 columns: lanes own a second column past lane 31; unfused head layers."""
    pol = _update_vs_oracle(40)
    assert not pol._engine.fused


@pytest.mark.gpu
def test_update_vs_oracle_value_clip_and_huber():
    _update_vs_oracle(14, vf_clip=0.5, use_huber_loss=True)


@pytest.mark.gpu
def test_rollout_to_dataset_and_checkpoint_round_trip(tmp_path):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    k = 7
    ro = mb_rollout(51, k, T=24, E=8)
    torch.manual_seed(2)
    pol = make_mb_policy(ro, k, act="relu", hidden=32)
    ds = run_device_rollout(pol, ro)
    src = ds.src_row.long().cpu().numpy()                                 # ring row = step * E + env (one agent)
    for name in ("raw_actions", "actions"):
        got = getattr(ds, name)
        assert got.dtype == torch.float32 and tuple(got.shape) == (len(ds), k)
        assert np.array_equal(got.cpu().numpy(), getattr(ro, name)["agent0"].reshape(-1, k)[src]), name
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=64, epochs_per_iter=1), _Loader(ds, 64), "pol")
    pol.save(str(tmp_path))
    torch.manual_seed(3)
    fresh = make_mb_policy(ro, k, act="relu", hidden=32)
    assert not torch.equal(fresh.nets.flat_params, pol.nets.flat_params)
    fresh.load(str(tmp_path))
    for name in ("flat_params", "adam_m", "adam_v", "adam_step"):
        assert torch.equal(getattr(fresh.nets, name), getattr(pol.nets, name)), name
    assert int(fresh.nets.adam_step.item()) > 0
