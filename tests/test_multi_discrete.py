"""
MultiDiscrete action spaces: the multi-categorical head through the C ABI, the update (both step engines), rollout
sampling, inference, the rollout ring and checkpoints.

There is no reference golden for this head, so the expected values come from a torch-CPU restatement built from
torch.distributions (below): softmax over the whole actor output row, one Categorical(probs=section) per section,
log-prob and entropy summed over the sections, sampling section after section from the global CPU generator.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import ACT_MODULES, make_policy, rel_err, run_device_rollout
from oracle.update import OracleUpdater, categorical_from_probs
from ppo_and_friends_b200.spaces import Box, MultiDiscrete


# ----------------------------------------------------------------------------------------- the restatement
def multi_categorical_log_prob_entropy(logits, actions, nvec):
    """(log_prob [n], entropy [n]) of int64 actions [n, len(nvec)] on the actor's logits [n, sum(nvec)]."""
    probs = torch.softmax(logits, dim=-1)
    lp = ent = 0.0
    for k, sec in enumerate(probs.split(list(nvec), dim=-1)):
        p, lg = categorical_from_probs(sec)
        lp = lp + lg.gather(-1, actions[:, k:k + 1].long()).reshape(-1)
        ent = ent - (p * lg).sum(dim=-1)
    return lp, ent


def multi_categorical_sample(probs, nvec):
    """Per-section Categorical.sample's draw protocol on softmax probs [n, sum(nvec)]: section after section,
    exponential_(1) of shape [n, n_k], a_k = first argmax(p~_k / q_k).  Returns (int64 actions [n, K], log_prob [n])."""
    acts, lp = [], 0.0
    for sec in probs.split(list(nvec), dim=-1):
        p, lg = categorical_from_probs(sec)
        q = torch.empty(sec.shape, dtype=torch.float32).exponential_(1)
        a = torch.argmax(p / q, dim=-1)
        acts.append(a)
        lp = lp + lg.gather(-1, a.reshape(-1, 1)).reshape(-1)
    return torch.stack(acts, dim=1), lp


class MultiCategoricalOracle(OracleUpdater):
    """OracleUpdater whose action head is the multi-categorical restatement (autograd through it)."""

    def __init__(self, actor_params, critic_params, activation, nvec, **kw):
        super().__init__(actor_params, critic_params, activation, True, **kw)
        self.nvec = [int(n) for n in nvec]

    def evaluate(self, critic_obs, obs, raw_actions):
        values = self.critic.forward(critic_obs).squeeze()
        pred = self.actor.forward(obs)
        lp, ent = multi_categorical_log_prob_entropy(pred, raw_actions.reshape(pred.shape[0], -1), self.nvec)
        return values, lp, ent


# ----------------------------------------------------------------------------------------- builders
def md_rollout(seed, nvec, T=32, E=16, obs_dim=12, critic_obs_dim=None, max_ts_per_ep=12):
    """Synthetic rollout whose stored actions are int64 [T, E, len(nvec)], entry k in [0, nvec[k])."""
    from ppo_and_friends_b200.synthetic import make_rollout
    ro = make_rollout(seed=seed, T=T, E=E, obs_dim=obs_dim, critic_obs_dim=critic_obs_dim, act_dim=len(nvec),
                      max_ts_per_ep=max_ts_per_ep, obs_scale=False)
    rng = np.random.default_rng(seed + 1)
    for a in ro.agents:
        act = np.stack([rng.integers(0, n, size=(T, E)) for n in nvec], axis=-1).astype(np.int64)
        ro.raw_actions[a] = act
        ro.actions[a] = act.copy()
    return ro


def make_md_policy(ro, nvec, act="tanh", hidden=64, depth=3, **policy_kw):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    pol = PPOPolicy("pol", MultiDiscrete(nvec), Box(-np.inf, np.inf, (ro.obs_dim,)),
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
def test_restatement_equals_per_section_torch_categorical():
    from torch.distributions import Categorical
    nvec = [3, 1, 5, 2]
    torch.manual_seed(0)
    logits = torch.randn(200, sum(nvec)) * 4
    logits[0, :3] = torch.tensor([40.0, -40.0, 0.0])                      # clamp to [eps, 1 - eps] bites
    acts = torch.stack([torch.randint(0, n, (200,)) for n in nvec], dim=1)
    lp, ent = multi_categorical_log_prob_entropy(logits, acts, nvec)
    dists = [Categorical(probs=s) for s in torch.softmax(logits, -1).split(nvec, dim=-1)]
    ref_lp = sum(d.log_prob(acts[:, k]) for k, d in enumerate(dists))
    ref_ent = sum(d.entropy() for d in dists)
    torch.testing.assert_close(lp, ref_lp, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(ent, ref_ent, rtol=1e-6, atol=1e-6)
    probs = torch.softmax(logits, -1)
    for seed in (1, 2):
        torch.manual_seed(seed)
        got, got_lp = multi_categorical_sample(probs, nvec)
        torch.manual_seed(seed)
        ref = torch.stack([Categorical(probs=s).sample() for s in probs.split(nvec, dim=-1)], 1)
        assert torch.equal(got, ref)
        lp_ref, _ = multi_categorical_log_prob_entropy(logits, ref, nvec)
        torch.testing.assert_close(got_lp, lp_ref, rtol=1e-6, atol=1e-6)


def _policy(action_space):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    return PPOPolicy("pol", action_space, Box(-1, 1, (4,)), Box(-1, 1, (4,)), envs_per_proc=2)


def test_policy_accepts_and_refuses_multidiscrete_spaces():
    from ppo_and_friends_b200 import _lib
    pol = _policy(MultiDiscrete([3, 5, 2]))
    assert (pol.action_dtype, pol.action_dim, pol.action_pred_size) == ("multi-discrete", 3, 10)
    assert pol.head == _lib.HEAD_MULTI_CATEGORICAL and pol.section_ends == (1 << 2) | (1 << 7) | (1 << 9)
    assert _policy(MultiDiscrete([64])).section_ends == 1 << 63
    assert _policy(MultiDiscrete([4, 4], start=[0, 0])).action_pred_size == 8
    for bad in (MultiDiscrete([40, 25]), MultiDiscrete([[2, 3], [4, 5]]), MultiDiscrete([3, 4], start=[1, 0]),
                MultiDiscrete([3, 0]), MultiDiscrete([])):
        with pytest.raises(RuntimeError):
            _policy(bad)


def _cfg(nvec, ends, act_dim):
    from ppo_and_friends_b200 import _lib
    cfg = _lib.UpdateCfg()
    cfg.actor = _lib.MlpDesc.make([6, 16, 16, sum(nvec)], "tanh")
    cfg.critic = _lib.MlpDesc.make([6, 16, 16, 1], "tanh")
    cfg.head, cfg.act_dim = _lib.HEAD_MULTI_CATEGORICAL, act_dim
    cfg.section_ends[0], cfg.section_ends[1] = ends & 0xFFFFFFFF, ends >> 32
    return cfg


def test_malformed_section_table_is_refused_through_the_c_abi():
    """The update entry points validate the configuration before they touch the device; so do the stand-alone head
    entry points (which then return without launching for zero rows)."""
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.build import build
    build()
    lib = _lib.load()
    nvec = [2, 2, 3]
    good = _lib.section_ends(nvec)
    assert good == 0b1001010
    bufs = _lib.UpdateBufs()
    msg = lambda: lib.ppoaf_last_error().decode()
    for fn in ("ppoaf_ppo_minibatch_grads", "ppoaf_ppo_fused_steps"):
        args = (C.byref(bufs), 1, None) if fn == "ppoaf_ppo_fused_steps" else (C.byref(bufs), None)
        for ends, act_dim in ((good, 2), (good >> 1, 3), (good | (1 << 9), 4), (0, 0)):
            assert getattr(lib, fn)(C.byref(_cfg(nvec, ends, act_dim)), *args) != 0
            assert "section table" in msg(), (fn, ends, act_dim, msg())
        assert getattr(lib, fn)(C.byref(_cfg(nvec, good, 3)), *args) != 0        # empty buffers: refused, but later
        assert "section table" not in msg(), msg()
    for ends, act_dim in ((good, 2), (good >> 1, 3), (1 << 64 - 1, 1)):
        assert lib.ppoaf_multi_categorical_evaluate(None, 7, ends & 0xFFFFFFFF, ends >> 32, None, act_dim, 0,
                                                    None, None, None) != 0
        assert "section table" in msg()
        assert lib.ppoaf_multi_categorical_sample(None, 7, ends & 0xFFFFFFFF, ends >> 32, None, act_dim, 0,
                                                  None, None, None) != 0
    assert lib.ppoaf_multi_categorical_evaluate(None, 7, good, 0, None, 3, 0, None, None, None) == 0
    assert lib.ppoaf_multi_categorical_sample(None, 7, good, 0, None, 3, 0, None, None, None) == 0


# ----------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("nvec", [[3, 5, 2, 4], [1, 6, 1], [9, 9, 9, 9, 9, 7, 2], [64], [1] * 20 + [44]])
def test_multi_categorical_evaluate_vs_restatement(nvec):
    from ppo_and_friends_b200 import _lib, ops
    torch.manual_seed(len(nvec) + sum(nvec))
    n = 300
    logits = torch.randn(n, sum(nvec)) * 3
    # rows 0..19: one column of every section 25 above the rest, so the others' p~ < eps and the clamp bites (without
    # a section whose probabilities all underflow, where the restatement itself is 0 / 0)
    for o, k in zip(np.cumsum([0] + nvec[:-1]), nvec):
        logits[torch.arange(20), int(o) + torch.randint(0, k, (20,))] += 25.0
    acts = torch.stack([torch.randint(0, k, (n,)) for k in nvec], dim=1)
    ref_lp, ref_ent = multi_categorical_log_prob_entropy(logits, acts, nvec)
    lp, ent = ops.multi_categorical_evaluate(logits.cuda(), _lib.section_ends(nvec), acts.cuda())
    np.testing.assert_allclose(lp.cpu().numpy(), ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ent.cpu().numpy(), ref_ent.numpy(), rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
def test_rollout_and_inference_actions_vs_restatement():
    nvec = [3, 5, 2, 4, 1]
    ro = md_rollout(21, nvec, T=2, E=257)
    torch.manual_seed(4)
    pol = make_md_policy(ro, nvec, act="leaky_relu", hidden=32)
    obs = [ro.obs["agent0"][t] for t in range(2)]
    probs = [pol.actor(o, softmax_out=True).cpu() for o in obs]
    torch.manual_seed(123)
    got = [pol.get_rollout_actions(o) for o in obs]
    torch.manual_seed(123)
    for (raw, act, lp), p in zip(got, probs):
        ref_a, ref_lp = multi_categorical_sample(p, nvec)
        assert raw.dtype == np.int64 and act.dtype == np.int64 and raw.shape == act.shape == (257, len(nvec))
        assert np.array_equal(act, ref_a.numpy()) and np.array_equal(raw, act)
        assert tuple(lp.shape) == (257, 1)
        np.testing.assert_allclose(lp.numpy()[:, 0], ref_lp.numpy(), rtol=1e-5, atol=1e-5)
    det = pol.get_inference_actions(obs[0], True)
    ref = torch.stack([s.argmax(-1) for s in probs[0].split(nvec, dim=1)], dim=1)
    assert det.dtype == torch.int64 and torch.equal(det, ref)
    assert tuple(pol.get_inference_actions(obs[0], False).shape) == (257, len(nvec))


@pytest.mark.gpu
def test_one_section_reproduces_discrete_exactly(gemm_backend):
    """MultiDiscrete([n]) and Discrete(n) on the same rollout, seeds and initial weights: identical sampled actions,
    log-probs, status scalars, parameters, Adam moments, dataset.values and PPOPolicy.evaluate's log-probs and
    entropies."""
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    from ppo_and_friends_b200.synthetic import make_rollout
    out = {}
    for kind in ("discrete", "multi"):
        ro = make_rollout(seed=31, T=32, E=16, obs_dim=12, n_discrete=6, max_ts_per_ep=12, obs_scale=False)
        torch.manual_seed(8)
        if kind == "discrete":
            pol = make_policy(ro, act="tanh", actor_hidden=64, critic_hidden=64, lr=1e-3)
        else:
            pol = make_md_policy(ro, [6], act="tanh", hidden=64, lr=1e-3)
        torch.manual_seed(9)
        raw, act, lp = pol.get_rollout_actions(ro.obs["agent0"][0])
        fill_old_outputs(pol, ro)
        ds = run_device_rollout(pol, ro)
        state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=2)
        loader = _Loader(ds, 128)
        for _ in range(2):
            ppo_batch_train(state, loader, "pol")
        _, eval_lp, eval_ent = pol.evaluate(ds.critic_observations, ds.observations, ds.raw_actions)
        out[kind] = dict(act=act, lp=lp.numpy(), params=pol.nets.flat_params.cpu(), m=pol.nets.adam_m.cpu(),
                         v=pol.nets.adam_v.cpu(), values=ds.values.cpu(), status=dict(state.status_dict["pol"]),
                         fused=pol._engine.fused, eval_lp=eval_lp.cpu(), eval_ent=eval_ent.cpu())
    a, b = out["discrete"], out["multi"]
    assert a["fused"] == b["fused"] == (gemm_backend == "fused")
    assert np.array_equal(a["act"], b["act"]) and np.array_equal(a["lp"], b["lp"])
    for k in ("params", "m", "v", "values", "eval_lp", "eval_ent"):
        assert torch.equal(a[k], b[k]), k
    assert a["status"] == b["status"]


def _update_vs_oracle(nvec, hidden=64, use_graphs=True, monkeypatch=None, **policy_kw):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    if monkeypatch is not None:
        monkeypatch.setenv("PPOAF_NO_GRAPH", "0" if use_graphs else "1")
    ro = md_rollout(41 + len(nvec), nvec)
    torch.manual_seed(5)
    pol = make_md_policy(ro, nvec, act="tanh", hidden=hidden, lr=1e-3, **policy_kw)
    fill_old_outputs(pol, ro)
    ds = run_device_rollout(pol, ro)
    assert ds.raw_actions.dtype == torch.int64 and tuple(ds.raw_actions.shape) == (len(ds), len(nvec))
    host = {k: getattr(ds, k).cpu().numpy().copy() for k in ("critic_observations", "observations", "raw_actions",
                                                               "advantages", "log_probs", "rewards_to_go", "values")}
    oracle = MultiCategoricalOracle({k: v.cpu().numpy() for k, v in pol.actor.state_dict().items()},
                                    {k: v.cpu().numpy() for k, v in pol.critic.state_dict().items()}, "tanh", nvec,
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
        for k, v in obj.state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref_state[f"{net}/param/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
    np.testing.assert_allclose(ds.values.cpu().numpy(), host["values"], rtol=1e-4, atol=1e-5)
    return pol


@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False])
def test_update_vs_oracle_fused_head_width(use_graphs, monkeypatch, gemm_backend):
    """nvec = [3, 5, 2, 4]: 14 actor outputs, so the head layers are fused into the loss (and the persistent engine runs)."""
    pol = _update_vs_oracle([3, 5, 2, 4], use_graphs=use_graphs, monkeypatch=monkeypatch)
    assert pol._engine.fused == (gemm_backend == "fused")


@pytest.mark.gpu
def test_update_vs_oracle_wide_head():
    """nvec = [9, 9, 9, 9, 9, 7, 2]: 54 actor outputs (sections cross the 32-column boundary; unfused head layers)."""
    _update_vs_oracle([9, 9, 9, 9, 9, 7, 2])


@pytest.mark.gpu
def test_update_vs_oracle_value_clip_and_huber():
    _update_vs_oracle([3, 5, 2, 4], vf_clip=0.5, use_huber_loss=True)


@pytest.mark.gpu
def test_rollout_to_dataset_and_checkpoint_round_trip(tmp_path):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    nvec = [4, 3, 7]
    ro = md_rollout(51, nvec, T=24, E=8)
    torch.manual_seed(2)
    pol = make_md_policy(ro, nvec, act="relu", hidden=32)
    ds = run_device_rollout(pol, ro)
    src = ds.src_row.long().cpu().numpy()                                 # ring row = step * E + env (one agent)
    for name in ("raw_actions", "actions"):
        got = getattr(ds, name)
        assert got.dtype == torch.int64 and tuple(got.shape) == (len(ds), len(nvec))
        assert np.array_equal(got.cpu().numpy(), getattr(ro, name)["agent0"].reshape(-1, len(nvec))[src]), name
    ppo_batch_train(PPOUpdateState({"pol": pol}, batch_size=64, epochs_per_iter=1), _Loader(ds, 64), "pol")
    pol.save(str(tmp_path))
    torch.manual_seed(3)
    fresh = make_md_policy(ro, nvec, act="relu", hidden=32)
    assert not torch.equal(fresh.nets.flat_params, pol.nets.flat_params)
    fresh.load(str(tmp_path))
    for k in ("flat_params", "adam_m", "adam_v", "adam_step"):
        assert torch.equal(getattr(fresh.nets, k), getattr(pol.nets, k)), k
    assert int(fresh.nets.adam_step.item()) > 0
