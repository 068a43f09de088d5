"""
The drop-in boundary (SURVEY.md §8b, INTEGRATION.md): the UNMODIFIED reference trainer driven through the four
INTEGRATION.md edits.

CPU (no GPU needed): every member the reference `PPO` touches on a policy object exists on the B200 `PPOPolicy`
with a compatible signature — checked against the reference's static surface recorded in
tests/golden/reference_surface.json (the members a regex over its ppo.py finds, the parameter names of its policy
methods and of generate_policy), so a missing member fails here instead of inside `PPO.__init__` on the GPU.
GPU: the real `PPO.__init__ -> rollout() -> learn()` for two iterations on a toy environment, once stock on the CPU and
once with the four edits applied by monkey-patching, must report the same status dictionary.

The tests that execute the reference need its source tree (PPOAF_REFERENCE_ROOT, or the git-ignored copy oracle/_ref
made by oracle/build_ref.py) and skip without it; with it, the static tests also check the record against the tree.
"""
import inspect
import json
import os
import re
import sys
import tempfile

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import ref_harness  # noqa: E402

requires_reference = pytest.mark.skipif(
    not ref_harness.available(),
    reason="runs the original LLNL/ppo_and_friends: set PPOAF_REFERENCE_ROOT to its source tree (or copy it to oracle/_ref "
           "with oracle/build_ref.py)")
with open(os.path.join(GOLDEN, "reference_surface.json")) as _fh:
    SURFACE = json.load(_fh)

# members of the reference policy that belong to subsystems outside the accelerated path (SURVEY.md §8: ICM, LSTM, MAT)
OUT_OF_SCOPE = {"icm_lr", "intr_reward_weight", "get_agent_shared_intrinsic_rewards", "get_intrinsic_reward", "icm_model",
                "icm_beta", "icm_optim"}
SET_BY_FINALIZE = {"actor", "critic", "actor_optim", "critic_optim", "agent_idxs", "dataset"}


def _reference():
    ref_harness.install()
    import ppo_and_friends.ppo as ref_ppo
    from ppo_and_friends.policies.ppo_policy import PPOPolicy as RefPolicy
    return ref_ppo, RefPolicy


def _b200_policy():
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.spaces import Box, Discrete
    return PPOPolicy("p", Discrete(2), Box(-np.inf, np.inf, (4,)), Box(-np.inf, np.inf, (4,)), envs_per_proc=2,
                     actor_kw_args={"activation": torch.nn.LeakyReLU()}, critic_kw_args={"activation": torch.nn.LeakyReLU()})


def _param_names(fn):
    return [p.name for p in inspect.signature(fn).parameters.values() if p.kind != p.VAR_KEYWORD]


def test_every_policy_member_the_reference_trainer_touches_exists():
    used = set(SURFACE["trainer_policy_members"])
    if ref_harness.available():
        _reference()
        src = open(os.path.join(ref_harness.REFERENCE_ROOT, "ppo.py")).read()
        live = set(re.findall(r"self\.policies\[[^\]]+\]\.([A-Za-z_][A-Za-z_0-9]*)", src))
        live |= set(re.findall(r"\bpolicy\.([A-Za-z_][A-Za-z_0-9]*)", src))
        assert live - OUT_OF_SCOPE <= used, sorted(live - OUT_OF_SCOPE - used)
    assert {"have_step_constraints", "have_reset_constraints", "seed", "freeze", "get_inference_actions",
            "apply_step_constraints", "add_episode_info", "end_episodes", "finalize_dataset"} <= used
    pol = _b200_policy()
    missing = sorted(m for m in used - OUT_OF_SCOPE - SET_BY_FINALIZE if not hasattr(pol, m))
    assert not missing, f"PPOPolicy lacks members the reference PPO uses: {missing}"
    fin = inspect.getsource(type(pol).finalize) + inspect.getsource(type(pol)._initialize_networks) + \
        inspect.getsource(type(pol).initialize_dataset)
    for m in SET_BY_FINALIZE & used:
        assert re.search(r"self\.%s\b" % m, fin), f"{m} is not set by finalize()/initialize_dataset()"


def test_policy_method_signatures_match_the_reference_class():
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    ref_methods, ref_ctor = SURFACE["policy_method_params"], set(SURFACE["policy_ctor_params"])
    assert len(ref_methods) == 25
    if ref_harness.available():
        _, RefPolicy = _reference()
        for name, params in ref_methods.items():
            assert _param_names(getattr(RefPolicy, name)) == params, name
        assert set(inspect.signature(RefPolicy.__init__).parameters) <= ref_ctor
    for name, params in ref_methods.items():
        assert _param_names(getattr(PPOPolicy, name)) == params, (name, str(inspect.signature(getattr(PPOPolicy, name))))
    # constructor: every keyword a runner file may pass is accepted under the same name
    our_ctor = inspect.signature(PPOPolicy.__init__).parameters
    assert ref_ctor - {"kw_args"} <= set(our_ctor), sorted(ref_ctor - set(our_ctor))


def test_generate_policy_hook_matches_reference_signature_and_rejects_other_classes():
    from ppo_and_friends_b200.policies.utils import generate_policy
    from ppo_and_friends_b200.spaces import Box, Discrete
    if ref_harness.available():
        _reference()
        from ppo_and_friends.policies.utils import generate_policy as ref_generate
        assert list(inspect.signature(ref_generate).parameters) == SURFACE["generate_policy_params"]
    assert list(inspect.signature(generate_policy).parameters) == SURFACE["generate_policy_params"]

    class MATPolicy:            # stands in for the reference's policies/mat_policy.py class: rejected by name
        pass
    box = Box(-np.inf, np.inf, (4,))
    pol = generate_policy(policy_name="p", policy_class=None, actor_observation_space=box, critic_observation_space=box,
                          action_space=Discrete(3), test_mode=False, envs_per_proc=1)
    assert type(pol).__name__ == "PPOPolicy" and pol.action_pred_size == 3
    with pytest.raises(RuntimeError):
        generate_policy(policy_name="p", policy_class=MATPolicy, actor_observation_space=box,
                        critic_observation_space=box, action_space=Discrete(3), test_mode=False, envs_per_proc=1)
    with pytest.raises(RuntimeError):          # a network class without a CUDA counterpart must not be silently ignored
        generate_policy(policy_name="p", policy_class=None, actor_observation_space=box, critic_observation_space=box,
                        action_space=Discrete(3), test_mode=False, envs_per_proc=1, ac_network=torch.nn.LSTM)


# ---------------------------------------------------------------------------------------------- end to end (GPU)
def _run_reference_trainer(device, swapped, monkeypatch, continuous, iters=2):
    ref_ppo, RefPolicy = _reference()
    import gymnasium.spaces as sp
    from toy_env import make_toy_env_class
    from ppo_and_friends.environments.gym.wrappers import SingleAgentGymWrapper
    from ppo_and_friends.networks.ppo_networks.feed_forward import FeedForwardNetwork
    from ppo_and_friends.policies.utils import get_single_policy_defaults
    ToyEnv = make_toy_env_class(sp.Box, sp.Discrete)
    env_generator = lambda: SingleAgentGymWrapper(ToyEnv(continuous=continuous))   # noqa: E731
    kw = {"activation": torch.nn.LeakyReLU(), "hidden_size": 32}
    policy_args = {"ac_network": FeedForwardNetwork, "actor_kw_args": kw, "critic_kw_args": dict(kw), "lr": 2e-3}
    policy_settings, policy_mapping_fn = get_single_policy_defaults(env_generator=env_generator, policy_args=policy_args)
    if swapped:      # the four edits of INTEGRATION.md §2, applied to the unmodified module
        from ppo_and_friends_b200.policies.utils import generate_policy
        from ppo_and_friends_b200.ppo import _Loader, ppo_batch_train
        from ppo_and_friends_b200.utils.misc import RunningStatNormalizer
        monkeypatch.setattr(ref_ppo, "generate_policy", generate_policy)                                   # (a)
        monkeypatch.setattr(ref_ppo, "RunningStatNormalizer", RunningStatNormalizer)                       # (b)
        monkeypatch.setattr(ref_ppo, "DataLoader", lambda dataset, batch_size, shuffle=True: _Loader(dataset, batch_size))  # (c)
        monkeypatch.setattr(ref_ppo.PPO, "_ppo_batch_train", lambda self, dl, pid: ppo_batch_train(self, dl, pid))  # (d)
    torch.manual_seed(0)
    np.random.seed(0)
    state = tempfile.mkdtemp()
    ppo = ref_ppo.PPO(env_generator=env_generator, policy_settings=policy_settings, policy_mapping_fn=policy_mapping_fn,
                      device=device, batch_size=64, ts_per_rollout=128, max_ts_per_ep=32, epochs_per_iter=2, random_seed=7,
                      envs_per_proc=2, obs_clip=(-10., 10.), reward_clip=(-10., 10.), normalize_obs=True,
                      normalize_rewards=True, normalize_adv=True, state_path=state, checkpoint_every=1000,
                      save_train_scores=False)
    return ppo


def _status(ppo):
    sd = ppo.status_dict["single_agent"]
    keys = ("actor loss", "critic loss", "kl avg", "weighted entropy", "score avg", "natural score avg", "top score")
    return {k: float(sd[k]) for k in keys}, dict(ppo.status_dict["global status"])


@requires_reference
@pytest.mark.gpu
@pytest.mark.parametrize("continuous", [False, True])
def test_unmodified_reference_trainer_runs_on_the_b200_path(monkeypatch, continuous):
    """PPO.__init__ -> learn() (2 iterations: rollout, dataset, 2 epochs each, checkpoint at the end) of the UNMODIFIED
    reference with the four edits, against the same trainer run stock on the CPU from the same initial weights."""
    ref = _run_reference_trainer("cpu", False, monkeypatch, continuous)
    init = {n: {k: v.detach().clone() for k, v in getattr(ref.policies["single_agent"], n).state_dict().items()}
            for n in ("actor", "critic")}
    torch.manual_seed(11)
    np.random.seed(11)
    ref.learn(num_timesteps=2 * 128 * 2)                 # stock, before the module is patched
    ours = _run_reference_trainer("cuda", True, monkeypatch, continuous)
    pol = ours.policies["single_agent"]
    assert type(pol).__module__.startswith("ppo_and_friends_b200")
    pol.actor.load_state_dict(init["actor"])
    pol.critic.load_state_dict(init["critic"])
    torch.manual_seed(11)
    np.random.seed(11)
    ours.learn(num_timesteps=2 * 128 * 2)
    (rs, rg), (os_, og) = _status(ref), _status(ours)
    assert rg["iteration"] == og["iteration"] == 2 and rg["timesteps"] == og["timesteps"]
    assert rg["total episodes"] == og["total episodes"] and rg["longest episode"] == og["longest episode"]
    for k in rs:
        assert abs(os_[k] - rs[k]) <= 2e-3 * max(abs(rs[k]), 1e-2), (k, os_[k], rs[k])
    # the policies end up with the same weights (two iterations x 2 epochs x 4 minibatches)
    for n in ("actor", "critic"):
        ref_sd = getattr(ref.policies["single_agent"], n).state_dict()
        for k, v in getattr(pol, n).state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref_sd[k].detach().numpy(), rtol=2e-3, atol=2e-5, err_msg=f"{n}/{k}")


@requires_reference
def test_reference_cpu_arm_runs_with_two_ranks_over_gloo():
    """bench.py's CPU arm: the unmodified reference in two worker processes, its mpi4py calls (mpi_avg_gradients,
    RunningMeanStd's allgather, broadcast_model_parameters) carried by gloo through the COMM_WORLD stand-in."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    from oracle import ref_bench
    w = dict(bench.WORKLOADS["c1"], ts=64, E=2, B=64, epochs=2)
    one = ref_bench.run(w, n_ranks=1, steps=1, warmup=0, epochs_timed=1, port=29731)
    two = ref_bench.run(w, n_ranks=2, steps=1, warmup=0, epochs_timed=1, port=29733)
    assert one["kind"] == two["kind"] == "reference" and two["ranks"] == 2
    assert two["threads_per_rank"] <= max(one["threads_per_rank"] // 2, 1)          # set_torch_threads: threads / num_procs
    assert one["value"] > 0 and two["value"] > 0

@requires_reference
@pytest.mark.timeout(600)
def test_reference_cpu_arm_under_a_torchrun_environment(monkeypatch):
    """`bench.py --impl reference --gpus N` is launched by torchrun for N > 1: rank 0 spawns the gloo workers with the
    elastic agent's environment inherited.  TORCHELASTIC_USE_AGENT_STORE would make the workers look for the agent's
    store on THEIR port (nobody serves it: the rendezvous hangs), so the workers must shed that environment."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    from oracle import ref_bench
    for k, v in dict(TORCHELASTIC_USE_AGENT_STORE="True", TORCHELASTIC_RUN_ID="none", TORCHELASTIC_RESTART_COUNT="0",
                     TORCHELASTIC_MAX_RESTARTS="0", LOCAL_RANK="0", RANK="0", WORLD_SIZE="2", LOCAL_WORLD_SIZE="2",
                     GROUP_RANK="0", ROLE_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29799", OMP_NUM_THREADS="1").items():
        monkeypatch.setenv(k, v)
    w = dict(bench.WORKLOADS["c1"], ts=32, E=2, B=32, epochs=1)
    two = ref_bench.run(w, n_ranks=2, steps=1, warmup=0, epochs_timed=1, port=29737)
    assert two["ranks"] == 2 and two["value"] > 0
