"""
PPOPolicy for the B200 path: the reference class's trainer-facing surface
(policies/ppo_policy.py:25-1419) with the hot half re-implemented on device.

Kept (same names, argument meaning, error text): constructor hyper-parameters (:33-300),
`register_agent`, `finalize` (:302-345), `initialize_episodes` (:474-504), `initialize_dataset`
(:506-526), `add_episode_info` (:545-651), `end_episodes` (:653-712), `finalize_dataset` (:714-719),
`clear_dataset` (:721-727), `evaluate` (:891-952), `get_critic_values` (:1057-1071),
`update_learning_rate` (:1073-1084), `get_bs_clip_range` (:1086-1112), attributes `actor`, `critic`,
`actor_optim`, `critic_optim`, `dataset`, `surr_clip`, `vf_clip`, `entropy_weight()`, `lr()`,
`kl_loss_weight`, `target_kl`, `use_huber_loss`, `using_lstm`, `frozen`, `enable_icm`.

Changed on purpose: there are no per-segment EpisodeInfo objects and no autograd.  The rollout goes
into a packed device ring, segments into a table, and `update_weights(actor_loss, critic_loss)` has
no counterpart because the losses never exist as tensors — the fused step in ppo.py
(`ppo_batch_train`) replaces `PPO._ppo_batch_train` + `evaluate` + `update_weights` as one unit.
MultiDiscrete action spaces take a multi-categorical head (reference MultiCategoricalDistribution,
networks/distributions.py:272-438, restated: softmax over the whole actor output, one Categorical per section, log-prob
and entropy summed over the sections); `nvec` must be 1-D with `start` = 0, every entry >= 1 and sum(nvec) <= 64.
MultiBinary action spaces take a Bernoulli head (reference BernoulliDistribution, networks/distributions.py:134-196,
restated: one Bernoulli(probs=sigmoid(actor output)) per column, log-prob and entropy summed over the columns, fp32 0/1
actions); the shape must be 1-D with 1 <= n <= 64.
Discrete spaces take 1 <= n <= 65536 actions (n <= 64: the multi-categorical head with one section; wider: the
Categorical head's wide kernels) and Box spaces 1 .. 4096 flattened dimensions.
Out of scope (raise): LSTM networks, ICM, MAT, Mixed action heads.
"""
import os

import numpy as np
import torch

from .. import _lib, ops
from ..networks.feed_forward import PolicyNetworks, _AdamView, hidden_sizes
from ..utils.episode_info import PPODataset, RolloutRing
from ..utils.misc import update_optimizer_lr
from ..utils.mpi_utils import abort, barrier, broadcast_model_parameters, get_rank, rank_print


MAX_DISCRETE_ACTIONS = 65536      # include/ppoaf_b200.h: the Categorical and Gaussian heads' widest rows
MAX_BOX_DIMS = 4096


class CallableValue:
    """utils/schedulers.py:11-29: a constant that looks like a scheduler."""

    def __init__(self, value):
        self.value = value

    def finalize(self, status_dict):
        pass

    def __call__(self):
        return self.value


def _as_callable(v):
    return v if callable(v) else CallableValue(v)


def space_dtype_str(space):
    """utils/misc.py:17-46, duck-typed so gymnasium itself is not required."""
    if hasattr(space, "spaces"):
        return "mixed"
    dt = np.dtype(getattr(space, "dtype", np.float32))
    if np.issubdtype(dt, np.floating):
        return "continuous"
    if np.issubdtype(dt, np.integer):
        name = type(space).__name__
        if name == "Discrete" or (hasattr(space, "n") and not hasattr(space, "nvec") and tuple(getattr(space, "shape", ())) == ()):
            return "discrete"
        if name == "MultiBinary":
            return "multi-binary"
        if name == "MultiDiscrete" or hasattr(space, "nvec"):
            return "multi-discrete"
    return "unknown"


def _flat_dim(space):
    shape = tuple(getattr(space, "shape", ()) or ())
    return int(np.prod(shape)) if len(shape) else 1


class PPOPolicy:

    def __init__(self, name, action_space, actor_observation_space, critic_observation_space, envs_per_proc,
                 bootstrap_clip=(-100., 100.), ac_network=None, actor_kw_args={}, critic_kw_args={}, icm_kw_args={},
                 target_kl=100., surr_clip=0.2, vf_clip=None, gradient_clip=0.5, lr=3e-4, icm_lr=3e-4,
                 entropy_weight=0.01, kl_loss_weight=0.0, use_gae=True, gamma=0.99, lambd=0.95,
                 dynamic_bs_clip=False, enable_icm=False, agent_shared_icm=False, icm_network=None,
                 intr_reward_weight=1.0, icm_beta=0.8, use_huber_loss=False, test_mode=False, verbose=False,
                 **kw_args):
        if enable_icm:
            abort("ERROR: ICM is outside the B200 update path (SURVEY.md §2 row 11).")
        if ac_network is not None and getattr(ac_network, "__name__", str(ac_network)) != "FeedForwardNetwork":
            # the reference instantiates `ac_network` (policies/ppo_policy.py:390-446); only its FeedForwardNetwork
            # (networks/ppo_networks/feed_forward.py) has a CUDA counterpart here, anything else must not be ignored
            abort("ERROR: ac_network {} is outside the B200 update path (FeedForwardNetwork only).".format(ac_network))
        self.name = name
        self.action_space = action_space
        self.actor_obs_space = actor_observation_space
        self.critic_obs_space = critic_observation_space
        self.enable_icm = False
        self.test_mode = test_mode
        self.use_gae, self.gamma, self.lambd = use_gae, gamma, lambd
        self.dynamic_bs_clip = dynamic_bs_clip
        self.using_lstm = False
        self.dataset = None
        self.device = torch.device("cpu")
        self.agent_ids = np.array([])
        self.target_kl, self.surr_clip, self.vf_clip = target_kl, surr_clip, vf_clip
        self.gradient_clip, self.kl_loss_weight = gradient_clip, kl_loss_weight
        self.envs_per_proc = envs_per_proc
        self.agent_grouping = False
        # read by PPO.__init__ (reference ppo.py:347-354); the base policy has no constraints (policies/ppo_policy.py:187-189)
        self.have_step_constraints = False
        self.have_reset_constraints = False
        self.agent_shared_icm = False
        self.verbose = verbose
        self.use_huber_loss = use_huber_loss
        self.frozen = False
        self.lr = _as_callable(lr)
        self.entropy_weight = _as_callable(entropy_weight)

        self.action_dtype = space_dtype_str(action_space)
        if self.action_dtype == "unknown":
            abort(f"ERROR: unknown action type: {type(action_space)} with dtype {getattr(action_space, 'dtype', None)}.")
        if self.action_dtype not in ("continuous", "discrete", "multi-discrete", "multi-binary"):
            abort(f"ERROR: {self.action_dtype} action heads are outside the B200 update path "
                  "(Gaussian, Categorical, MultiCategorical and Bernoulli only, SURVEY.md §2 row 8).")
        rank_print("{} policy using {} actions.".format(self.name, self.action_dtype))

        self.have_bootstrap_clip = bootstrap_clip is not None
        if self.have_bootstrap_clip:
            self.bootstrap_clip = (_as_callable(bootstrap_clip[0]), _as_callable(bootstrap_clip[1]))
        else:
            self.bootstrap_clip = None

        # a Discrete space of up to 64 actions is the multi-categorical head's table of one section; a wider one runs
        # the Categorical head's wide kernels and has no section table
        if self.action_dtype == "discrete":
            if not 1 <= int(action_space.n) <= MAX_DISCRETE_ACTIONS:
                abort(f"ERROR: Discrete n = {int(action_space.n)} is outside the 1 .. {MAX_DISCRETE_ACTIONS} actions the "
                      "Categorical head supports.")
            self.nvec = [int(action_space.n)]
        elif self.action_dtype == "multi-discrete":
            nvec = np.asarray(action_space.nvec)
            start = getattr(action_space, "start", None)
            if nvec.ndim != 1 or nvec.size == 0:
                abort(f"ERROR: MultiDiscrete nvec must be a non-empty 1-D array on the B200 path, got shape {nvec.shape}.")
            if start is not None and np.any(np.asarray(start) != 0):
                abort("ERROR: MultiDiscrete spaces with a nonzero start are outside the B200 update path.")
            if np.any(nvec < 1):
                abort(f"ERROR: every MultiDiscrete nvec entry must be >= 1, got {nvec.tolist()}.")
            if int(nvec.sum()) > 64:
                abort(f"ERROR: MultiDiscrete sum(nvec) = {int(nvec.sum())} exceeds the 64 actor outputs the "
                      "multi-categorical head supports.")
            self.nvec = [int(n) for n in nvec]
        elif self.action_dtype == "multi-binary":
            shape = tuple(getattr(action_space, "shape", ()) or ())
            if len(shape) != 1:
                abort(f"ERROR: MultiBinary spaces must be 1-D on the B200 path, got shape {shape}.")
            if not 1 <= int(shape[0]) <= 64:
                abort(f"ERROR: MultiBinary n = {int(shape[0])} is outside the 1 .. 64 actor outputs the Bernoulli "
                      "head supports.")
        elif self.action_dtype == "continuous" and not 1 <= _flat_dim(action_space) <= MAX_BOX_DIMS:
            abort(f"ERROR: Box spaces of {_flat_dim(action_space)} dimensions are outside the 1 .. {MAX_BOX_DIMS} the "
                  "Gaussian head supports.")
        if self.action_dtype in ("continuous", "multi-binary"):
            self.action_dim = _flat_dim(action_space)
            self.action_pred_size = self.action_dim
        else:
            self.action_dim = len(self.nvec)
            self.action_pred_size = sum(self.nvec)
            if not self.wide_categorical:
                self.section_ends = _lib.section_ends(self.nvec)
        self.actor_kw_args = dict(actor_kw_args)
        self.critic_kw_args = dict(critic_kw_args)
        self._ring = None
        self._engine = None

    # ------------------------------------------------------------------------------------------------
    def register_agent(self, agent_id):
        """ppo_policy.py:352-362 (set union, so the order is not insertion order)."""
        self.agent_ids = np.array(list(set(self.agent_ids).union({agent_id})))

    def finalize(self, status_dict, device):
        self.device = torch.device(device)
        _lib.require_cuda()
        ops.runtime_init()
        self.agent_idxs = np.arange(len(self.agent_ids))
        self.num_agents = self.agent_idxs.size
        self._agent_col = {a: i for i, a in enumerate(self.agent_ids)}
        self._initialize_networks()
        for sched in (self.lr, self.entropy_weight):
            sched.finalize(status_dict)
        if self.have_bootstrap_clip:
            self.bootstrap_clip[0].finalize(status_dict)
            self.bootstrap_clip[1].finalize(status_dict)
        self.actor_optim = _AdamView(self.lr(), self.actor)
        self.critic_optim = _AdamView(self.lr(), self.critic)
        self.icm_optim = None

    def _initialize_networks(self):
        """ppo_policy.py:390-472: actor then critic, broadcast from rank 0."""
        gaussian = self.action_dtype == "continuous"
        akw, ckw = self.actor_kw_args, self.critic_kw_args
        a_hidden = hidden_sizes(akw.get("hidden_size", 128), akw.get("hidden_depth", 3))
        c_hidden = hidden_sizes(ckw.get("hidden_size", 128), ckw.get("hidden_depth", 3))
        do, dc = _flat_dim(self.actor_obs_space), _flat_dim(self.critic_obs_space)
        self.min_std = float(akw.get("min_std", 0.01))
        self.nets = PolicyNetworks(
            self.device, [do] + a_hidden + [self.action_pred_size], [dc] + c_hidden + [1],
            akw.get("activation", torch.nn.ReLU()), ckw.get("activation", torch.nn.ReLU()), gaussian,
            self.action_dim, std_offset=akw.get("std_offset", 0.5))
        self.actor, self.critic = self.nets.actor, self.nets.critic
        if gaussian:
            lo = akw.get("distribution_min", getattr(self.action_space, "low", -1.0))
            hi = akw.get("distribution_max", getattr(self.action_space, "high", 1.0))
            self.dist_min = np.asarray(lo, dtype=np.float32).reshape(-1)
            self.dist_max = np.asarray(hi, dtype=np.float32).reshape(-1)
            if np.isinf(self.dist_min).any() or np.isinf(self.dist_max).any():
                abort("ERROR: the gaussian distribution min/max must not be inf; set "
                      "actor_kw_args['distribution_min'/'distribution_max'].")
        broadcast_model_parameters(self.nets.flat_params)
        barrier()

    def seed(self, seed):
        """policies/ppo_policy.py:347-352 (called by PPO.__init__, ppo.py:595): seed the spaces (duck-typed)."""
        for space in (self.action_space, self.actor_obs_space):
            if hasattr(space, "seed"):
                space.seed(seed)

    def freeze(self):
        """policies/ppo_policy.py:1322-1326 (ppo.py:661)."""
        self.frozen = True

    def unfreeze(self):
        self.frozen = False

    def apply_step_constraints(self, *args):
        """policies/ppo_policy.py:1114-1135: the base policy constrains nothing."""
        return args

    def apply_reset_constraints(self, *args):
        """policies/ppo_policy.py:1137-1150."""
        return args

    def shuffle_agent_ids(self):
        """policies/ppo_policy.py:364-371 (only called for agent-grouping policies, ppo.py:1643-1644)."""
        np.random.shuffle(self.agent_ids)

    @property
    def wide_categorical(self):
        """A Discrete space of more than 64 actions: the Categorical head's own entry points, no section table."""
        return self.action_dtype == "discrete" and self.nvec[0] > 64

    @property
    def head(self):
        return {"continuous": _lib.HEAD_GAUSSIAN_TANH, "discrete": _lib.HEAD_CATEGORICAL,
                "multi-discrete": _lib.HEAD_MULTI_CATEGORICAL, "multi-binary": _lib.HEAD_BERNOULLI}[self.action_dtype]

    def to(self, device):
        self.device = torch.device(device)

    def train(self):
        pass

    def eval(self):
        pass

    # -- A0: dataset / episode lifecycle ----------------------------------------------------------------
    def initialize_episodes(self, env_batch_size, status_dict):
        E = int(env_batch_size)
        if self._ring is None or self._ring.E != E or self._ring.A != len(self.agent_ids):
            self._ring = RolloutRing(self.device, E, len(self.agent_ids), _flat_dim(self.actor_obs_space),
                                     _flat_dim(self.critic_obs_space), self.action_dim,
                                     self.action_dtype in ("discrete", "multi-discrete"),
                                     capacity_steps=max(64, getattr(self, "rollout_steps_hint", 64)))
        self._ring.reset()
        if self.dataset is not None:
            self.dataset.ring = self._ring
        A = len(self.agent_ids)
        self._open_t0 = np.zeros((A, E), dtype=np.int64)        # ring step where the open segment began
        self._open_start_ts = np.zeros((A, E), dtype=np.int64)  # EpisodeInfo.starting_ts of the open segment
        clip = self.get_bs_clip_range(None)
        self._open_clip = np.empty((A, E, 2), dtype=np.float64)
        self._open_clip[:] = (np.nan, np.nan) if clip is None else clip

    def initialize_dataset(self):
        self.dataset = PPODataset(self.device, self.action_dtype, sequence_length=1, ring=self._ring,
                                  use_gae=self.use_gae, gamma=self.gamma, lambd=self.lambd)

    def validate_agent_id(self, agent_id):
        if agent_id not in self._agent_col:
            abort(f"ERROR: agent {agent_id} has not been registered with policy {self.name}. "
                  "Make sure that you've set up your policies correctly.")

    # -- A1 ------------------------------------------------------------------------------------------------
    def add_episode_info(self, agent_id, critic_observations, observations, next_observations, raw_actions,
                         actions, values, log_probs, rewards, where_done):
        self.validate_agent_id(agent_id)
        self._ring.add_step(self._agent_col[agent_id], critic_observations, observations, next_observations,
                            raw_actions, actions, values, log_probs, rewards)

    # -- A2 ------------------------------------------------------------------------------------------------
    def end_episodes(self, agent_id, env_idxs, episode_lengths, terminal, ending_values, ending_rewards):
        if self.frozen:
            return
        self.validate_agent_id(agent_id)
        a = self._agent_col[agent_id]
        ring = self._ring
        t_now = int(ring.steps[a])
        ev = _host(ending_values)
        er = _host(ending_rewards)
        env_idxs = np.asarray(env_idxs, dtype=np.int64).reshape(-1)
        k = env_idxs.size
        if k == 0:
            return
        if not (self.have_bootstrap_clip and self.dynamic_bs_clip):
            # every environment of the call at once (the reference loops in Python: policies/ppo_policy.py:676-712).
            # bootstrap arrays are indexed by POSITION in env_idxs, exactly like the reference (:684-689; SURVEY Q5)
            pos = np.arange(k)
            ending_ts = np.asarray(episode_lengths).reshape(-1)[env_idxs].astype(np.int64)
            t0 = self._open_t0[a, env_idxs]
            ending_value = ev[pos].astype(np.float64)
            ending_reward = er[pos].astype(np.float64)
            if self.have_bootstrap_clip:
                clip = self._open_clip[a, env_idxs]
                ending_reward = np.clip(ending_reward, clip[:, 0], clip[:, 1])              # episode_info.py:450-454
            term = np.asarray([bool(terminal[i]) for i in range(k)]) if not isinstance(terminal, np.ndarray) \
                else terminal.reshape(-1)[:k].astype(bool)
            self.dataset.add_segments(a * ring.E + env_idxs, t0, t_now - t0, term, ending_value, ending_reward,
                                      self._open_start_ts[a, env_idxs], ending_ts)
            if self.have_bootstrap_clip:
                self._open_clip[a, env_idxs] = self.get_bs_clip_range(None)
            self._open_start_ts[a, env_idxs] = np.where(term, 0, ending_ts)
            self._open_t0[a, env_idxs] = t_now
            return
        for idx, env_i in enumerate(env_idxs):
            env_i = int(env_i)
            ending_ts = int(episode_lengths[env_i])
            t0 = int(self._open_t0[a, env_i])
            length = t_now - t0
            ending_value = float(ev[idx])
            ending_reward = float(er[idx])
            clip = self._open_clip[a, env_i]
            ending_reward = float(np.clip(ending_reward, clip[0], clip[1]))       # episode_info.py:450-454
            col = a * ring.E + env_i
            self.dataset.add_segment(col, t0, length, bool(terminal[idx]), ending_value, ending_reward,
                                     int(self._open_start_ts[a, env_i]), ending_ts)
            seg_r = ring.segment_rewards(col, t0, length)                         # dynamic clip: this segment's reward range
            self._open_clip[a, env_i] = (float(seg_r.min()), float(seg_r.max()))
            self._open_start_ts[a, env_i] = 0 if terminal[idx] else ending_ts
            self._open_t0[a, env_i] = t_now

    def finalize_dataset(self):
        self.dataset.build()

    def clear_dataset(self):
        self.dataset = None

    def get_bs_clip_range(self, ep_rewards):
        if not self.have_bootstrap_clip:
            return None
        if self.dynamic_bs_clip and ep_rewards is not None:
            return (min(ep_rewards), max(ep_rewards))
        return (self.bootstrap_clip[0](), self.bootstrap_clip[1]())

    # -- P1: forward-only evaluation (also what rollout-time inference builds on) ---------------------------
    def evaluate(self, batch_critic_obs, batch_obs, batch_actions):
        """(values, log_probs, entropy) for a batch, through the CUDA MLP + head kernels."""
        values = self.critic(batch_critic_obs).reshape(-1)
        pred = self.actor(batch_obs)
        acts = batch_actions if torch.is_tensor(batch_actions) else torch.as_tensor(np.asarray(batch_actions))
        if self.action_dtype == "continuous":
            acts = acts.to(self.device, torch.float32).reshape(pred.shape[0], -1).contiguous()
            lp, ent = ops.head_evaluate(self.head, pred, self.actor.state_dict()["distribution.log_std"], acts,
                                        self.min_std)
        elif self.action_dtype == "multi-binary":
            acts = acts.to(self.device, torch.float32).reshape(pred.shape[0], -1).contiguous()
            lp, ent = ops.head_evaluate(self.head, pred, None, acts)
        elif self.wide_categorical:
            acts = acts.to(self.device, torch.int64).reshape(pred.shape[0], -1).contiguous()
            lp, ent = ops.head_evaluate(self.head, pred, None, acts)
        else:
            acts = acts.to(self.device, torch.int64).reshape(pred.shape[0], -1).contiguous()
            lp, ent = ops.multi_categorical_evaluate(pred, self.section_ends, acts)
        return values, lp, ent

    def get_rollout_actions(self, obs):
        """
        (raw_action, action, log_prob) for a batch of observations, with natural exploration
        (reference policies/ppo_policy.py:729-794).  The actor forward, the std scaling, the tanh squashing / range
        mapping and the log-prob run on the device; the random draws come from torch's global CPU generator in exactly
        the order the reference's CPU sampling consumes them (Normal.sample -> normal_(0, 1) of shape [n, act_dim];
        Categorical.sample -> exponential_(1) of shape [n, n_actions]; MultiDiscrete: one Categorical.sample per section,
        in section order; MultiBinary: Bernoulli.sample -> rand of shape [n, n_binary]), so a seeded run reproduces the
        reference's actions.  Returns numpy raw_action / action and a CPU log_prob tensor, like the reference.
        """
        obs = np.asarray(obs) if not torch.is_tensor(obs) else obs
        if len(obs.shape) < 2:
            abort("ERROR: get_rollout_actions expects a batch of observations but "
                  "instead received shape {}.".format(tuple(obs.shape)))
        t_obs = torch.as_tensor(obs, dtype=torch.float32).to(self.device).reshape(obs.shape[0], -1).contiguous()
        n = t_obs.shape[0]
        discrete = self.action_dtype in ("discrete", "multi-discrete")
        action_pred = self.actor(t_obs, softmax_out=discrete)
        if self.wide_categorical:
            noise = torch.empty(n, self.nvec[0], dtype=torch.float32).exponential_(1)
            raw, act, lp = ops.head_sample(self.head, action_pred, None, noise.to(self.device, non_blocking=True))
        elif discrete:
            noise = torch.cat([torch.empty(n, k, dtype=torch.float32).exponential_(1).reshape(-1) for k in self.nvec])
            act, lp = ops.multi_categorical_sample(action_pred, self.section_ends,
                                                   noise.to(self.device, non_blocking=True), len(self.nvec))
            raw = act
        elif self.action_dtype == "multi-binary":
            noise = torch.rand(n, self.action_dim, dtype=torch.float32)
            raw, act, lp = ops.head_sample(self.head, action_pred, None, noise.to(self.device, non_blocking=True),
                                           act_dim=self.action_dim)
        else:
            noise = torch.empty(n, self.action_dim, dtype=torch.float32).normal_(0, 1)
            rescale = bool((self.dist_min != -1.0).any() or (self.dist_max != 1.0).any())
            raw, act, lp = ops.head_sample(self.head, action_pred, self.actor.state_dict()["distribution.log_std"],
                                           noise.to(self.device, non_blocking=True), self.min_std,
                                           self._dist_dev("min") if rescale else None,
                                           self._dist_dev("max") if rescale else None, act_dim=self.action_dim)
        # the reference aborts on NaN observations / predictions (:758-775); one check of the results covers both
        bad = torch.isnan(t_obs).any() | torch.isnan(action_pred).any()
        # ONE device->host transfer and one sync per call: the three results and the NaN flag travel as one byte buffer
        parts = [raw.contiguous().view(torch.uint8).reshape(-1), act.contiguous().view(torch.uint8).reshape(-1),
                 lp.contiguous().view(torch.uint8).reshape(-1), bad.to(torch.uint8).reshape(1)]
        packed = torch.cat(parts)
        host = self._host_out(packed.numel())
        host.copy_(packed, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        o0, o1, o2 = parts[0].numel(), parts[0].numel() + parts[1].numel(), packed.numel() - 1
        raw_h = host[:o0].clone().view(raw.dtype).reshape(raw.shape)
        act_h = host[o0:o1].clone().view(act.dtype).reshape(act.shape)
        lp_h = host[o1:o2].clone().view(lp.dtype).reshape(lp.shape)
        bad_h = bool(host[o2].item())
        if bad_h:
            abort("ERROR: get_rollout_actions received observations or produced action predictions "
                  "containing nan values!")
        if discrete:
            lp_h = lp_h.unsqueeze(-1)
        return raw_h.numpy(), act_h.numpy(), lp_h

    def get_inference_actions(self, obs, deterministic):
        """
        Environment actions only, for `ppoaf test` (reference policies/ppo_policy.py:796-888; ppo.py:972, 1023).
        deterministic: tanh(mean) mapped to the action range (Gaussian, networks/distributions.py:596-631), the arg-max
        class (Categorical, :251-269), the arg-max class of every section ([n, n_sections], MultiDiscrete) or
        [sigmoid(z) > 0.5] as fp32 0/1 ([n, n_binary], MultiBinary); otherwise a sample drawn with the rollout protocol.
        """
        obs = np.asarray(obs) if not torch.is_tensor(obs) else obs
        if len(obs.shape) < 2:
            abort("ERROR: get_inference_actions expects a batch of observations but "
                  "instead received shape {}.".format(tuple(obs.shape)))
        if not deterministic:
            return torch.as_tensor(self.get_rollout_actions(obs)[1])
        t_obs = torch.as_tensor(obs, dtype=torch.float32).to(self.device).reshape(obs.shape[0], -1).contiguous()
        discrete = self.action_dtype in ("discrete", "multi-discrete")
        action_pred = self.actor(t_obs, softmax_out=discrete)
        if self.action_dtype == "multi-discrete":
            return torch.stack([s.argmax(dim=-1) for s in action_pred.split(self.nvec, dim=1)], dim=1).cpu()
        if discrete:
            return torch.argmax(action_pred, dim=-1).cpu()
        n = t_obs.shape[0]
        if self.action_dtype == "multi-binary":
            half = torch.full((n, self.action_dim), 0.5, dtype=torch.float32, device=self.device)   # u = 0.5: p > 0.5
            _, act, _ = ops.head_sample(self.head, action_pred, None, half, act_dim=self.action_dim)
            return act.cpu()
        rescale = bool((self.dist_min != -1.0).any() or (self.dist_max != 1.0).any())
        zeros = torch.zeros(n, self.action_dim, dtype=torch.float32, device=self.device)   # no noise: raw = mean
        _, act, _ = ops.head_sample(self.head, action_pred, self.actor.state_dict()["distribution.log_std"], zeros,
                                    self.min_std, self._dist_dev("min") if rescale else None,
                                    self._dist_dev("max") if rescale else None, act_dim=self.action_dim)
        return act.cpu()

    def _host_out(self, n_bytes):
        """Pinned staging buffer for the per-step device->host result transfer."""
        buf = self.__dict__.get("_host_out_buf")
        if buf is None or buf.numel() < n_bytes:
            buf = torch.empty(max(n_bytes, 4096), dtype=torch.uint8, pin_memory=True)
            self._host_out_buf = buf
        return buf[:n_bytes]

    def _dist_dev(self, which):
        """The Gaussian head's output range as device tensors (built once)."""
        cache = self.__dict__.setdefault("_dist_dev_cache", {})
        if which not in cache:
            src = self.dist_min if which == "min" else self.dist_max
            full = np.broadcast_to(src, (self.action_dim,)).astype(np.float32)
            cache[which] = torch.as_tensor(np.ascontiguousarray(full)).to(self.device)
        return cache[which]

    def get_critic_values(self, obs):
        """Values of a batch of critic observations (reference policies/ppo_policy.py:1057-1071)."""
        return self.critic(obs)

    def update_weights(self, actor_loss, critic_loss):
        raise _lib.PpoafError(
            "PPOPolicy.update_weights(actor_loss, critic_loss) has no counterpart on the B200 path: losses are "
            "never materialised as autograd tensors. Use ppo_and_friends_b200.ppo.ppo_batch_train, which replaces "
            "PPO._ppo_batch_train + evaluate + update_weights as one fused step.")

    # -- checkpoints (reference policies/ppo_policy.py:1152-1300): same directory layout and file formats ----------
    def save(self, save_path, tag="latest"):
        policy_save_path = os.path.join(save_path, "{}-policy".format(self.name), str(tag))
        if get_rank() == 0 and not os.path.exists(policy_save_path):
            os.makedirs(policy_save_path)
        barrier()
        self._save_policies(policy_save_path)
        self._save_optimizers(policy_save_path)

    def load(self, load_path, tag="latest"):
        policy_load_path = os.path.join(load_path, "{}-policy".format(self.name), str(tag))
        self._load_policies(policy_load_path)
        self._load_optimizers(policy_load_path)

    def _save_policies(self, save_path):
        self.actor.save(save_path, get_rank())
        self.critic.save(save_path, get_rank())

    def _load_policies(self, load_path):
        self.actor.load(load_path, get_rank())
        self.critic.load(load_path, get_rank())

    def _save_optimizers(self, save_path):
        if self.test_mode:
            return
        # the NVLS exchange keeps each rank's moments current only on the slice it owns: assemble them first
        peer = getattr(self._engine, "peer", None)
        if hasattr(peer, "gather_moments"):
            peer.gather_moments(self.nets)
        torch.save(self.actor_optim.state_dict(), os.path.join(save_path, f"actor_optim_{get_rank()}"))
        torch.save(self.critic_optim.state_dict(), os.path.join(save_path, f"critic_optim_{get_rank()}"))

    def _load_optimizers(self, load_path):
        if self.test_mode:
            return
        try:
            files = []
            for which in ("actor", "critic"):
                f = os.path.join(load_path, f"{which}_optim_{get_rank()}")
                if not os.path.exists(f):
                    f = os.path.join(load_path, f"{which}_optim_0")
                files.append(f)
            self.nets._loaded_adam_step = None
            self.actor_optim.load_state_dict(torch.load(files[0], weights_only=False))
            self.critic_optim.load_state_dict(torch.load(files[1], weights_only=False))
        except FileNotFoundError:
            rank_print("WARNING: unable to find saved optimizers to load. Skipping...")

    def direct_load(self, policy_load_path):
        self.actor.load(policy_load_path, get_rank())
        self.critic.load(policy_load_path, get_rank())

    def update_learning_rate(self):
        if self.frozen:
            return
        update_optimizer_lr(self.actor_optim, self.lr())
        update_optimizer_lr(self.critic_optim, self.lr())


def _host(x):
    if torch.is_tensor(x):
        return x.detach().cpu().numpy().reshape(-1)
    return np.asarray(x).reshape(-1)
