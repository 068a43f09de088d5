"""Shared builders for the GPU parity tests (the same golden fixtures that pin the oracle), and the float64 clip + Adam
reference of the optimizer kernels (its bounds are derived in test_forward_optim_kernels.py)."""
import math

import numpy as np
import torch

from ppo_and_friends_b200.spaces import Box, Discrete

ACT_MODULES = {"leaky_relu": torch.nn.LeakyReLU, "tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}


def make_policy(ro, act="leaky_relu", actor_hidden=32, critic_hidden=32, depth=3, dist_range=1.0, device="cuda",
                **policy_kw):
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    if ro.n_discrete:
        action_space = Discrete(ro.n_discrete)
    else:
        action_space = Box(-dist_range, dist_range, (ro.act_dim,))
    pol = PPOPolicy("pol", action_space, Box(-np.inf, np.inf, (ro.obs_dim,)), Box(-np.inf, np.inf, (ro.critic_obs_dim,)),
                    envs_per_proc=ro.E,
                    actor_kw_args=dict(activation=ACT_MODULES[act](), hidden_size=actor_hidden, hidden_depth=depth),
                    critic_kw_args=dict(activation=ACT_MODULES[act](), hidden_size=critic_hidden, hidden_depth=depth),
                    **policy_kw)
    for a in ro.agents:
        pol.register_agent(a)
    # the reference's agent order is a set-union order; keep the rollout's order for deterministic columns
    pol.agent_ids = np.array(ro.agents)
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device(device))
    return pol


def policy_kwargs_from_golden(g, prefix=""):
    kw = {}
    if (prefix + "have_bootstrap_clip") in g:
        if bool(g[prefix + "have_bootstrap_clip"]):
            bc = g[prefix + "bootstrap_clip"]
            kw["bootstrap_clip"] = (float(bc[0]), float(bc[1]))
        else:
            kw["bootstrap_clip"] = None
    for k in ("use_gae", "dynamic_bs_clip"):
        if (prefix + k) in g:
            kw[k] = bool(g[prefix + k])
    for k in ("gamma", "lambd"):
        if (prefix + k) in g:
            kw[k] = float(g[prefix + k])
    return kw


def run_device_rollout(pol, ro, tensor_bootstrap=False):
    from ppo_and_friends_b200.synthetic import replay_rollout
    pol.initialize_dataset()
    pol.initialize_episodes(ro.E, {"global status": {"iteration": 0, "timesteps": 0}})
    wrap = (lambda x: torch.tensor(x, requires_grad=True)) if tensor_bootstrap else None
    replay_rollout(lambda a: pol, ro, to_bootstrap=wrap)
    pol.finalize_dataset()
    return pol.dataset


def rel_err(a, b, floor):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


# ---- float64 clip + Adam reference (csrc/optim.cu, csrc/peer.cu) -----------------------------------------------------
U = 2.0 ** -24
HP_BASE = dict(LR=3e-4, GRAD_CLIP=0.5, BETA1=0.9, BETA2=0.999, ADAM_EPS=1e-5, INV_WORLD=1.0)


def f32(x):
    return float(np.float32(x))


def clip_coef64(sumsq, max_norm, inv_world, f32_scalars=True):
    """torch clip_grad_norm_'s coefficient of a network whose summed gradient has this sum of squares."""
    if max_norm < 0:
        return 1.0
    mn, tiny = (f32(max_norm), f32(1e-6)) if f32_scalars else (max_norm, 1e-6)
    with np.errstate(invalid="ignore"):
        c = mn / (math.sqrt(sumsq) * inv_world + tiny) if not math.isnan(sumsq) else math.nan
    return c if math.isnan(c) else min(c, 1.0)


def adam_scalars(hp, t, f32_scalars=True):
    """The scalars of one step (optim.cu adam_update_kernel), with torch's beta^t."""
    lr, b1, b2, eps, iw = hp["LR"], hp["BETA1"], hp["BETA2"], hp["ADAM_EPS"], hp["INV_WORLD"]
    s = dict(neg_step=-(lr / (1 - b1 ** t)), bc2s=math.sqrt(1 - b2 ** t), w1=1 - b1, b2=b2, w2=1 - b2, eps=eps, iw=iw)
    return {k: f32(v) for k, v in s.items()} if f32_scalars else s


def adam_step64(p, g, m, v, t, hp, n_actor, f32_scalars=True, g_err=None):
    """One clip + Adam step in float64 -> (p, m, v, [coef_a, coef_c], bounds dict).  g_err: an absolute bound per
    element on the error of the gradient the kernel sees (a sum in an unspecified order); it enters the clip
    coefficient as ||g_err|| / ||g|| per network and the scaled gradient as inv_world coef g_err."""
    p, g, m, v = (np.asarray(a, np.float64) for a in (p, g, m, v))
    s = adam_scalars(hp, t, f32_scalars)
    with np.errstate(invalid="ignore", over="ignore"):
        # float32 squares, as torch's float32 norm and the kernel take them (a 1e20 entry overflows to inf)
        sq = np.square(g.astype(np.float32)).astype(np.float64) if f32_scalars else np.square(g)
        coefs = [clip_coef64(float(sq[:n_actor].sum()), hp["GRAD_CLIP"], s["iw"], f32_scalars),
                 clip_coef64(float(sq[n_actor:].sum()), hp["GRAD_CLIP"], s["iw"], f32_scalars)]
        coef = np.empty_like(g)
        coef[:n_actor], coef[n_actor:] = coefs
        gk = g * s["iw"] * coef
        m1 = m + s["w1"] * (gk - m)
        v1 = v * s["b2"] + s["w2"] * gk * gk
        denom = np.sqrt(v1) / s["bc2s"] + s["eps"]
        step = s["neg_step"] * m1 / denom
        p1 = p + step
        # error bounds of the kernel's float32 evaluation (module docstring)
        coef_rel = np.where(coef < 1.0, 7 * U, 0.0)
        gk_err = (2 * U + coef_rel) * np.abs(gk)
        if g_err is not None:
            g_err = np.broadcast_to(np.asarray(g_err, np.float64), g.shape)
            for sl in (slice(0, n_actor), slice(n_actor, None)):
                norm = math.sqrt(float(sq[sl].sum()))
                if norm > 0:
                    coef_rel[sl] += np.where(coef[sl] < 1.0, float(np.linalg.norm(g_err[sl])) / norm + U, 0.0)
            gk_err = (2 * U + coef_rel) * np.abs(gk) + s["iw"] * coef * g_err
        e_m = 4 * U * (np.abs(m) + s["w1"] * np.abs(gk)) + s["w1"] * gk_err
        e_v = 3 * U * (s["b2"] * np.abs(v) + s["w2"] * gk * gk) + 2 * s["w2"] * np.abs(gk) * gk_err
        rel_v = np.divide(e_v, v1, out=np.zeros_like(v1), where=v1 > 0)
        e_p = abs(s["neg_step"]) * e_m / denom + (18 * U + rel_v / 2) * np.abs(step) + U * np.abs(p1)
    return p1, m1, v1, coefs, dict(p=e_p, m=e_m, v=e_v)
