#!/usr/bin/env python
"""
bench.py — PPO-AF post-rollout update path on B200.

    python bench.py --gpus N --steps K --warmup W [--workload c4|c3|c5|c1] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: launched by torch.distributed.run, one rank per GPU, NCCL)

Metric (BASELINE.json): "PPO update env-steps/sec at 1/2/4/8 B200; GAE+norm GB/s vs HBM peak".

One STEP = one pass of the hot path over one synthetic rollout shard per rank:
    finalize_dataset (segment table -> flat map -> ring gathers -> GAE/RTG segmented scan)
    + every epoch / minibatch of the PPO update (forward, fused loss, backward, [NCCL all-reduce],
      clip, Adam), KL early stop disabled so every step does the same K_epochs*ceil(N/B) minibatches.
`value` = env-steps/s with the rollout ring already resident in HBM; `e2e` = the same pass started
from the pinned HOST ring (bulk H2D of the ring + segment table inside the timed region, D2H of the
epoch statistics).  The GAE + normalisation microbench (BASELINE configs[1]: 2^22 timesteps, obs 376)
runs on rank 0 in the same invocation and feeds `microbench` (with its own HBM roofline); `roofline` describes the
dominant kernel of the timed region, the grouped GEMM launches of the minibatch step.  `step_engines` (N = 1) times the opt-in
one-launch TMA + tcgen05 engine (PPOAF_STEP=fused) on the same workload right after the default launch chain.  With KL early
stop disabled the trainer keeps one epoch in flight (no host wait between epochs; PPOAF_PIPELINE_EPOCHS=0 turns that off).
The CPU baseline is the UNMODIFIED reference (oracle/_ref: a git-ignored copy made by oracle/build_ref.py in the
build container, which travels to the GPU box like the built .so) timed on this box's host cores on a bounded
sample; the oracle port (oracle/) is reported beside it.  `--impl reference` prints the reference arm on its own,
with --gpus N ranks over gloo.
"""
import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # SURVEY.md §8(d).  ts = steps per rollout, E = envs per rank, A = agents sharing the policy
    "c4": dict(name="M-C4 Humanoid-shaped DD-PPO update", ts=512, E=64, agents=1, Do=376, Dc=376, Da=17, n_disc=0,
               actor_hidden=256, critic_hidden=256, act="tanh", dist_range=0.4, lr=1e-4, B=512, epochs=8,
               max_ts_per_ep=16, shared_critic=False),
    "c3": dict(name="M-C3 LunarLanderContinuous-shaped update", ts=1024, E=64, agents=1, Do=8, Dc=8, Da=2, n_disc=0,
               actor_hidden=64, critic_hidden=256, act="leaky_relu", dist_range=1.0, lr=3e-4, B=512, epochs=16,
               max_ts_per_ep=32, shared_critic=False),
    "c5": dict(name="M-C5 MPE simple_spread-shaped MAPPO update", ts=256, E=64, agents=3, Do=18, Dc=54, Da=1, n_disc=5,
               actor_hidden=128, critic_hidden=256, act="leaky_relu", dist_range=1.0, lr=3e-4, B=128, epochs=10,
               max_ts_per_ep=64, shared_critic=True),
    "c1": dict(name="M-C1 CartPole-shaped update", ts=256, E=1, agents=1, Do=4, Dc=4, Da=1, n_disc=2,
               actor_hidden=128, critic_hidden=128, act="leaky_relu", dist_range=1.0, lr=2e-3, B=256, epochs=10,
               max_ts_per_ep=32, shared_critic=False),
}

STATUS_KEYS = ("actor loss", "critic loss", "kl avg", "weighted entropy")   # order of status.npy (--dump-outputs)
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p["bf16_tflops"]),
                    bf16_tflops_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def build_workload(w, rank, device):
    """Synthetic rollout shard + policy; old values / log-probs come from the same random nets."""
    from helpers import make_policy
    from ppo_and_friends_b200.synthetic import make_rollout
    agents = tuple(f"agent_{i}" for i in range(w["agents"]))
    ro = make_rollout(seed=1234 + rank, T=w["ts"], E=w["E"], agents=agents, obs_dim=w["Do"], critic_obs_dim=w["Dc"],
                      act_dim=w["Da"], n_discrete=w["n_disc"], max_ts_per_ep=w["max_ts_per_ep"], obs_scale=False,
                      shared_critic_obs=w["shared_critic"])
    torch.manual_seed(4321)                       # same init on every rank (then broadcast from rank 0 anyway)
    pol = make_policy(ro, act=w["act"], actor_hidden=w["actor_hidden"], critic_hidden=w["critic_hidden"],
                      dist_range=w["dist_range"], lr=w["lr"], target_kl=float("inf"), device=device)
    rng = np.random.default_rng(99 + rank)
    T, E = ro.T, ro.E
    for a in agents:
        obs = ro.obs[a].reshape(T * E, -1)
        cobs = ro.critic_obs[a].reshape(T * E, -1)
        ro.values[a] = pol.critic(cobs).cpu().numpy().reshape(T, E)
        ro.next_values[a] = np.roll(ro.values[a], -1, axis=0)
        pred = pol.actor(obs)
        if w["n_disc"]:
            probs = torch.softmax(pred, -1)
            act = torch.multinomial(probs, 1)
            ro.raw_actions[a] = act.cpu().numpy().reshape(T, E, 1)
            ro.actions[a] = ro.raw_actions[a].copy()
            _, lp, _ = pol.evaluate(cobs, obs, act)
        else:
            sd = max(math.log1p(math.exp(-0.5)), 0.01)
            raw = (pred.cpu().numpy() + sd * rng.standard_normal((T * E, w["Da"]))).astype(np.float32)
            ro.raw_actions[a] = raw.reshape(T, E, -1)
            ro.actions[a] = np.tanh(ro.raw_actions[a])
            _, lp, _ = pol.evaluate(cobs, obs, raw)
        ro.log_probs[a] = lp.cpu().numpy().reshape(T, E)
    return ro, pol


class HotPath:
    """The timed unit: rollout ring (+ segment table) -> dataset -> all epochs."""

    def __init__(self, w, ro, pol):
        from ppo_and_friends_b200.ppo import PPOUpdateState
        from ppo_and_friends_b200.synthetic import replay_rollout
        self.w, self.ro, self.pol = w, ro, pol
        pol.initialize_dataset()
        pol.initialize_episodes(ro.E, {})
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        replay_rollout(lambda a: pol, ro)                 # the caller side of the path: add_episode_info / end_episodes per step
        pol._ring.wait_copies()
        torch.cuda.synchronize()
        self.record_s = time.perf_counter() - t0          # host cost of A1/A2 for the whole rollout (incl. the per-step H2D)
        self.seg = pol.dataset._seg                       # the segment table recorded by end_episodes
        self.state = PPOUpdateState({"pol": pol}, batch_size=w["B"], epochs_per_iter=w["epochs"])
        self.n = ro.T * ro.E * len(ro.agents)
        self.n_mb = (self.n + w["B"] - 1) // w["B"]
        self.h2d_events = []

    def step(self, from_host=False):
        from ppo_and_friends_b200.ppo import train_policies
        pol = self.pol
        if from_host:                                     # e2e: the pinned host ring crosses PCIe inside the timed region
            ring = pol._ring
            used = int(ring.steps.max())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ring.dev[:used].copy_(ring.host[:used], non_blocking=True)
            e1.record()
            self.h2d_events.append((e0, e1))
        pol.initialize_dataset()
        pol.dataset.ring = pol._ring
        pol.dataset._seg = self.seg
        pol.finalize_dataset()
        epochs = train_policies(self.state)
        return epochs["pol"]

    def h2d_bytes(self):
        ring = self.pol._ring
        used = int(ring.steps.max())
        seg = len(self.seg["col"]) * (4 + 4 + 4 + 1 + 4 + 4) + (len(self.seg["col"]) + 1) * 8
        perm = self.n * 8 * self.w["epochs"]
        return used * ring.C * ring.row_words * 4 + seg + perm

    def d2h_bytes(self):
        return 64 * self.w["epochs"]

    def outputs(self):
        """What a caller of `step` receives from its last call: the status scalars, the trained actor / critic parameters,
        the dataset's advantages, rewards-to-go and values, and the value normaliser's running statistics."""
        sd = self.state.status_dict["pol"]
        out = {"status": np.array([sd[k] for k in STATUS_KEYS], dtype=np.float64)}
        for net in ("actor", "critic"):
            for k, v in getattr(self.pol, net).state_dict().items():
                out[f"{net}.{k}"] = v.detach().float().cpu().numpy()
        ds = self.pol.dataset
        for k in ("advantages", "rewards_to_go", "values"):
            out[k] = getattr(ds, k).float().cpu().numpy()
        out["value_normalizer"] = self.state.value_normalizers["pol"].running_stats.state.double().cpu().numpy()
        return out

    def launches_per_step(self):
        """Kernels of libppoaf_b200.so launched per step (torch's own fills / copies are not counted)."""
        world = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
        layers = 4                                         # Linear layers per net (hidden_depth 3 + output)
        # grouped fwd (heads are fused into the loss kernel), loss + heads, grouped bwd, optimizer (R > 1: the fused
        # exchange + clip + Adam kernel; only the NCCL fallback adds a norm pass)
        nccl = world > 1 and os.environ.get("PPOAF_PEER", "1") == "0"
        per_mb = (layers - 1) + 1 + (layers - 1) + 1 + (1 if nccl else 0)
        per_epoch = 2 + per_mb * self.n_mb                 # epoch_prepare + value_stats_sequence
        finalize = 1 + 8 + 1                               # flat map, 8 field gathers, segmented scan
        return finalize + per_epoch * self.w["epochs"]


def flops_per_sample_visit(w):
    def pmm(dims):
        return sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    pred = w["n_disc"] if w["n_disc"] else w["Da"]
    a = pmm([w["Do"]] + [w["actor_hidden"]] * 3 + [pred])
    c = pmm([w["Dc"]] + [w["critic_hidden"]] * 3 + [1])
    return 6 * (a + c)


def measure_fp32_peak(n=4096, iters=5):
    """cuBLAS SGEMM with TF32 off: the fp32 FMA throughput this GPU sustains (the pipe the update's GEMM tiles run on)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        a = torch.randn(n, n, device="cuda"); b = torch.randn(n, n, device="cuda")
        torch.matmul(a, b); torch.cuda.synchronize()
        best = 1e9
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def kernel_shares(hp):
    """Device time per kernel name over one hot-path step (untimed, after the measurement), from CUPTI activity records."""
    try:
        from torch.profiler import ProfilerActivity, profile
        hp.step(False); torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            hp.step(False)
            torch.cuda.synchronize()
        kernels, total = {}, 0.0
        for e in prof.key_averages():
            us = float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
            if us <= 0 or "memcpy" in e.key.lower() or "memset" in e.key.lower():
                continue
            kernels[e.key[:96]] = {"us": us, "count": int(e.count)}
            total += us
        if not kernels:
            return None
        top = dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us"])[:8])
        return {"total_us": total, "kernels": top}
    except Exception:
        return None


def dump_outputs(outputs, out_dir):
    """One `<name>.npy` per output array (float32 / float64), so that two builds can be compared array by array."""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in outputs.items():
        assert arr.dtype in (np.float32, np.float64), (name, arr.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def time_steps(fn, steps, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if torch.distributed.is_initialized():
        torch.distributed.barrier()
    total_ms = 0.0
    for _ in range(steps):
        if flush is not None:
            flush.add_(1)                                  # evict L2 (256 MB > 126 MB) between timed iterations
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        total_ms += e0.elapsed_time(e1)
    if torch.distributed.is_initialized():
        torch.distributed.barrier()
        t = torch.tensor([total_ms], device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        total_ms = float(t.item())
    return total_ms


# ------------------------------------------------------------------------------------------------------
def microbench_c2(pk, iters=5):
    """BASELINE configs[1]: 2^22 timesteps, obs dim 376, fp32.  Each piece timed alone with CUDA events."""
    from ppo_and_friends_b200 import ops
    from ppo_and_friends_b200.utils.stats import RunningMeanStd
    n, D = 1 << 22, 376
    rng = np.random.default_rng(1234)
    # segments: forced end every 64 steps + Bernoulli(0.02) ends (terminated or truncated)
    lens = []
    left = n
    geo = rng.geometric(0.02, size=n // 16)
    gi = 0
    while left > 0:
        L = int(min(left, 64, geo[gi])); gi += 1
        lens.append(L); left -= L
    lens = np.asarray(lens, dtype=np.int64)
    n_seg = len(lens)
    off = np.zeros(n_seg + 1, dtype=np.int64); np.cumsum(lens, out=off[1:])
    term = rng.random(n_seg) < 0.5
    flag = np.zeros(n, dtype=np.uint8); flag[off[1:] - 1] = 1 + 2 * term.astype(np.uint8)
    d = lambda x: torch.as_tensor(x).cuda()
    g = torch.Generator(device="cuda"); g.manual_seed(1234)
    r = torch.randn(n, device="cuda", generator=g); v = torch.randn(n, device="cuda", generator=g)
    vb = torch.where(d(term), torch.zeros(n_seg, device="cuda"), torch.randn(n_seg, device="cuda", generator=g))
    rb = vb.clamp(-100, 100)
    flag_d, off_d = d(flag), d(off)
    mu = torch.empty(D, device="cuda").uniform_(-3, 3, generator=g)
    sd = torch.empty(D, device="cuda").uniform_(0.1, 10, generator=g)
    obs = torch.randn((n, D), device="cuda", generator=g).mul_(sd).add_(mu)
    out = torch.empty_like(obs)
    adv = torch.empty(n, device="cuda"); rtg = torch.empty(n, device="cuda"); rtg_n = torch.empty(n, device="cuda")
    rms = RunningMeanStd(shape=(D,)); vrms = RunningMeanStd(shape=())
    triple = torch.empty(2 * D + 1, dtype=torch.float64, device="cuda")
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")

    def timed(fn):
        # each piece is captured into a CUDA graph so that the number is device time of its kernels, not the
        # Python launch path (the real pipeline replays these inside graphs as well)
        fn(); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        g.replay(); torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.add_(1); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.mean(ts))

    pieces = {}
    ms = timed(lambda: ops.gae_rtg_segscan(r, v, flag_d, off_d, vb, rb, 0.99, 0.95, True, adv, rtg))
    pieces["segscan"] = dict(ms=ms, bytes=17 * n + 9 * n_seg)
    ms = timed(lambda: ops.batch_moments(obs, D, triple))
    pieces["obs_moments"] = dict(ms=ms, bytes=4 * D * n)
    ops.stats_merge(rms.state, triple, D)
    ms = timed(lambda: ops.normalize_clip(obs, rms.state, D, 1e-8, -10.0, 10.0, out))
    pieces["obs_normalize_clip"] = dict(ms=ms, bytes=8 * D * n)

    vtriple = torch.empty(3, dtype=torch.float64, device="cuda")

    def value_norm():
        t = ops.batch_moments(rtg, 1, vtriple)
        ops.stats_merge(vrms.state, t, 1)
        ops.normalize_clip(rtg, vrms.state, 1, 1e-8, 1.0, -1.0, rtg_n)
    ms = timed(value_norm)
    pieces["value_normalize"] = dict(ms=ms, bytes=12 * n)
    tot_ms = sum(p["ms"] for p in pieces.values())
    tot_b = sum(p["bytes"] for p in pieces.values())
    for p in pieces.values():
        p["gbs"] = p["bytes"] / p["ms"] / 1e6
        p["frac_of_hbm_peak"] = p["gbs"] / pk["hbm_gbs"]
    res = dict(workload="M-C2: 2^22 timesteps, obs dim 376, fp32, segments<=64, Bernoulli(0.02) ends",
               n_timesteps=n, n_segments=int(n_seg), pieces=pieces, total_ms=tot_ms,
               total_gbs=tot_b / tot_ms / 1e6, total_frac_of_hbm_peak=tot_b / tot_ms / 1e6 / pk["hbm_gbs"],
               env_steps_per_s=n / (tot_ms / 1e3), l2="flushed between iterations (256 MB write)")
    del obs, out
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------------
def cpu_reference_sample(w, sample_minibatches=8, seed=1234):
    """
    The oracle port of the reference path on the host cores, on a bounded sample of the workload:
    `sample_minibatches` minibatches of B rows (one partial epoch: permutation, value normaliser,
    advantage normalisation, evaluate, losses, backward, clip, Adam — torch CPU fp32, all threads) plus
    GAE / reward-to-go for the same number of timesteps (pure-Python scans, one core, like the reference).
    Returns env-steps/s extrapolated to the full update: every env step is visited `epochs` times.
    """
    from oracle.segments import segment_returns
    from oracle.update import OracleUpdater
    rng = np.random.default_rng(seed)
    B, A = w["B"], w["agents"]
    n = sample_minibatches * B
    pred = w["n_disc"] if w["n_disc"] else w["Da"]

    def net(dims, gain_out):
        p = {}
        stems = ["sequential_net.0", "sequential_net.2.0", "sequential_net.2.2", "sequential_net.3"]
        for i, s in enumerate(stems):
            lin = torch.nn.Linear(dims[i], dims[i + 1])
            torch.nn.init.orthogonal_(lin.weight, gain_out if i == 3 else math.sqrt(2))
            p[s + ".weight"] = lin.weight.detach().numpy()
            p[s + ".bias"] = np.zeros(dims[i + 1], np.float32)
        return p

    actor = net([w["Do"]] + [w["actor_hidden"]] * 3 + [pred], 0.01)
    if not w["n_disc"]:
        actor["distribution.log_std"] = np.full(w["Da"], -0.5, np.float32)
    critic = net([w["Dc"]] + [w["critic_hidden"]] * 3 + [1], 1.0)
    upd = OracleUpdater(actor, critic, w["act"], bool(w["n_disc"]), lr=w["lr"])
    ds = dict(critic_observations=rng.standard_normal((n, w["Dc"])).astype(np.float32),
              observations=rng.standard_normal((n, w["Do"])).astype(np.float32),
              raw_actions=(rng.integers(0, w["n_disc"], (n, 1)) if w["n_disc"]
                           else rng.standard_normal((n, w["Da"])).astype(np.float32)),
              advantages=rng.standard_normal(n).astype(np.float32),
              log_probs=(-1 - rng.random(n)).astype(np.float32),
              rewards_to_go=rng.standard_normal(n).astype(np.float32), values=np.zeros(n, np.float32))
    rewards = rng.standard_normal(n).astype(np.float32)
    values = rng.standard_normal(n).astype(np.float32)
    t0 = time.perf_counter()
    L = w["max_ts_per_ep"]
    for s in range(0, n, L):
        segment_returns(rewards[s:s + L], values[s:s + L], 0.3, 0.3, 0.99, 0.95, True, (-100.0, 100.0))
    t_adv = time.perf_counter() - t0
    t0 = time.perf_counter()
    upd.batch_train([ds], [torch.randperm(n).numpy()], B)
    t_upd = time.perf_counter() - t0
    # env steps covered by the sample: n agent-samples / A agents; the full update visits each `epochs` times
    env_steps = n / A
    secs_per_env_step = (t_adv + w["epochs"] * t_upd) / env_steps
    return dict(value=1.0 / secs_per_env_step, unit="env-steps/s", cores=torch.get_num_threads(), kind="port",
                sample=f"{sample_minibatches} minibatches of {B} rows through the oracle update (torch-CPU fp32, "
                       f"{torch.get_num_threads()} threads) x {w['epochs']} epochs + GAE/RTG of {n} timesteps "
                       f"(python scans, 1 core); t_update={t_upd:.3f}s t_adv={t_adv:.3f}s"), t_adv + t_upd


def workload_label(w):
    """One string for both arms (`config.workload`)."""
    return (f"{w['name']} (obs {w['Do']}, critic obs {w['Dc']}, act {w['Da'] if not w['n_disc'] else w['n_disc']}, "
            f"{w['actor_hidden']}/{w['critic_hidden']}-wide MLPs, ts={w['ts']}, E={w['E']} per rank, "
            f"B={w['B']}, epochs={w['epochs']}, KL early stop off)")


def reference_available():
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    try:
        import ref_harness
        return ref_harness.available()
    except Exception:
        return False


def run_reference_arm(args, w):
    """`--impl reference`: the UNMODIFIED reference (oracle/_ref) on the host cores, args.gpus ranks over gloo (one process
    per rank, spawned here by rank 0), on our arm's workload.  Falls back to the oracle port only when the reference copy is
    missing."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    R = max(int(args.gpus), 1)
    steps = args.steps
    if reference_available():
        from oracle import ref_bench
        wu = 1 if args.warmup > 0 else 0
        res = ref_bench.run(w, n_ranks=R, steps=steps, warmup=wu, epochs_timed=1)
        v, secs = res["value"], res["per_step_s"]
        note = ("unmodified reference on the host cores: value = ranks x shard env-steps / slowest rank's step time; "
                f"{steps} timed step(s) after {wu} warm-up step(s)")
    else:
        for _ in range(args.warmup):
            cpu_reference_sample(w, sample_minibatches=2)
        vals, tot = [], 0.0
        for _ in range(steps):
            res, t = cpu_reference_sample(w, sample_minibatches=64)
            vals.append(res["value"]); tot += t
        v = float(np.mean(vals)) * R
        res["value"] = v
        secs = tot / steps
        note = "oracle port (the reference copy oracle/_ref is missing); single-rank figure scaled by the rank count"
    line = {"impl": "reference", "metric": "ppo_update_env_steps_per_s", "value": v, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label(w), "note": note},
            "cpu_baseline": res, "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                                         "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-microbench", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (status scalars, trained parameters, advantages, "
                         "rewards-to-go, values, value-normaliser state) as DIR/<name>.npy; inputs are seeded, so two "
                         "builds run with the same arguments can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the device path computed; the reference arm has none")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, w)
        return

    rank, world, local = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the product path has no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    pk = peaks()
    args.warmup = max(args.warmup, 3)

    ro, pol = build_workload(w, rank, f"cuda:{local}")
    hp = HotPath(w, ro, pol)
    ring_mb = hp.h2d_bytes() / 1e6
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")      # 256 MB > 126 MB L2

    sampler = ClockSampler(local)
    sampler.start()
    ms = time_steps(lambda: hp.step(False), args.steps, args.warmup, flush)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:                      # before the passes below train the policy further
        dump_outputs(hp.outputs(), args.dump_outputs)
    ms_e2e = time_steps(lambda: hp.step(True), args.steps, args.warmup, flush)
    h2d_ms = float(np.mean([a.elapsed_time(b) for a, b in hp.h2d_events[-args.steps:]]))   # the ring copy alone, per step

    env_steps = w["ts"] * w["E"] * world                    # multi-agent: env steps exclude the xA factor
    value = env_steps * args.steps / (ms / 1e3)
    e2e = env_steps * args.steps / (ms_e2e / 1e3)
    mb_steps = hp.n_mb * w["epochs"]
    us_per_mb = 1e3 * (ms / args.steps) / mb_steps
    flops_step = flops_per_sample_visit(w) * w["B"]
    upd_tflops = flops_step / (us_per_mb * 1e-6) / 1e12

    line = {"metric": "ppo_update_env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label(w),
                       "per_rank_samples": hp.n, "minibatch_steps_per_step": mb_steps, "us_per_minibatch_step": us_per_mb,
                       "parallelism": f"dp{world}", "l2": "256 MB flush write between timed iterations; ring "
                                                          f"{ring_mb:.0f} MB", "peaks": pk["source"]},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": hp.h2d_bytes(),
                    "d2h_bytes_per_step": hp.d2h_bytes(), "ms_per_step": ms_e2e / args.steps, "h2d_ms": h2d_ms,
                    "h2d_gbs": hp.h2d_bytes() / h2d_ms / 1e6,
                    "note": "same pass started from the pinned host ring; h2d_ms = CUDA-event time of the ring copy alone"},
            "gpu_launches": hp.launches_per_step() * args.steps,
            "host_record": {"us_per_env_step": 1e6 * hp.record_s / (w["ts"] * w["E"]), "total_s": hp.record_s,
                            "note": "third timer (not part of value / e2e): wall time of the caller side of the path, "
                                    "PPOPolicy.add_episode_info + end_episodes for every step of the rollout shard, with the "
                                    "per-step pinned-slab H2D; the reference's own figure is in cpu_baseline.sample "
                                    "(add_episode_info caller side)"},
            }
    # live per-kernel device time of one extra (untimed) step: kernels replayed from CUDA graphs have no event of their own,
    # so their durations come from CUPTI activity records (torch.profiler); fallback: the share of the committed launch list
    # (single-rank runs only: the extra step is a collective operation when R > 1 and every rank would have to take it)
    shares = kernel_shares(hp) if (rank == 0 and world == 1) else None
    gk = None
    if shares:
        gk = next((v for k, v in shares["kernels"].items() if "grouped_gemm_kernel" in k), None)
    gemm_share = (gk["us"] / shares["total_us"]) if gk else 0.80
    fp32 = measure_fp32_peak() if rank == 0 else None
    line["roofline"] = {
        "bound": "tensor", "kernel": "grouped_gemm_kernel (6 of the 8 launches of a minibatch step)",
        "achieved": upd_tflops / gemm_share, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
        "frac": upd_tflops / gemm_share / pk["bf16_tflops_sustained"], "traffic": None,
        "algorithmic_flops_per_step": flops_step, "step_us": us_per_mb, "whole_step_tflops": upd_tflops,
        "fp32_peak_tflops_measured": fp32, "frac_of_fp32_peak": (upd_tflops / gemm_share / fp32) if fp32 else None,
        "kernel_share_of_step": gemm_share, "kernel_avg_launch_us": (gk["us"] / gk["count"]) if gk else None,
        "kernel_launches_per_step": (gk["count"]) if gk else None,
        "share_source": "CUPTI activity records of one extra untimed step (torch.profiler)" if gk else "profiles/r02_launches_c4_summary.txt",
        "step_kernels": shares["kernels"] if shares else None,
        "note": f"dominant kernel of the timed region: {flops_step / 1e9:.2f} GFLOP per minibatch step (6*P_mm*B, SURVEY.md §8d) over "
                f"{gemm_share:.2f} x the CUDA-event step time of {us_per_mb:.1f} us (the kernel's share comes from the committed "
                "launch list; it runs inside a CUDA graph, so it has no event of its own).  The kernel is fp32 FFMA: the tensor peak "
                f"({pk['source']} bf16 sustained) is the contract's denominator, fp32_peak_tflops_measured (cuBLAS SGEMM 4096^3, TF32 "
                "off, measured in this run) the pipe it actually uses.  At B=512 the step is a chain of 8 dependent launches of "
                "~40-270 MFLOP each: latency-bound, see DESIGN.md §3.3-3.4"}
    if rank == 0 and world == 1 and os.environ.get("PPOAF_STEP", "chain") == "chain":
        # the opt-in one-launch engine (csrc/fused_step.cu: TMA boxes + tcgen05 3xTF32 tiles with A in TMEM) on the same
        # workload, same box, same timing rules: reported beside the default launch chain, not instead of it
        os.environ["PPOAF_STEP"] = "fused"
        pol._engine = None                                  # the engine is rebuilt (and re-reads PPOAF_STEP) on the next epoch
        ms_f, used, fused_err = None, False, None
        try:
            ms_f = time_steps(lambda: hp.step(False), args.steps, args.warmup, flush)
            used = bool(getattr(pol._engine, "fused", False))
        except Exception as exc:                            # the secondary engine must never take the headline line down
            fused_err = f"{type(exc).__name__}: {exc}"[:300]
        finally:
            os.environ["PPOAF_STEP"] = "chain"
            pol._engine = None
        line["step_engines"] = {
            "chain (default): 8 PDL launches per minibatch step replayed from one CUDA graph per epoch, fp32 FFMA tiles":
                {"value": value, "us_per_minibatch_step": us_per_mb},
            "fused (PPOAF_STEP=fused): one persistent cooperative launch per epoch, TMA + tcgen05 kind::tf32 3xTF32, grid barriers":
                ({"value": env_steps * args.steps / (ms_f / 1e3), "us_per_minibatch_step": 1e3 * (ms_f / args.steps) / mb_steps}
                 if used and ms_f else {"unavailable": fused_err or "ppoaf_ppo_fused_supported() refused this configuration"}),
            "note": "same pass, same timing rules, measured back to back in this process; DESIGN.md 3.4"}
    if rank == 0 and world == 1 and not args.no_microbench:
        mb = microbench_c2(pk)
        dom = max(mb["pieces"].items(), key=lambda kv: kv[1]["ms"])
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r01_c2_traffic.json")      # dram bytes per launch from the ncu --set full capture
        if os.path.exists(tpath):
            k = json.load(open(tpath))["kernels"].get(dom[0])
            if k:
                traffic = k["dram_bytes_read"] + k["dram_bytes_write"]
        mb["roofline"] = {"bound": "hbm", "achieved": dom[1]["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                          "frac": dom[1]["gbs"] / pk["hbm_gbs"], "traffic": traffic, "algorithmic_bytes": dom[1]["bytes"],
                          "kernel": dom[0],
                          "note": f"dominant HBM kernel of the GAE+normalisation microbench; peak = {pk['source']} copy bandwidth"}
        line["microbench"] = mb
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        port, _ = cpu_reference_sample(w, sample_minibatches=64)
        if reference_available():
            from oracle import ref_bench
            line["cpu_baseline"] = ref_bench.run(w, n_ranks=1, steps=1, warmup=0, epochs_timed=1)
            line["cpu_baseline_port"] = port
        else:
            line["cpu_baseline"] = port
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
