"""
Cost of the hidden activations at C4-shaped networks (actor 376-256^3-17, critic 376-256^3-1, Box(17), B = 512):
device time per minibatch step for Tanh (the control), ELU, Sigmoid (derivative from the output), SiLU and GELU
(derivative stored by the forward: one extra store and load of B x 256 floats per hidden layer and network), on the
launch chain and, for the ids it takes, on the one-launch engine (PPOAF_STEP=fused).  Runs alternate activations
inside each pass, two passes; the card's name and power limit are read in the same run.

    python scratch/activation_cost.py [--epochs 10] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

OBS, HIDDEN, ACT, B, T, E = 376, 256, 17, 512, 64, 128
MODULES = {"tanh": nn.Tanh, "elu": nn.ELU, "sigmoid": nn.Sigmoid, "silu": nn.SiLU, "gelu": nn.GELU}
ENGINES = {"chain": list(MODULES), "fused": ["tanh", "elu", "sigmoid"]}


def step_time(act, engine, epochs, repeats):
    from helpers import run_device_rollout
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    from ppo_and_friends_b200.spaces import Box
    from ppo_and_friends_b200.synthetic import make_rollout
    os.environ["PPOAF_STEP"] = engine
    ro = make_rollout(seed=5, T=T, E=E, obs_dim=OBS, act_dim=ACT, max_ts_per_ep=32, obs_scale=False)
    torch.manual_seed(0)
    pol = PPOPolicy("pol", Box(-1.0, 1.0, (ACT,)), Box(-np.inf, np.inf, (OBS,)), Box(-np.inf, np.inf, (OBS,)),
                    envs_per_proc=E,
                    actor_kw_args=dict(activation=MODULES[act](), hidden_size=HIDDEN, hidden_depth=3),
                    critic_kw_args=dict(activation=MODULES[act](), hidden_size=HIDDEN, hidden_depth=3))
    pol.register_agent("agent0")
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device("cuda"))
    ds = run_device_rollout(pol, ro)
    state = PPOUpdateState({"pol": pol}, batch_size=B, epochs_per_iter=1)
    loader = _Loader(ds, B)
    for _ in range(3):                                                     # warm-up: graph capture, module loads
        ppo_batch_train(state, loader, "pol")
    assert pol._engine.fused == (engine == "fused"), (act, engine)
    steps = len(ds) // B
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(epochs):
            ppo_batch_train(state, loader, "pol")
        t1.record()
        torch.cuda.synchronize()
        times.append(t0.elapsed_time(t1) * 1e3 / (epochs * steps))
    return dict(act=act, engine=engine, steps_per_epoch=steps, us_per_step=[round(t, 2) for t in times])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(gpu=smi[0] if smi else "unknown")), flush=True)
    for _ in range(2):                                                     # two alternating passes: run-to-run spread
        for engine, acts in ENGINES.items():
            for act in acts:
                print(json.dumps(step_time(act, engine, args.epochs, args.repeats)), flush=True)


if __name__ == "__main__":
    main()
