"""
CPU tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/ppoaf_b200.h
declares, the host-side logic (permutation protocol, parameter layout, ring layout, communicator
layer on gloo with world_size 2) behaves, and the product path refuses to run without CUDA.
No compute entry point is called here.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200.build import build
    build()
    header = open(os.path.join(ROOT, "include", "ppoaf_b200.h")).read()
    declared = set(re.findall(r"\b(ppoaf_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(_lib.EXPORTED_SYMBOLS) == declared
    assert lib.ppoaf_abi_version() == 1


def test_sizing_queries_without_gpu():
    import ctypes as C
    from ppo_and_friends_b200 import _lib
    lib = _lib.load()
    desc = _lib.MlpDesc.make([376, 256, 256, 256, 17], "tanh")
    offs, total = _lib.param_layout(desc, 17)
    # W0 b0 W1 b1 W2 b2 W3 b3 log_std, every tensor on a 4-float boundary
    assert offs[0] == 0 and offs[1] == 376 * 256 and all(o % 4 == 0 for o in offs)
    assert total == offs[-1] + 20
    assert lib.ppoaf_segscan_workspace_bytes(1 << 22) == (1 << 22) // 1024 * 64 + 64
    cfg = _lib.UpdateCfg()
    cfg.actor, cfg.critic = desc, _lib.MlpDesc.make([376, 256, 256, 256, 1], "tanh")
    cfg.head, cfg.act_dim = _lib.HEAD_GAUSSIAN_TANH, 17
    assert lib.ppoaf_update_workspace_bytes(C.byref(cfg), 512) > 512 * 256 * 4 * 12


def test_no_cpu_fallback():
    from ppo_and_friends_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.PpoafError):
        _lib.require_cuda()
    from helpers import make_policy
    from ppo_and_friends_b200.synthetic import make_rollout
    with pytest.raises(_lib.PpoafError):
        make_policy(make_rollout(0, 4, 2), device="cpu")


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "ppo_and_friends_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"
                assert "/root/reference" not in src, f


def test_permutation_protocol_matches_dataloader():
    """Row U1: same global-RNG draws and the same indices as DataLoader(shuffle=True)."""
    from torch.utils.data import DataLoader
    from ppo_and_friends_b200.ppo import draw_minibatch_permutation

    class DS(torch.utils.data.Dataset):
        def __len__(self):
            return 193

        def __getitem__(self, i):
            return i

    for seed in (0, 1, 12345):
        torch.manual_seed(seed)
        loader = DataLoader(DS(), batch_size=64, shuffle=True)
        ref = [torch.cat([b for b in loader]) for _ in range(3)]          # three epochs
        state_after_ref = torch.random.get_rng_state()
        torch.manual_seed(seed)
        got = [draw_minibatch_permutation(193) for _ in range(3)]
        for a, b in zip(ref, got):
            assert torch.equal(a, b)
        assert torch.equal(torch.random.get_rng_state(), state_after_ref)


def test_hidden_sizes_and_key_stems():
    from ppo_and_friends_b200.networks.feed_forward import hidden_sizes, layer_key_stems
    assert hidden_sizes(64, 3) == [64, 64, 64] and hidden_sizes([32, 16], 9) == [32, 16] and hidden_sizes(0, 0) == []
    with pytest.raises(ValueError):
        hidden_sizes(0, 2)
    assert layer_key_stems(3) == ["sequential_net.0", "sequential_net.2.0", "sequential_net.2.2", "sequential_net.3"]
    assert layer_key_stems(1) == ["sequential_net.0", "sequential_net.3"] and layer_key_stems(0) == ["sequential_net.0"]


def test_reference_init_order_matches_torch_sequential():
    """Same torch seed -> same weights as building nn.Linear layers the way the reference does."""
    from ppo_and_friends_b200.networks.feed_forward import reference_init
    torch.manual_seed(3)
    mine = reference_init([6, 8, 8, 2], 0.01)
    torch.manual_seed(3)
    ref = []
    for i, (a, b) in enumerate(((6, 8), (8, 8), (8, 2))):
        lin = torch.nn.Linear(a, b)
        torch.nn.init.orthogonal_(lin.weight, 0.01 if i == 2 else np.sqrt(2))
        torch.nn.init.constant_(lin.bias, 0.0)
        ref.append(lin)
    for (w, b), lin in zip(mine, ref):
        assert torch.equal(w, lin.weight.detach()) and torch.equal(b, lin.bias.detach())


def test_replay_driver_event_order():
    """Terminated envs are closed before maxed ones at the same step; truncation beats termination."""
    from ppo_and_friends_b200.synthetic import make_rollout, replay_rollout

    class Rec:
        def __init__(self):
            self.calls = []

        def add_episode_info(self, **kw):
            self.calls.append(("add", kw["agent_id"]))

        def end_episodes(self, agent_id, env_idxs, episode_lengths, terminal, ending_values, ending_rewards):
            self.calls.append(("end", agent_id, tuple(int(e) for e in env_idxs), bool(terminal[0]), len(ending_values)))

    ro = make_rollout(1, T=4, E=3, agents=("a", "b"), max_ts_per_ep=2, p_term=0.0, p_trunc=0.0)
    ro.terminated[1, 0] = True
    ro.terminated[2, 1] = True
    ro.truncated[2, 1] = True                                            # both set: truncated wins
    rec = Rec()
    replay_rollout(lambda a: rec, ro)
    ends = [c for c in rec.calls if c[0] == "end"]
    assert ends[0] == ("end", "a", (0,), True, 1) and ends[1] == ("end", "b", (0,), True, 1)   # t=1 terminal
    assert ends[2] == ("end", "a", (1, 2), False, 3)                                            # t=1 maxed, full [E] arrays
    assert ends[4] == ("end", "a", (1,), False, 3)                                              # t=2: env1 truncated (not terminal)
    assert ends[-1] == ("end", "b", (0, 1, 2), False, 3)                                        # rollout end closes every env


GLOO_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["PPOAF_ROOT"])
from ppo_and_friends_b200.utils import mpi_utils
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["PPOAF_PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
r = mpi_utils.get_rank()
assert mpi_utils.get_num_procs() == 2
p = torch.full((10,), float(r + 1))
mpi_utils.broadcast_model_parameters(p)            # rank 0's parameters everywhere
assert torch.equal(p, torch.ones(10))
g = torch.arange(6, dtype=torch.float32) * (r + 1)
mpi_utils.mpi_avg_gradients(g)                     # SUM; 1/R is applied by the Adam kernel
assert torch.equal(g, torch.arange(6, dtype=torch.float32) * 3)
assert abs(mpi_utils.mpi_avg(float(r)) - 0.5) < 1e-12
assert np.allclose(mpi_utils.mpi_avg(np.array([r, 2.0 * r])), [0.5, 1.0])
tr = torch.tensor([[r, 1.0, 2.0]], dtype=torch.float64)
allg = mpi_utils.all_gather_cat(tr)
assert allg.shape == (2, 1, 3) and allg[1, 0, 0] == 1.0 and allg[0, 0, 0] == 0.0
s = torch.tensor([1.0, float(r)])
mpi_utils.allreduce_sum_(s)
assert torch.equal(s, torch.tensor([2.0, 1.0]))
mpi_utils.barrier()
print("rank", r, "ok")
"""


def test_comm_layer_gloo_world_size_2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    port = str(29000 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), PPOAF_ROOT=ROOT, PPOAF_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
    assert "rank 0 ok" in outs[0] and "rank 1 ok" in outs[1]


def test_value_stat_merge_order_matches_allgather_semantics():
    """Multi-rank value normaliser: pooling per-rank (mean, M2, n) triples in rank order equals the
    reference's allgather + concatenate + np.mean/np.var (utils/stats.py:47-59)."""
    from oracle.stats import OracleRunningMeanStd
    rng = np.random.default_rng(2)
    a, b = rng.normal(0, 2, 64).astype(np.float32), rng.normal(1, 1, 64).astype(np.float32)
    ref = OracleRunningMeanStd()
    ref.update(a, [b])

    def triple(x):
        x = x.astype(np.float64)
        return x.mean(), ((x - x.mean()) ** 2).sum(), float(len(x))

    (m1, s1, n1), (m2, s2, n2) = triple(a), triple(b)
    n = n1 + n2
    d = m2 - m1
    mean, M2 = m1 + d * n2 / n, s1 + s2 + d * d * n1 * n2 / n
    mine = OracleRunningMeanStd()
    mine.integrate(mean, M2 / n, n)
    assert abs(mine.mean - ref.mean) < 1e-6 and abs(mine.variance - ref.variance) < 1e-5 * ref.variance


def test_speculated_permutation_keeps_the_generator_protocol():
    """The permutation of the next epoch is drawn ahead of time (while the GPU runs the current epoch); it may only be
    used if nothing touched torch's global generator in between, and the generator must end up exactly where the
    reference's DataLoader would have left it."""
    import types
    from ppo_and_friends_b200.ppo import UpdateEngine, draw_minibatch_permutation
    eng = types.SimpleNamespace(_spec_perm=None)
    n = 257
    # reference sequence: two epochs drawn back to back, then one more global draw
    torch.manual_seed(99)
    ref = [draw_minibatch_permutation(n), draw_minibatch_permutation(n)]
    ref_next = torch.empty((), dtype=torch.int64).random_().item()
    # speculated sequence
    torch.manual_seed(99)
    p0 = draw_minibatch_permutation(n)
    UpdateEngine._speculate_next_permutation(eng, n)
    p1 = UpdateEngine._take_speculated_permutation(eng, n)
    assert p1 is not None and torch.equal(p0, ref[0]) and torch.equal(p1, ref[1])
    assert torch.empty((), dtype=torch.int64).random_().item() == ref_next
    # the epoch loop stops early: the speculation must leave no trace in the generator
    torch.manual_seed(99)
    draw_minibatch_permutation(n)
    UpdateEngine._speculate_next_permutation(eng, n)
    other = torch.empty((), dtype=torch.int64).random_().item()          # e.g. rollout sampling
    torch.manual_seed(99)
    draw_minibatch_permutation(n)
    assert other == torch.empty((), dtype=torch.int64).random_().item()
    # ... and a speculation made before that foreign draw must be discarded
    assert UpdateEngine._take_speculated_permutation(eng, n) is None
    # a different dataset size also discards it
    UpdateEngine._speculate_next_permutation(eng, n)
    assert UpdateEngine._take_speculated_permutation(eng, n + 1) is None


def test_epoch_pipelining_order_and_when_it_is_allowed(monkeypatch):
    """train_policies keeps ONE epoch in flight only when no host decision separates two epochs (target_kl = inf / None):
    enqueue(0), enqueue(1), finish(0), enqueue(2), finish(1), ..., finish(last); the status dictionary comes from the last
    epoch.  With a finite target_kl (the reference's default is 100) every epoch is finished before the next one starts."""
    import types
    import ppo_and_friends_b200.ppo as P
    from ppo_and_friends_b200._lib import ST
    log = []

    class FakeEngine:
        peer = None

        def __init__(self):
            self.k = 0

        def enqueue_epoch(self, ds, speculate=False):
            log.append(("enqueue", self.k, speculate))
            self.k += 1
            return self.k - 1

        def finish_epoch(self, token):
            log.append(("finish", token))
            st = np.zeros(ST["COUNT"])
            st[ST["COUNTER"]], st[ST["KL"]], st[ST["ACTOR_LOSS"]] = 2.0, 4.0 * (token + 1), 6.0
            return torch.as_tensor(st)

        def run_epoch(self, ds):
            return self.finish_epoch(self.enqueue_epoch(ds, speculate=True))

    eng = FakeEngine()
    monkeypatch.setattr(P, "_get_engine", lambda ppo, pid, bs: eng)
    recalcs = []
    ds = types.SimpleNamespace(recalculate_advantages=lambda: recalcs.append(len(log)))
    pol = types.SimpleNamespace(frozen=False, dataset=ds, target_kl=float("inf"), entropy_weight=lambda: 0.5,
                                device="cpu")
    ppo = types.SimpleNamespace(policies={"pol": pol}, batch_size=64, epochs_per_iter=4, recalc_advantages=True,
                                status_dict={"pol": {}}, verbose=False)
    assert P.train_policies(ppo) == {"pol": 4}
    assert log == [("enqueue", 0, False), ("enqueue", 1, False), ("finish", 0), ("enqueue", 2, False), ("finish", 1),
                   ("enqueue", 3, False), ("finish", 2), ("finish", 3)]
    assert recalcs == [1, 3, 5]                        # before every epoch but the first, right before its enqueue
    assert ppo.status_dict["pol"]["kl avg"] == 4.0 * 4 / 2.0 and ppo.status_dict["pol"]["actor loss"] == 3.0

    # finite target: epoch by epoch, with the early stop decided from each epoch's own statistics
    log.clear()
    eng.k = 0
    pol.target_kl = 100.0
    assert P.train_policies(ppo) == {"pol": 4}
    assert log == [x for k in range(4) for x in (("enqueue", k, True), ("finish", k))]
    log.clear()
    eng.k = 0
    pol.target_kl = 3.0                                # kl avg of epoch 0 is 2, of epoch 1 is 4
    assert P.train_policies(ppo) == {"pol": 2}
    # the switch
    log.clear()
    eng.k = 0
    pol.target_kl = None
    monkeypatch.setenv("PPOAF_PIPELINE_EPOCHS", "0")
    P.train_policies(ppo)
    assert log[:3] == [("enqueue", 0, True), ("finish", 0), ("enqueue", 1, True)]


def test_adam_view_state_dict_is_torch_adam_compatible():
    """The optimizer stand-in of the fused update reads and writes torch.optim.Adam state dicts (the format of the
    reference's `actor_optim_<rank>` checkpoint files, policies/ppo_policy.py:1228-1247).  Host-only: buffers on CPU."""
    from ppo_and_friends_b200.networks.feed_forward import PolicyNetworks, _AdamView
    torch.manual_seed(3)
    nets = PolicyNetworks("cpu", [5, 8, 8, 3], [5, 6, 1], torch.nn.Tanh(), torch.nn.Tanh(), gaussian=True, act_dim=3)
    nets.adam_m.copy_(torch.randn_like(nets.adam_m))
    nets.adam_v.copy_(torch.rand_like(nets.adam_v))
    nets.adam_step.fill_(7)
    views = {"actor": _AdamView(1e-3, nets.actor), "critic": _AdamView(1e-3, nets.critic)}
    saved = {}
    for name, view in views.items():
        net = getattr(nets, name)
        sd = view.state_dict()
        saved[name] = sd
        params = [torch.nn.Parameter(v.detach().clone()) for v in net.state_dict().values()]
        opt = torch.optim.Adam(params, lr=5e-4, eps=1e-5)
        opt.load_state_dict(sd)                                   # a real torch Adam accepts the file
        st = opt.state_dict()["state"]
        m, v = net.adam_dicts()
        assert len(st) == len(m)
        for i, k in enumerate(m):
            assert torch.equal(st[i]["exp_avg"], m[k]) and torch.equal(st[i]["exp_avg_sq"], v[k])
            assert float(st[i]["step"]) == 7.0
        assert opt.state_dict()["param_groups"][0]["lr"] == 1e-3
    # and back: wipe the buffers, load what torch wrote
    nets2 = PolicyNetworks("cpu", [5, 8, 8, 3], [5, 6, 1], torch.nn.Tanh(), torch.nn.Tanh(), gaussian=True, act_dim=3)
    for name in ("actor", "critic"):
        _AdamView(1e-3, getattr(nets2, name)).load_state_dict(saved[name])
    for name in ("actor", "critic"):                             # (the flat buffers also hold alignment padding)
        (m1, v1), (m2, v2) = getattr(nets, name).adam_dicts(), getattr(nets2, name).adam_dicts()
        for k in m1:
            assert torch.equal(m1[k], m2[k]) and torch.equal(v1[k], v2[k])
    assert int(nets2.adam_step.item()) == 7
    # different step counts for actor and critic cannot be represented by the single fused counter
    bad = {k: dict(v) for k, v in saved["critic"]["state"].items()}
    for v in bad.values():
        v["step"] = torch.tensor(9.0)
    nets3 = PolicyNetworks("cpu", [5, 8, 8, 3], [5, 6, 1], torch.nn.Tanh(), torch.nn.Tanh(), gaussian=True, act_dim=3)
    _AdamView(1e-3, nets3.actor).load_state_dict(saved["actor"])
    with pytest.raises(ValueError):
        _AdamView(1e-3, nets3.critic).load_state_dict(dict(state=bad, param_groups=saved["critic"]["param_groups"]))
    # a fresh optimizer (no step yet) has an empty state, like torch's
    nets4 = PolicyNetworks("cpu", [5, 8, 8, 3], [5, 6, 1], torch.nn.Tanh(), torch.nn.Tanh(), gaussian=True, act_dim=3)
    assert _AdamView(1e-3, nets4.actor).state_dict()["state"] == {}


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in _lib.py must have the layout the C compiler gives the structs of include/ppoaf_b200.h
    (sizes and the offsets of the fields added last)."""
    import ctypes as C
    import shutil
    import subprocess
    from ppo_and_friends_b200 import _lib
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ppoaf_b200.h"\n'
                   'int main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(ppoaf_mlp_desc), sizeof(ppoaf_update_cfg),\n'
                   '         sizeof(ppoaf_update_bufs), offsetof(ppoaf_update_bufs, n_flat), offsetof(ppoaf_update_bufs, batch),\n'
                   '         offsetof(ppoaf_update_bufs, n_mirror), offsetof(ppoaf_update_bufs, mirror_delta));\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    want = [C.sizeof(_lib.MlpDesc), C.sizeof(_lib.UpdateCfg), C.sizeof(_lib.UpdateBufs), _lib.UpdateBufs.n_flat.offset,
            _lib.UpdateBufs.batch.offset, _lib.UpdateBufs.n_mirror.offset, _lib.UpdateBufs.mirror_delta.offset]
    assert got == want, (got, want)


def test_bench_rejects_arguments_it_would_not_honour(tmp_path):
    """`--steps` is the number of timed steps (no fewer than one), and `--dump-outputs` has nothing to write for the
    reference arm: both are refused before any work starts."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "dump")]):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *args], capture_output=True, text=True)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-500:])
    assert not (tmp_path / "dump").exists()
