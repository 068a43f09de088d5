"""
torchrun worker of tests/test_peer_kernels.py: the fused all-reduce + clip + Adam kernels of csrc/peer.cu on R GPUs,
driven through PeerGroup / NvlsGroup (utils/peer.py) with gradients the worker writes itself, against the stand-alone
ppoaf_clip_adam_step and the float64 adam_step64 (bounds: the module docstring of test_peer_kernels.py).

Every rank draws all R gradients from one shared seed, so rank 0 can build the reference.  Each rank writes only its
own gradient, as production does: the push exchange stores it into slot [parity][rank] of every peer's receive buffer
through the mapped pointers of PeerGroup.ptrs (the same stores as the backward's mirror writes); the NVLS exchange
copies it into its symmetric gradient buffer of that parity.  An ordinary copy therefore always separates two kernel
calls (the kernels fetch params / m / v before their dependency wait), and every case gets a fresh group, so a fresh
`ctrl` per network size.

At R = 2 the worker also trains one epoch under NVLS and under the push exchange, saves both policies and checks the
optimizer files: identical on every rank, equal to the push run's to trajectory tolerance, loadable by torch.optim.Adam.

Prints one `PEER_KERNEL_CHECK PASS|FAIL world R` line on rank 0; `NVLS_SKIPPED <reason>` when the system offers no
multicast mapping.
"""
import ctypes as C
import math
import os
import sys
import zlib
from collections import namedtuple

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import HP_BASE, U, adam_step64  # noqa: E402

PEER_THREADS, PEER_SLOTS, PEER_MAX_RANKS = 1024, 2, 8     # peer.cu kPeerThreads, kPeerMaxVec, kPeerMaxRanks
RANKS = (2, 3, 4, 8)


def cdiv(a, b):
    return -(-a // b)


# ---- restated launch plans (they name cases and choose shapes; nothing is compared with them) ----------------------
def push_plan(nv, sm):
    """(grid, float4 slots per thread, accepted) of ppoaf_peer_allreduce_adam."""
    grid = max(1, min(sm, cdiv(nv, PEER_THREADS)))
    return grid, max(1, cdiv(nv, grid * PEER_THREADS)), nv <= grid * PEER_THREADS * PEER_SLOTS


def nvls_plan(nv, R, sm):
    """(slice, grid, slots, accepted, owned [lo, hi) per rank) of ppoaf_nvls_allreduce_adam, in float4 rows."""
    sl = cdiv(nv, R)
    grid = max(1, min(sm, cdiv(sl, PEER_THREADS)))
    owned = [(min(nv, r * sl), min(nv, (r + 1) * sl)) for r in range(R)]
    return sl, grid, max(1, cdiv(sl, grid * PEER_THREADS)), sl <= grid * PEER_THREADS * PEER_SLOTS, owned


# ---- case table ----------------------------------------------------------------------------------------------------
# kind: plain | probe (one step with beta1 = 0, INV_WORLD = 1, no clip: m holds the summed gradient exactly) |
# cache (resume at step 10^4 with carried moments and an empty cache, then a betas change and an lr change) |
# nan / inf / 1e20 (planted on one rank only at the last step)
Case = namedtuple("Case", "name exch nv na steps kind")


def worker_cases(R, S):
    c = []
    for exch in ("push", "nvls"):
        if exch == "push":
            shapes = [("1cta-1slot-nv1-na0", 1, 0), ("2cta-nv1025-nahalf", 1025, 512), ("1cta-nv1025-naall", 1025, 1025),
                      ("fullgrid-2slot-nv1024S+1-na1023", 1024 * S + 1, 1023),
                      ("fullgrid-2slot-nv1024S+1-na1025", 1024 * S + 1, 1025),
                      ("largest-nv2048S-na1024S-1", 2048 * S, 1024 * S - 1),
                      ("largest-nv2048S-na1024S+1", 2048 * S, 1024 * S + 1)]
            probe, big = 1024 * S + 1, 2048 * S
        else:
            k = 1000
            shapes = [("empty-slices-nv1-na1", 1, 1), ("nv-kR-nahalf", k * R, k * R // 2),
                      ("ragged-nv-kR+1-na-slice", k * R + 1, k + 1),
                      ("straddle-nv3000R+1-na-slice-1", 3000 * R + 1, 3000), ("straddle-nv3000R+1-na-slice+1", 3000 * R + 1, 3002),
                      ("fullgrid-2slot-nv1024SR+R-nahalf", 1024 * S * R + R, (1024 * S * R + R) // 2),
                      ("largest-nv2048SR-na-slice+1024", 2048 * S * R, 2048 * S + 1024)]
            if R > 2:
                shapes.insert(1, ("empty-slice-nvR-1-na0", R - 1, 0))
            probe, big = 4096 * R + 3, 2048 * S * R
        c.append(Case(f"{exch}-probe-nv{probe}", exch, probe, probe // 2, 1, "probe"))
        for name, nv, na in shapes:
            c.append(Case(f"{exch}-{name}", exch, nv, na, 2 if nv == big else 4, "plain"))
        c.append(Case(f"{exch}-cache-resume-betas-lr", exch, 2049, 1000, 5, "cache"))
        for kind in ("nan", "inf", "1e20"):
            c.append(Case(f"{exch}-{kind}-on-one-rank", exch, 3001, 1500, 3, kind))
    return c


def plant(kind, R, n, na):
    """(rank, element, value) of the bad gradient of a nan / inf / 1e20 case: one rank only."""
    if kind == "nan":
        return R - 1, na // 2, np.nan
    if kind == "inf":
        return min(1, R - 1), na + (n - na) // 3, np.inf
    return 0, 7, 1e20


def step_hp(case, k, R):
    hp = dict(HP_BASE, INV_WORLD=1.0 / R)
    if case.kind == "probe":
        hp.update(BETA1=0.0, INV_WORLD=1.0, GRAD_CLIP=-1.0)
    if case.kind == "cache":
        if k >= 2:
            hp.update(BETA1=0.5, BETA2=0.9)
        if k >= 3:
            hp.update(LR=1e-3)
    return hp


def draw_grads(rng, R, n, na, k, keep):
    """R float32 rows of n (rows r with keep(r) False are drawn and dropped): step k % 3 = 0 clips the actor (averaged
    norm ~4x the 0.5 limit), 1 the critic, 2 neither."""
    norms = ((2.0, 0.05), (0.05, 2.0), (0.05, 0.05))[k % 3]
    scale = np.empty(n, np.float32)
    for lo, hi, target in ((0, na, norms[0]), (na, n, norms[1])):
        if hi > lo:
            scale[lo:hi] = target * math.sqrt(R) / math.sqrt(hi - lo)
    rows = []
    for r in range(R):
        x = rng.standard_normal(n, dtype=np.float32)
        rows.append(x * scale if keep(r) else None)
    return rows


def gamma(d):
    return d * U / (1 - d * U)


def exact_coef(sumsq, hp):
    """True when both kernels' clip coefficient of a network is exactly determined (1, 0 or NaN), whatever order they
    sum its squares in: clipping off, at 0, a non-finite norm, or a ratio clearly above 1."""
    if hp["GRAD_CLIP"] <= 0 or not math.isfinite(sumsq):
        return True
    iw = float(np.float32(hp["INV_WORLD"]))
    return hp["GRAD_CLIP"] / (math.sqrt(sumsq) * iw + 1e-6) >= 1.0 + 1e-3


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def within(name, got, ref, bnd):
    """NaN pattern equal, the rest within the bound; returns the worst error / bound."""
    nan_ref = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan_ref), f"{name}: NaN pattern differs"
    ok = ~nan_ref
    err = np.abs(got[ok].astype(np.float64) - ref[ok])
    b = bnd[ok]
    assert (err <= b).all(), f"{name}: max err {err.max():.3e}, max err/bound {np.max(err / np.maximum(b, 1e-300)):.3f}"
    return float(np.max(np.divide(err, b, out=np.zeros_like(err), where=b > 0))) if err.size else 0.0


# ---- device side ---------------------------------------------------------------------------------------------------
def _cuda_memcpy():
    """cuMemcpyDtoDAsync: a plain stream-ordered copy to a peer-mapped address."""
    cu = C.CDLL("libcuda.so.1")
    fn = cu.cuMemcpyDtoDAsync_v2
    fn.restype = C.c_int
    fn.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p]
    return fn


def run_case(case, R, rank, S, dev, stats):
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace
    from ppo_and_friends_b200._lib import HP, load, stream_ptr
    from ppo_and_friends_b200.utils.peer import NvlsGroup, PeerGroup

    nv, n, na = case.nv, 4 * case.nv, 4 * case.na
    rng = np.random.default_rng([20261022, zlib.crc32(case.name.encode())])
    p0 = rng.standard_normal(n).astype(np.float32)
    t0 = 10 ** 4 if case.kind == "cache" else 0
    if case.kind == "cache":
        m0 = (rng.standard_normal(n) * 0.01).astype(np.float32)
        v0 = (np.square(rng.standard_normal(n)) * 1e-4).astype(np.float32)
    else:
        m0, v0 = np.zeros(n, np.float32), np.zeros(n, np.float32)
    nets = SimpleNamespace(flat_params=torch.from_numpy(p0).to(dev), adam_m=torch.from_numpy(m0).to(dev),
                           adam_v=torch.from_numpy(v0).to(dev), adam_step=torch.full((1,), t0, dtype=torch.int64, device=dev),
                           n_actor=na, n_critic=n - na)
    cursor = torch.zeros(1, dtype=torch.int32, device=dev)
    grp = PeerGroup(n, dev) if case.exch == "push" else NvlsGroup(n, dev)
    memcpy = _cuda_memcpy()
    ref = None
    if rank == 0 and case.exch == "push":                 # the stand-alone kernel on copies of the state
        ref = SimpleNamespace(p=torch.empty_like(nets.flat_params), m=torch.empty_like(nets.adam_m),
                              v=torch.empty_like(nets.adam_v), step=torch.empty_like(nets.adam_step),
                              ws=torch.zeros(1 << 16, dtype=torch.uint8, device=dev), lib=load())
    before = (p0, m0, v0)
    try:
        for k in range(case.steps):
            hp = step_hp(case, k, R)
            h = torch.zeros(HP["COUNT"], dtype=torch.float64)
            for key, val in hp.items():
                h[HP[key]] = val
            hd = h.to(dev)
            G = draw_grads(rng, R, n, na, k, keep=lambda r: rank == 0 or r == rank)
            if case.kind in ("nan", "inf", "1e20") and k == case.steps - 1:
                r_bad, j, val = plant(case.kind, R, n, na)
                if G[r_bad] is not None:
                    G[r_bad][j] = val
            parity = k & 1
            src = torch.from_numpy(G[rank]).to(dev)
            if case.exch == "push":             # slot [parity][rank] of every rank's receive buffer, own included
                for q in range(R):
                    dst = grp.ptrs[q][0] + (parity * R + rank) * grp.slot_bytes
                    assert memcpy(dst, src.data_ptr(), 4 * n, stream_ptr().value) == 0, "cuMemcpyDtoDAsync"
            else:
                grp.grads[parity].copy_(src)
            torch.cuda.synchronize(dev)
            dist.barrier()                      # the ranks enter the kernel together (its spin budget covers skew)
            grp.allreduce_adam(parity, nets, cursor, hd, stream_ptr())
            torch.cuda.synchronize(dev)
            if case.exch == "nvls":
                grp.gather_moments(nets)        # m, v are current only on each owner's slice
            # every rank must hold the same parameters, moments and counters, bit for bit (collectives first: every rank
            # runs all of them whatever it finds)
            same = True
            for t in (nets.flat_params, nets.adam_m, nets.adam_v, nets.adam_step, cursor):
                mine = t.view(torch.int32) if t.dtype == torch.float32 else t
                r0 = mine.clone()
                dist.broadcast(r0, 0)
                same &= bool(torch.equal(r0, mine))
            msg = ""
            try:
                assert same, "ranks disagree"
                assert grp.error_flag() == 0, f"error word {grp.error_flag()}"
                assert int(nets.adam_step.item()) == t0 + k + 1 and int(cursor.item()) == k + 1, "counters"
                got = tuple(x.cpu().numpy() for x in (nets.flat_params, nets.adam_m, nets.adam_v))
                if rank == 0:
                    check_step(case, k, R, G, hp, before, got, t0 + k + 1, stats, ref, hd)
                before = got
            except AssertionError as e:
                msg = f"{case.name} step {k}: {e}"
            flag = torch.tensor([0 if msg else 1], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if msg:
                raise AssertionError(msg)
            if not int(flag.item()):
                raise AssertionError(f"{case.name} step {k}: another rank failed")
    finally:
        grp.close()


def check_step(case, k, R, G, hp, before, got, t, stats, ref, hd):
    import torch
    from ppo_and_friends_b200._lib import check, ptr, stream_ptr
    p0, m0, v0 = before
    G = np.stack(G)
    n, na = G.shape[1], 4 * case.na
    s32 = G[0].copy()
    for r in range(1, R):                       # the push kernel's sum: float32, rank order
        s32 += G[r]
    with np.errstate(invalid="ignore", over="ignore"):
        s64 = G.astype(np.float64).sum(0)
        err64 = gamma(R - 1) * np.abs(G.astype(np.float64)).sum(0)
    err64 = np.where(np.isfinite(err64), err64, 0.0)
    if case.exch == "push":
        g, g_err = s32, None
    else:
        g, g_err = s64, err64
    rp, rm, rv, coefs, bnd = adam_step64(p0, g, m0, v0, t, hp, na, g_err=g_err)
    # NVLS: the moments were gathered from their owners after the step, so m and v are each owner's slice
    worst = max(within(name, x, r_, bnd[name]) for name, x, r_ in (("p", got[0], rp), ("m", got[1], rm), ("v", got[2], rv)))
    stats[case.exch] = max(stats.get(case.exch, 0.0), worst)
    if case.kind == "probe":                    # beta1 = 0, INV_WORLD = 1, no clip: m is the summed gradient itself
        m = got[1].astype(np.float64)
        if case.exch == "push":
            assert same_bits(got[1], s32), "push: m is not the float32 rank-order sum"
        else:
            b = gamma(R - 1) * np.abs(G.astype(np.float64)).sum(0)
            ratio = float(np.max(np.divide(np.abs(m - s64), b, out=np.zeros_like(b), where=b > 0)))
            assert ratio <= 1.0, f"in-switch sum error {ratio:.3f} of (R-1) u sum|g|"
            rn = s64.astype(np.float32)
            stats["nvls_sum"] = dict(err_over_bound=ratio, rank_order=float(np.mean(got[1] == s32)),
                                     correctly_rounded=float(np.mean(got[1] == rn)))
    if case.exch == "push":
        # the stand-alone kernel on the same state and the float32 sum: the same element arithmetic, bit for bit on
        # every network whose clip coefficient is exactly determined
        gd = torch.from_numpy(s32).to(ref.p.device)
        for a, b in ((ref.p, p0), (ref.m, m0), (ref.v, v0)):
            a.copy_(torch.from_numpy(b))
        ref.step.fill_(t - 1)
        check(ref.lib.ppoaf_clip_adam_step(ptr(ref.p), ptr(gd), ptr(ref.m), ptr(ref.v), ptr(ref.step), ptr(hd), na, n - na,
                                       ptr(ref.ws), ref.ws.numel(), stream_ptr()), "ppoaf_clip_adam_step")
        torch.cuda.synchronize()
        out = [x.cpu().numpy() for x in (ref.p, ref.m, ref.v)]
        with np.errstate(over="ignore"):
            sq = np.square(s32).astype(np.float64)
        for sl in (slice(0, na), slice(na, n)):
            if exact_coef(float(sq[sl].sum()), hp):
                for name, a, b in zip("pmv", got, out):
                    assert same_bits(a[sl], b[sl]), f"{name} differs from ppoaf_clip_adam_step"
    if case.kind == "nan" and k == case.steps - 1 and hp["GRAD_CLIP"] >= 0:
        assert np.isnan(got[0][:na]).all() and np.isfinite(got[0][na:]).all()


# ---- checkpoints under NVLS (R = 2) --------------------------------------------------------------------------------
def checkpoint_case(rank, world, local, tmp):
    import torch
    import torch.distributed as dist
    from helpers import make_policy, run_device_rollout
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    from ppo_and_friends_b200.synthetic import make_rollout

    files = {}
    for exch in ("nvls", "push"):
        os.environ["PPOAF_NVLS"] = "1" if exch == "nvls" else "0"
        ro = make_rollout(seed=500 + rank, T=24, E=8, obs_dim=12, act_dim=3, max_ts_per_ep=8, obs_scale=False)
        torch.manual_seed(1000 + rank)
        pol = make_policy(ro, act="tanh", actor_hidden=32, critic_hidden=48, lr=1e-3, device=f"cuda:{local}")
        ds = run_device_rollout(pol, ro)
        state = PPOUpdateState({"pol": pol}, batch_size=64, epochs_per_iter=1, device=f"cuda:{local}")
        torch.manual_seed(77 + rank)
        ppo_batch_train(state, _Loader(ds, 64), "pol")
        got = type(pol._engine.peer).__name__
        assert got == {"nvls": "NvlsGroup", "push": "PeerGroup"}[exch], f"{exch}: the engine chose {got}"
        path = os.path.join(tmp, exch)
        pol.save(path)
        dist.barrier()
        d = os.path.join(path, "pol-policy", "latest")
        files[exch] = {w: [os.path.join(d, f"{w}_optim_{r}") for r in range(world)] for w in ("actor", "critic")}
        pol._engine.peer.close()
    os.environ.pop("PPOAF_NVLS")
    if rank != 0:
        return
    for w in ("actor", "critic"):
        sds = [torch.load(f, weights_only=False) for f in files["nvls"][w]]
        push = torch.load(files["push"][w][0], weights_only=False)
        for r, sd in enumerate(sds[1:], 1):
            for i, st in sd["state"].items():
                for key in ("step", "exp_avg", "exp_avg_sq"):
                    assert torch.equal(st[key], sds[0]["state"][i][key]), f"nvls {w}_optim_{r} differs from rank 0: {i}/{key}"
        for i, st in sds[0]["state"].items():
            assert torch.equal(st["step"], push["state"][i]["step"])
            for key in ("exp_avg", "exp_avg_sq"):
                a, b = st[key].double().numpy(), push["state"][i][key].double().numpy()
                tol = 1e-4 * (np.abs(b) + 1e-3 * np.abs(b).max())
                assert (np.abs(a - b) <= tol).all(), f"nvls {w} {i}/{key} vs push: {np.max(np.abs(a - b) / tol):.2f} x tol"
        params = [torch.zeros(st["exp_avg"].shape, requires_grad=True) for _, st in sorted(sds[0]["state"].items())]
        opt = torch.optim.Adam(params, lr=1e-3, eps=1e-5)
        opt.load_state_dict(sds[0])
        for j, prm in enumerate(params):
            assert torch.equal(opt.state[prm]["exp_avg"], sds[0]["state"][j]["exp_avg"])
    print("NVLS checkpoint: optimizer files identical on every rank, match the push run, load into torch.optim.Adam")


def main():
    import tempfile
    import traceback
    import torch
    import torch.distributed as dist
    from ppo_and_friends_b200 import ops
    from ppo_and_friends_b200.utils.peer import NvlsGroup

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    S = ops.device_info()["sm_count"]
    # does the system offer a multicast mapping?  every rank must agree
    ok = torch.zeros(1, dtype=torch.int32, device=dev)
    reason = ""
    try:
        NvlsGroup(16, dev).close()
        ok += 1
    except Exception as e:                    # no multicast / no VMM support
        reason = f"{type(e).__name__}: {e}"
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    nvls = int(ok.item()) == 1
    if rank == 0 and not nvls:
        print("NVLS_SKIPPED", reason or "a peer has no multicast mapping", flush=True)
    stats, failures = {}, []
    for case in worker_cases(world, S):
        if case.exch == "nvls" and not nvls:
            continue
        try:
            run_case(case, world, rank, S, dev, stats)
            status = 1
        except AssertionError:
            failures.append(case.name)
            if rank == 0:
                traceback.print_exc()
            status = 0
        flag = torch.tensor([status], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if rank == 0:
            print(f"case {case.name}: {'ok' if int(flag.item()) else 'FAIL'}", flush=True)
        if not int(flag.item()) and case.name not in failures:
            failures.append(case.name)
    if world == 2 and nvls:
        tmp = [tempfile.mkdtemp(prefix="ppoaf_ckpt_") if rank == 0 else None]
        dist.broadcast_object_list(tmp, src=0)
        try:
            checkpoint_case(rank, world, local, tmp[0])
            status = 1
        except AssertionError:
            traceback.print_exc()
            status = 0
        flag = torch.tensor([status], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not int(flag.item()):
            failures.append("nvls-checkpoint")
        if rank == 0:
            print(f"case nvls-checkpoint: {'ok' if int(flag.item()) else 'FAIL'}", flush=True)
    if rank == 0:
        print("worst error / bound:", {k: v for k, v in stats.items()}, flush=True)
        print("PEER_KERNEL_CHECK", "FAIL " + ",".join(failures) if failures else "PASS", "world", world, flush=True)
    dist.destroy_process_group()
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
