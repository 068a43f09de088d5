"""
The fused gradient all-reduce + clip + Adam kernels of csrc/peer.cu: the push exchange (ppoaf_peer_allreduce_adam) on one
GPU at R = 1, and both exchanges (push and NVLS, ppoaf_nvls_allreduce_adam) on R = 2, 3, 4 and 8 GPUs through the torchrun
worker tests/peer_kernel_worker.py, against the stand-alone ppoaf_clip_adam_step and the float64 adam_step64 (helpers.py).

`push_plan` and `nvls_plan` (peer_kernel_worker.py) restate the host's launch plans: 1024-thread CTAs, grid
max(1, min(S, ceil(rows / 1024))) over nv = n_total / 4 float4 rows (push) or over one slice of ceil(nv / R) rows (NVLS),
each thread holding at most 2 rows in registers, so a call is accepted iff rows <= 2048 grid.  They name the cases and
choose shapes at plan edges; no result is compared with anything they compute.  After n calls the push kernel's grid
barrier word holds n * grid, which the R = 1 tests read back, so the plan a case names is the plan that ran.

Bounds, with u = 2^-24:
  push vs ppoaf_clip_adam_step  The element arithmetic is the same code (optim.cu adam_vec, the loop of peer.cu) and
                    the scalars are the same float64 -> float32 expressions; only the fp64 sum of the squares runs in
                    another order (CTA partials of 1024 threads against the 256-thread norm pass), so the clip
                    coefficients can differ by an ulp.  Wherever a network's coefficient is exactly determined -- clipping
                    off (1), max_norm 0 (0), a non-finite norm (0 or NaN), or max_norm / (norm + 1e-6) >= 1 + 1e-3, far
                    beyond the 7u the coefficient can move -- p, m and v must be equal bit for bit on that network.  The
                    beta-power caches of both see the same sequence of (t, betas), so both take pow() or the chained
                    product at the same steps.
  push vs float64   adam_step64 from the kernel's own state before the step, with its bound (derived in the docstring
                    of test_forward_optim_kernels.py: coefficient within 7u when clipping binds, then m, v and the
                    step with their counted roundings).  On R ranks the summed gradient is the float32 sum in rank
                    order, which numpy reproduces exactly (sequential float32 additions), with INV_WORLD = 1/R.
  NVLS vs float64   The switch adds the R replicas in an unspecified order: |g~ - sum g_r| <= gamma(R - 1) sum |g_r|
                    for any order of R - 1 float32 additions (gamma(d) = d u / (1 - d u)).  adam_step64 takes the exact
                    sum with that as g_err: the clip coefficient gains ||g_err|| / ||g|| + u relative (the norm of a
                    perturbed vector moves by at most the perturbation's norm; u for the float32 rounding of the exact
                    sum the reference squares), the scaled gradient gains INV_WORLD coef g_err.
  probe step        beta1 = 0, INV_WORLD = 1, no clip, zero moments: w1 = 1, so m = 0 + 1 (g - 0) is the summed gradient
                    exactly.  Push: the rank-order float32 sum, bit for bit.  NVLS: within gamma(R - 1) sum |g_r|; the
                    worker prints how often it equals the rank-order sum and the correctly rounded sum.
  across ranks      bit for bit: the push kernel sums in rank order on every rank; NVLS reduces each element once, on
                    its owner, and every rank gathers the owners' results.  adam_step and mb_cursor equal everywhere.
"""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import HP_BASE, U, adam_step64, f32
from peer_kernel_worker import (PEER_MAX_RANKS, PEER_SLOTS, PEER_THREADS, RANKS, exact_coef, nvls_plan, push_plan,
                                same_bits, worker_cases)

# ---- R = 1 cases: nv = a * S + b float4 rows (S = SM count), n_actor likewise ------------------------------------------
PUSH_NV = [(0, 1), (0, 1023), (0, 1024), (0, 1025), (1024, -1), (1024, 0), (1024, 1), (1536, 0), (2048, -1), (2048, 0)]
ALL = "all"
PUSH_SPLITS = [(0, 0), ALL, (0, 1023), (0, 1024), (0, 1025), (1024, -1), (1024, 0), (1024, 1)]   # on nv = 2048 S
LARGEST = (2048, 0)


def sym(ab):
    if ab == ALL:
        return "all"
    a, b = ab
    return f"{a}S{b:+d}" if a else str(b)


def resolve(ab, sm, nv=None):
    return nv if ab == ALL else ab[0] * sm + ab[1]


def push_cases():
    cases = [(nv, "half") for nv in PUSH_NV]
    cases += [(LARGEST, na) for na in PUSH_SPLITS]
    return cases


def split_where(na, nv, sm):
    """Where the actor / critic boundary falls in the push plan of nv rows."""
    grid, _, _ = push_plan(nv, sm)
    stride = grid * PEER_THREADS
    if na == 0:
        return "none"
    if na == nv:
        return "all"
    for edge, name in ((PEER_THREADS, "cta-edge"), (stride, "slot-stride")):
        if abs(na - edge) <= 1:
            return f"{name}{na - edge:+d}"
    return "inside"


def push_id(c, sm=148):
    nv_s, na_s = c
    nv = resolve(nv_s, sm)
    grid, slots, _ = push_plan(nv, sm)
    g = "fullgrid" if grid == sm else f"{grid}cta"
    na = nv // 2 if na_s == "half" else resolve(na_s, sm, nv)
    return f"{g}-{slots}slot-nv{sym(nv_s)}-na{'half' if na_s == 'half' else sym(na_s)}-{split_where(na, nv, sm)}"


def resolve_case(c, sm):
    nv = resolve(c[0], sm)
    na = nv // 2 if c[1] == "half" else resolve(c[1], sm, nv)
    return nv, na


# ---- CPU checks of the restatements and case tables ---------------------------------------------------------------
@pytest.mark.parametrize("sm", [132, 148, 160])
def test_case_tables_reach_every_launch_plan(sm):
    """(CPU) the R = 1 table reaches grids of 1, 2 and S CTAs, one and two register slots, the largest accepted network
    and the actor / critic boundary at 0, everything, a CTA edge +-1 and the slot stride +-1; case names do not depend
    on S.  The worker's table, for every R, reaches the same push plans, and for NVLS: empty slices (nv < R), nv = kR
    and kR + 1, a boundary on a slice edge +-1, a multi-CTA slice with two slots and the largest accepted slice."""
    plans = {push_plan(resolve_case(c, sm)[0], sm)[:2] for c in push_cases()}
    assert {(1, 1), (2, 1), (sm, 1), (sm, 2)} <= plans
    assert all(push_plan(resolve_case(c, sm)[0], sm)[2] for c in push_cases())
    assert not push_plan(2048 * sm + 1, sm)[2] and push_plan(2048 * sm, sm)[2]
    assert {push_id(c, sm) for c in push_cases()} == {push_id(c) for c in push_cases()}
    where = {split_where(*reversed(resolve_case(c, sm)), sm) for c in push_cases() if c[0] == LARGEST}
    assert where == {"none", "all", "cta-edge-1", "cta-edge+0", "cta-edge+1", "slot-stride-1", "slot-stride+0",
                     "slot-stride+1"}
    for R in RANKS:
        assert R <= PEER_MAX_RANKS
        cases = worker_cases(R, sm)
        assert len({c.name for c in cases}) == len(cases)
        push = [c for c in cases if c.exch == "push"]
        assert {push_plan(c.nv, sm)[:2] for c in push} >= {(1, 1), (2, 1), (sm, 2)}
        assert any(c.nv == 2048 * sm for c in push) and all(push_plan(c.nv, sm)[2] for c in push)
        assert {split_where(c.na, c.nv, sm)[:8] for c in push} >= {"none", "all", "cta-edge", "slot-str"}
        nv_cases = [c for c in cases if c.exch == "nvls"]
        plans = [nvls_plan(c.nv, R, sm) for c in nv_cases]
        assert all(p[3] for p in plans)
        assert any(c.nv < R for c in nv_cases)                                       # some ranks own nothing
        assert any(c.nv % R == 0 and c.nv >= R for c in nv_cases) and any(c.nv % R == 1 and c.nv > R for c in nv_cases)
        assert any(p[1] == sm and p[2] == 2 for p in plans)
        assert any(p[0] == 2048 * sm for p in plans)
        edges = {c.na - p[0] for c, p in zip(nv_cases, plans) if abs(c.na - p[0]) <= 1 and c.nv > p[0]}
        assert edges == {-1, 0, 1}
        assert {c.kind for c in nv_cases} == {c.kind for c in push} == {"plain", "probe", "cache", "nan", "inf", "1e20"}


def test_adam_reference_gradient_error_term():
    """(CPU) adam_step64's g_err: a zero one leaves the unclipped network's bounds as they were and adds only u to the
    clipped network's coefficient term (the float32 rounding of the exact sum); a positive one widens every bound and
    leaves the values alone."""
    rng = np.random.default_rng(3)
    n, na = 64, 24
    p, g = rng.standard_normal(n), rng.standard_normal(n) * np.r_[np.full(na, 1.0), np.full(n - na, 1e-3)]
    m, v = rng.standard_normal(n) * 0.01, rng.random(n) * 1e-4
    hp = dict(HP_BASE, INV_WORLD=1 / 3)
    base = adam_step64(p, g, m, v, 5, hp, na)
    zero = adam_step64(p, g, m, v, 5, hp, na, g_err=np.zeros(n))
    wide = adam_step64(p, g, m, v, 5, hp, na, g_err=1e-6 * np.abs(g))
    assert base[3][0] < 1.0 and base[3][1] == 1.0
    for k in "pmv":
        np.testing.assert_array_equal(base[4][k][na:], zero[4][k][na:])
        assert (zero[4][k][:na] > base[4][k][:na]).all() and (zero[4][k][:na] < base[4][k][:na] * 1.2).all()
        assert (wide[4][k] > zero[4][k]).all()
    for a, b in zip(base[:3], wide[:3]):
        np.testing.assert_array_equal(a, b)


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _sm_count():
    from ppo_and_friends_b200 import ops
    return ops.device_info()["sm_count"]


def _hp_dev(hp):
    from ppo_and_friends_b200._lib import HP
    h = torch.zeros(HP["COUNT"], dtype=torch.float64)
    for k, val in hp.items():
        h[HP[k]] = val
    return h.cuda()


def _ptrs(*tensors):
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


class PushRun:
    """One parameter set on the push kernel at R = 1 (peer_grads[0] and peer_flags[0] are local buffers, fresh ctrl),
    with ppoaf_clip_adam_step run on copies of its state before every step as the reference (its own workspace)."""

    def __init__(self, nv, na, rng, t0=0, moments=False, cursor=True):
        from ppo_and_friends_b200._lib import load
        self.lib = load()
        self.n, self.na = 4 * nv, 4 * na
        n = self.n
        self.p = torch.from_numpy(rng.standard_normal(n).astype(np.float32)).cuda()
        m = rng.standard_normal(n).astype(np.float32) * 0.01 if moments else np.zeros(n, np.float32)
        v = np.square(rng.standard_normal(n)).astype(np.float32) * 1e-4 if moments else np.zeros(n, np.float32)
        self.m, self.v = torch.from_numpy(m).cuda(), torch.from_numpy(v).cuda()
        self.step = torch.full((1,), t0, dtype=torch.int64, device="cuda")
        self.t0 = t0
        self.cursor = torch.zeros(1, dtype=torch.int32, device="cuda") if cursor else None
        self.g = torch.zeros(n, dtype=torch.float32, device="cuda")
        self.flags = torch.zeros(64, dtype=torch.int32, device="cuda")
        self.ctrl = torch.zeros(self.lib.ppoaf_peer_ctrl_bytes(), dtype=torch.uint8, device="cuda")
        self.ref = [torch.empty_like(x) for x in (self.p, self.m, self.v, self.step)]
        self.ws = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
        self.calls = 0

    def words(self):
        """The control words: [0] calls so far, [2] grid barrier count, [3] ticket, [4] error word."""
        return self.ctrl[-256:].view(torch.int32)[:8].cpu().numpy()

    def state(self):
        return self.p.cpu().numpy(), self.m.cpu().numpy(), self.v.cpu().numpy(), int(self.step.item())

    def launch(self, g, hp):
        from ppo_and_friends_b200._lib import check, ptr, stream_ptr
        hd = _hp_dev(hp)
        g_host = torch.from_numpy(np.ascontiguousarray(g, np.float32))
        for a, b in zip(self.ref, (self.p, self.m, self.v, self.step)):
            a.copy_(b)
        gd = g_host.cuda()
        check(self.lib.ppoaf_clip_adam_step(ptr(self.ref[0]), ptr(gd), ptr(self.ref[1]), ptr(self.ref[2]), ptr(self.ref[3]),
                                            ptr(hd), self.na, self.n - self.na, ptr(self.ws), self.ws.numel(),
                                            stream_ptr()), "ppoaf_clip_adam_step")
        self.g.copy_(g_host)           # an ordinary copy right before the peer kernel, as the gradient writes in a step
        check(self.lib.ppoaf_peer_allreduce_adam(_ptrs(self.g), _ptrs(self.flags), 1, 0, ptr(self.p), ptr(self.m),
                                                 ptr(self.v), ptr(self.step), ptr(self.cursor), ptr(hd), self.na,
                                                 self.n - self.na, ptr(self.ctrl), stream_ptr()),
              "ppoaf_peer_allreduce_adam")
        torch.cuda.synchronize()
        self.calls += 1

    def step_and_check(self, g, hp, nan_ok=False):
        """One step: bit for bit against ppoaf_clip_adam_step on every network whose coefficient is exactly determined,
        within adam_step64's bound everywhere; the counters advance.  Returns the coefficients and the worst ratio."""
        p0, m0, v0, t0 = self.state()
        self.launch(g, hp)
        got = self.state()
        assert got[3] == t0 + 1 and int(self.ref[3].item()) == t0 + 1
        if self.cursor is not None:
            assert int(self.cursor.item()) == self.calls
        w = self.words()
        grid = push_plan(self.n // 4, _sm_count())[0]
        assert (w[0], w[2], w[3], w[4]) == (self.calls, self.calls * grid, 0, 0), w
        ref = [x.cpu().numpy() for x in self.ref[:3]]
        with np.errstate(over="ignore"):
            sq = np.square(np.asarray(g, np.float32)).astype(np.float64)
        for sl in (slice(0, self.na), slice(self.na, self.n)):
            if exact_coef(float(sq[sl].sum()), hp):
                for name, a, b in zip("pmv", got[:3], ref):
                    assert same_bits(a[sl], b[sl]), f"{name}[{sl.start}:{sl.stop}] differs from ppoaf_clip_adam_step"
        rp, rm, rv, coefs, bnd = adam_step64(p0, g, m0, v0, t0 + 1, hp, self.na)
        worst = 0.0
        for name, x, r in (("p", got[0], rp), ("m", got[1], rm), ("v", got[2], rv)):
            nan_ref = np.isnan(r)
            assert np.array_equal(np.isnan(x), nan_ref), f"{name}: NaN pattern differs"
            ok = ~nan_ref
            if not nan_ok:
                assert ok.all()
            err = np.abs(x[ok].astype(np.float64) - r[ok])
            b = bnd[name][ok]
            assert (err <= b).all(), f"{name}: max err/bound {np.max(err / np.maximum(b, 1e-300)):.3f}"
            if err.size:
                worst = max(worst, float(np.max(np.divide(err, b, out=np.zeros_like(err), where=b > 0))))
        return coefs, worst


def _grads(rng, n, na, actor_norm, critic_norm):
    g = rng.standard_normal(n)
    g[:na] *= actor_norm / math.sqrt(max(na, 1))
    g[na:] *= critic_norm / math.sqrt(max(n - na, 1))
    return g.astype(np.float32)


# ---- GPU: R = 1 ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", push_cases(), ids=push_id)
def test_push_r1_plans(case):
    """Three steps from zero moments on every plan: the actor clipped and the critic not, then the other way round, then
    neither; the first step shows the coefficient directly (m = (1 - b1) coef g)."""
    sm = _sm_count()
    nv, na = resolve_case(case, sm)
    rng = np.random.default_rng(nv + 7 * na)
    run = PushRun(nv, na, rng)
    n, n_a = run.n, run.na
    g = _grads(rng, n, n_a, 2.0, 0.1)
    coefs, _ = run.step_and_check(g, HP_BASE)
    m1 = run.state()[1]
    nz = g != 0
    observed = m1[nz].astype(np.float64) / (f32(1 - HP_BASE["BETA1"]) * g[nz].astype(np.float64))
    expect = np.where(np.arange(n)[nz] < n_a, coefs[0], coefs[1])
    assert np.all(np.abs(observed - expect) <= 11 * U * expect)
    if n_a:
        assert coefs[0] < 0.5
    if n - n_a:
        assert coefs[1] == 1.0
    run.step_and_check(_grads(rng, n, n_a, 0.1, 2.0), HP_BASE)
    run.step_and_check(_grads(rng, n, n_a, 0.1, 0.1), HP_BASE)


@pytest.mark.gpu
@pytest.mark.parametrize("cursor", [True, False], ids=["cursor", "null-cursor"])
def test_push_r1_trajectory(cursor):
    """12 steps with fresh gradients (the clip binding on alternate networks), each checked from the kernel's own
    state; adam_step, mb_cursor, the call count and the grid barrier count advance, the error word stays 0.  A NULL
    mb_cursor is accepted."""
    sm = _sm_count()
    rng = np.random.default_rng(11)
    run = PushRun(1024 * sm + 1, 1024 + 1, rng, cursor=cursor)
    for t in range(12):
        norms = ((2.0, 0.1), (0.1, 2.0), (0.1, 0.1))[t % 3]
        run.step_and_check(_grads(rng, run.n, run.na, *norms), HP_BASE)
    assert run.state()[3] == 12


SCALAR_KINDS = ["betas-change", "resume-1e4-empty-cache", "lr-change", "clip-off", "clip-zero", "inv-world-1/3",
                "inv-world-1/7"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SCALAR_KINDS)
def test_push_r1_cache_and_scalars(kind):
    """The kernel's own beta-power cache and scalars: betas changing twice, a resume at step 10^4 with carried moments
    and an empty cache, the learning rate changing every step, clipping off and at 0, an inexact INV_WORLD."""
    sm = _sm_count()
    rng = np.random.default_rng(SCALAR_KINDS.index(kind))
    run = PushRun(1024 * sm + 1, (1024 * sm + 1) // 3, rng, t0=10 ** 4 if kind.startswith("resume") else 0,
                  moments=kind.startswith("resume"))
    hp = dict(HP_BASE)
    if kind == "clip-off":
        hp["GRAD_CLIP"] = -1.0
    if kind == "clip-zero":
        hp["GRAD_CLIP"] = 0.0
    if kind.startswith("inv-world"):
        hp["INV_WORLD"] = 1.0 / int(kind[-1])
    for t in range(7):
        if kind == "betas-change" and t in (3, 5):
            hp.update(BETA1=(0.5, 0.8)[t == 5], BETA2=(0.9, 0.99)[t == 5])
        if kind == "lr-change":
            hp["LR"] = (3e-4, 1e-3, 1e-4, 2.5e-4)[t % 4]
        scale = 1.0 / hp["INV_WORLD"]
        coefs, _ = run.step_and_check(_grads(rng, run.n, run.na, 3.0 * scale, 0.05 * scale), hp)
        if kind == "clip-off":
            assert coefs == [1.0, 1.0]
        elif kind == "clip-zero":
            assert coefs == [0.0, 0.0]
        else:
            assert coefs[0] < 0.25 and coefs[1] == 1.0
    if kind == "clip-zero":
        _, m, v, _ = run.state()
        assert not m.any() and not v.any()
    assert run.state()[3] == run.t0 + 7


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["actor", "critic"])
@pytest.mark.parametrize("value", [np.nan, np.inf, 1e20], ids=["nan", "inf", "1e20"])
def test_push_r1_nonfinite_gradient(value, net):
    """A NaN makes every parameter of its network NaN and leaves the other finite (torch clip_grad_norm_); +Inf gives a
    zero coefficient (its own element NaN, the rest of the network only decays its moments); a 1e20 square overflows
    float32 the same way.  Bit for bit against ppoaf_clip_adam_step in every case."""
    sm = _sm_count()
    rng = np.random.default_rng(21)
    nv = 1024 * sm + 1
    run = PushRun(nv, nv // 3, rng)
    run.step_and_check(_grads(rng, run.n, run.na, 2.0, 0.1), HP_BASE)
    g = _grads(rng, run.n, run.na, 2.0, 0.1)
    j = run.na // 2 if net == "actor" else run.na + (run.n - run.na) // 2
    g[j] = value
    coefs, _ = run.step_and_check(g, HP_BASE, nan_ok=True)
    p = run.state()[0]
    bad, good = (slice(0, run.na), slice(run.na, run.n)) if net == "actor" else (slice(run.na, run.n), slice(0, run.na))
    if math.isnan(value):
        assert math.isnan(coefs[net == "critic"])
        assert np.isnan(p[bad]).all()
    else:
        assert coefs[net == "critic"] == 0.0
        assert np.flatnonzero(np.isnan(p)).tolist() == ([j] if value == np.inf else [])
    assert np.isfinite(p[good]).all()


@pytest.mark.gpu
def test_refusals_launch_nothing():
    """Arguments the host code refuses before any launch: rank counts and ranks out of range, segments that are not
    float4 multiples, one float4 over the register-resident limit, and for NVLS a single rank or NULL pointers."""
    from ppo_and_friends_b200._lib import load, ptr, stream_ptr
    lib = load()
    sm = _sm_count()
    run = PushRun(1025, 512, np.random.default_rng(0))
    hd = _hp_dev(HP_BASE)
    before = run.state()
    over = 4 * (PEER_THREADS * PEER_SLOTS * sm + 1)          # one float4 past grid x 2048 at grid = S

    def push(n_ranks=1, my_rank=0, na=run.na, nc=run.n - run.na):
        grads = _ptrs(*([run.g] * max(n_ranks, 1)))
        flags = _ptrs(*([run.flags] * max(n_ranks, 1)))
        return lib.ppoaf_peer_allreduce_adam(grads, flags, n_ranks, my_rank, ptr(run.p), ptr(run.m), ptr(run.v),
                                             ptr(run.step), ptr(run.cursor), ptr(hd), na, nc, ptr(run.ctrl), stream_ptr())

    def nvls(n_ranks=2, my_rank=0, g_mc=True, staging=True, blocks=True, na=run.na, nc=run.n - run.na):
        arr = _ptrs(run.g, run.g)
        return lib.ppoaf_nvls_allreduce_adam(C.c_void_p(run.g.data_ptr()) if g_mc else None, arr if staging else None,
                                             arr if blocks else None, n_ranks, my_rank, ptr(run.p), ptr(run.m),
                                             ptr(run.v), ptr(run.step), ptr(run.cursor), ptr(hd), na, nc, ptr(run.ctrl),
                                             stream_ptr())

    refused = {
        "push n_ranks 0": push(n_ranks=0), "push n_ranks 9": push(n_ranks=PEER_MAX_RANKS + 1),
        "push my_rank -1": push(my_rank=-1), "push my_rank = n_ranks": push(my_rank=1),
        "push n_actor % 4": push(na=run.na + 2, nc=run.n - run.na - 2), "push n_critic % 4": push(nc=run.n - run.na - 1),
        "push over the register limit": push(na=0, nc=over),
        "nvls n_ranks 1": nvls(n_ranks=1), "nvls n_ranks 9": nvls(n_ranks=PEER_MAX_RANKS + 1),
        "nvls my_rank 2": nvls(my_rank=2), "nvls NULL g_mc": nvls(g_mc=False), "nvls NULL staging": nvls(staging=False),
        "nvls NULL flag_blocks": nvls(blocks=False), "nvls n_actor % 4": nvls(na=run.na + 1),
        "nvls over the register limit": nvls(na=0, nc=2 * over - 4),
    }
    torch.cuda.synchronize()
    assert [k for k, rc in refused.items() if rc == 0] == []
    after = run.state()
    for a, b in zip(before[:3], after[:3]):
        assert same_bits(a, b)
    assert after[3] == before[3] and int(run.cursor.item()) == 0 and not run.words().any()
    # the limit itself is accepted (one call, then the state moved)
    nv = PEER_THREADS * PEER_SLOTS * sm
    big = PushRun(nv, nv // 2, np.random.default_rng(1))
    big.step_and_check(_grads(np.random.default_rng(2), big.n, big.na, 2.0, 0.1), HP_BASE)
    assert nvls_plan(2 * nv, 2, sm)[3] and not nvls_plan(2 * nv + 1, 2, sm)[3]


# ---- GPU: R ranks under torchrun ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("R", RANKS)
def test_peer_kernels_on_r_gpus(R):
    """Both exchanges on R GPUs (tests/peer_kernel_worker.py): every launch plan of the worker's case table against
    ppoaf_clip_adam_step and adam_step64, bit-identical ranks, one bad rank, and at R = 2 the NVLS checkpoint."""
    if torch.cuda.device_count() < R:
        pytest.skip(f"needs {R} GPUs, this machine has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29600 + (os.getpid() + R) % 1000
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={R}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(root, "tests", "peer_kernel_worker.py")], capture_output=True, text=True,
                         timeout=900)
    out = res.stdout + res.stderr
    assert res.returncode == 0 and f"PEER_KERNEL_CHECK PASS world {R}" in res.stdout, out[-6000:]
    print("\n".join(line for line in res.stdout.splitlines() if line.startswith(("worst", "NVLS"))))
    skipped = [line for line in res.stdout.splitlines() if line.startswith("NVLS_SKIPPED")]
    if skipped:
        pytest.skip(f"push cases passed at R = {R}; NVLS cases skipped: {skipped[0][len('NVLS_SKIPPED '):]}")
