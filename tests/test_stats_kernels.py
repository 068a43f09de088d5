"""
The statistics kernels of csrc/stats.cu, each through the C ABI against a float64 restatement of the reference
semantics (oracle/stats.py, oracle/filters.py), at the launch plans the host code picks among.

`plan_fold`, `moments_grid` and `normalize_grid` below restate the host-side plan selection of stats.cu.  They are used
only to choose row counts at plan boundaries, to name the cases and to place sentinel rows; no result is compared with
anything they compute, so if they drift from the C code the placement weakens but no comparison becomes wrong.

Bounds, with u = 2^-24 (the unit roundoff of float32):
  batch moments    n exact; |mean - mean64| <= 1e-6 (sd64 + |mean64|); M2 within 1e-5 relative, exactly 0 for a
                   constant column (fp32 Welford per thread, fp64 merges).
  stats_merge      1e-12 relative against the oracle fed the same rows (fp64 throughout).
  normalize        (x - mu) * (1 / sd): three roundings, so |y - ref| <= 3u |ref| with ref evaluated in float64 from
                   the float32 mu and sd the kernel uses; denormalize is one fmaf, |y - ref| <= u |ref|.
  epoch_prepare    advantage mean within 1 ulp of float32(mean64), std within 2 ulp of float32(std64) + 1e-8f;
                   value triples (fp64 accumulation) within 1e-10 relative.
  value stats      final state 1e-12 relative, per-minibatch float32 (mean, sd) within 1 ulp.
  reward filters   running rewards bit-exact, statistics 1e-9 relative (1e-5 for an ill-conditioned batch whose
                   environments agree to 1e-5), reward scaling bit-exact against float32(float64(r) / sqrt(var + eps)).
"""
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle.filters import OracleFilterStack
from oracle.stats import OracleRunningMeanStd

U32 = 2.0 ** -24

# ---- restated launch plans (stats.cu: plan_fold, ppoaf_batch_moments, launch_normalize) ---------------------------
STAT_ROWS, STAT_UNROLL, MAX_FOLD_WIDTH = 8, 4, 128
Plan = namedtuple("Plan", "fold width rows tail bx")


def plan_fold(n, dim, misaligned=False):
    """The vectorised plan for n rows of `dim` floats, or None where the generic per-column path runs."""
    if misaligned:
        return None
    fold = 1
    if dim < MAX_FOLD_WIDTH:
        fold = MAX_FOLD_WIDTH // dim
        while fold > 1 and (dim * fold) % 4:
            fold -= 1
    if (dim * fold) % 4:
        return None
    bx = (dim * fold // 4 + 31) // 32 * 32
    if bx * STAT_ROWS > 1024 or n // fold == 0:
        return None
    return Plan(fold, dim * fold, n // fold, n % fold, bx)


def _grid(rows, rows_per_cta, cap):
    return max(1, min(-(-rows // rows_per_cta), cap))


def moments_grid(p, sm):
    return _grid(p.rows, STAT_ROWS * STAT_UNROLL * (2 if p.fold > 1 else 8), 4 * sm)


def normalize_grid(p, sm):
    return _grid(p.rows, STAT_ROWS * STAT_UNROLL * 4, 32 * sm)


def plan_id(n, dim, x_off=0, y_off=0):
    if x_off:
        return f"generic-unaligned{4 * x_off}B"
    p = plan_fold(n, dim)
    if p is None:
        fold = plan_fold(1 << 30, dim)
        return "generic-short" if fold is not None and n < fold.fold else "generic-width"
    name = f"fold{p.fold}-{'tail' if p.tail else 'notail'}" if p.fold > 1 else f"fold1-bx{p.bx}"
    return name + (f"-out-unaligned{4 * y_off}B" if y_off else "")


def capped_rows(dim, rows_per_cta, cap):
    """n whose super-rows overflow the grid cap so that the last CTA of the capped grid gets no rows:
    ceil(rows / grid) * (grid - 1) >= rows.  Folded plans also get a tail."""
    fold = plan_fold(1 << 30, dim).fold
    per = rows_per_cta + 1
    while True:
        rows = per * (cap - 1)
        if -(-rows // rows_per_cta) > cap and -(-rows // cap) == per:
            return rows * fold + (fold - 1)
        per += 1


def boundary_rows(n, dim, misaligned, grid_fn, sm):
    """Row 0, the last row, and where the plan splits the rows: the first and last row of CTA 1 and of the last CTA
    that has rows, the last folded row and the first tail row."""
    rows = {0, n - 1, n // 2}
    p = plan_fold(n, dim, misaligned)
    if p is not None:
        grid = grid_fn(p, sm)
        per = -(-p.rows // grid)
        for b in (1, -(-p.rows // per) - 1):
            lo, hi = b * per, min((b + 1) * per, p.rows)
            if 0 <= lo < hi:
                rows |= {lo * p.fold, hi * p.fold - 1}
        rows.add(p.rows * p.fold - 1)
        if p.tail:
            rows.add(p.rows * p.fold)
    return sorted(r for r in rows if 0 <= r < n)


def column_of(r, dim):
    return (r * 7 + 3) % dim


# ---- cases --------------------------------------------------------------------------------------------------------
CAPPED = -1          # n derived from the device's SM count so that the moments grid is capped with an empty last CTA
NORM_CAPPED = -2     # the same for the normaliser's grid


def _moment_cases():
    cases = []
    for dim in (1, 2, 3, 5, 7, 24, 31, 64, 100, 127):         # narrow rows folded into 128-float super-rows
        fold = plan_fold(1 << 30, dim)
        fold = fold.fold if fold is not None else 1
        cases.append((dim, fold * 1000, 0))
        if fold > 1:
            cases.append((dim, fold * 1000 + fold - 1, 0))
    cases += [(3, 10, 0), (5, 1, 0), (128, 1, 0)]               # n < fold, n = 1
    cases += [(dim, 3001, 0) for dim in (128, 132, 256, 376, 380, 384, 388, 448, 512)]
    cases += [(130, 3001, 0), (377, 2000, 0), (516, 2000, 0), (1030, 2000, 0), (7056, 600, 0)]
    cases += [(5, 3001, 1), (5, 3001, 2), (128, 3001, 1), (512, 3001, 2)]
    cases += [(128, CAPPED, 0), (5, CAPPED, 0), (1, 1 << 22, 0)]
    return cases


def _case_id(c):
    dim, n, x_off = c[:3]
    y_off = c[3] if len(c) > 3 else 0
    if n in (CAPPED, NORM_CAPPED):
        return f"grid-capped-empty-cta-{plan_id(1 << 30, dim)}-d{dim}"
    return f"{plan_id(n, dim, x_off, y_off)}-d{dim}-n{n}"


MOMENT_CASES = _moment_cases()
NORMALIZE_CASES = ([c + (0,) for c in MOMENT_CASES] + [(5, 3001, 0, 1), (128, 3001, 0, 1), (512, 3001, 0, 2)]
                   + [(128, NORM_CAPPED, 0, 0)])
ILL_CASES = [(5, 24 * 1000 + 23, 0), (128, 3001, 0), (448, 3001, 0), (130, 3001, 0), (128, 3001, 1)]
EPOCH_BATCH_SIZES = (1, 31, 32, 33, 63, 64, 65, 255, 256, 257, 512, 4096)


def epoch_threads(batch_size):
    return 256 if batch_size >= 256 else (64 if batch_size >= 64 else 32)


def test_case_tables_reach_every_launch_plan():
    """(CPU) the parametrisations cover every plan family, so a plan the host code can pick is not left untested."""
    ids = {_case_id(c).split("-d")[0] for c in MOMENT_CASES}
    for want in ("generic-short", "generic-width", "generic-unaligned4B", "generic-unaligned8B", "fold1-bx32",
                 "fold1-bx64", "fold1-bx96", "fold1-bx128", "fold2-notail", "fold16-tail", "fold128-notail"):
        assert any(i == want or i.endswith(want) for i in ids), want
    assert any(i.startswith("grid-capped-empty-cta-fold1") for i in ids)
    assert any(i.startswith("grid-capped-empty-cta-fold24") for i in ids)
    # the 384..512-wide rows that need more than the default 48 KB of shared memory in moments_partial_kernel
    assert {d for d, *_ in MOMENT_CASES
            if plan_fold(3001, d) and 8 * plan_fold(3001, d).width * 16 + 32 > 48 * 1024} == {384, 388, 448, 512}
    assert {epoch_threads(b) for b in EPOCH_BATCH_SIZES} == {32, 64, 256}


# ---- helpers ------------------------------------------------------------------------------------------------------
def _sm_count():
    from ppo_and_friends_b200 import ops
    return ops.device_info()["sm_count"]


def _resolve_n(n, dim, sm):
    """The row count of a case; for the capped cases, derived from the SM count and checked to leave the last CTA of the
    capped grid without rows."""
    if n not in (CAPPED, NORM_CAPPED):
        return n
    grid_fn, cap = (moments_grid, 4 * sm) if n == CAPPED else (normalize_grid, 32 * sm)
    rows_per_cta = STAT_ROWS * STAT_UNROLL * (4 if n == NORM_CAPPED else (2 if plan_fold(1 << 30, dim).fold > 1 else 8))
    n = capped_rows(dim, rows_per_cta, cap)
    p = plan_fold(n, dim)
    assert grid_fn(p, sm) == cap and -(-p.rows // cap) * (cap - 1) >= p.rows
    return n


def _placed(x, off, pad=4, fill=0.0):
    """A contiguous [n, dim] view of x whose base is `off` floats past a 16-byte aligned allocation."""
    buf = torch.full((x.numel() + off + pad,), fill, dtype=torch.float32, device="cuda")
    view = buf[off:off + x.numel()].view(x.shape)
    view.copy_(x)
    assert view.data_ptr() % 16 == 4 * off
    return buf, view


def _moments64(x):
    x64 = np.asarray(x, dtype=np.float64)
    mean = x64.mean(0)
    return mean, np.square(x64 - mean).sum(0)


def assert_moments(tri, x, mean_tol=1e-6, m2_tol=1e-5):
    n, dim = x.shape
    t = tri.cpu().numpy()
    assert t[2 * dim] == n
    mean, m2 = t[:dim], t[dim:2 * dim]
    mean64, m2_64 = _moments64(x)
    sd64 = np.sqrt(m2_64 / n)
    err = np.abs(mean - mean64)
    assert np.all(err <= mean_tol * (sd64 + np.abs(mean64))), float(np.max(err / (sd64 + np.abs(mean64) + 1e-300)))
    pos = m2_64 > 0
    assert np.all(m2[~pos] == 0)
    rel = np.abs(m2 - m2_64)[pos] / m2_64[pos]
    assert np.all(rel <= m2_tol), float(np.max(rel))


def oracle64(shape=()):
    """The oracle's RunningMeanStd with its initial state in float64.  It starts from float32 zeros and ones, and under
    NumPy's promotion rules `variance * count` on those stays float32, which alone moves the variance by ~1e-12."""
    ref = OracleRunningMeanStd(shape=shape)
    ref.mean, ref.variance = np.zeros(shape), np.ones(shape)
    return ref


def _rel_ok(got, ref, tol, scale=None):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    scale = np.abs(ref) if scale is None else scale
    return bool(np.all(np.abs(got - ref) <= tol * scale))


# ---- batch moments ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim,n,x_off", MOMENT_CASES, ids=[_case_id(c) for c in MOMENT_CASES])
def test_batch_moments_vs_float64(dim, n, x_off):
    from ppo_and_friends_b200 import ops
    sm = _sm_count()
    n = _resolve_n(n, dim, sm)
    rng = np.random.default_rng(dim * 7919 + n)
    mu = rng.uniform(-3, 3, dim)
    sd = rng.uniform(0.1, 10, dim)
    x = (rng.standard_normal((n, dim)) * sd + mu).astype(np.float32)
    rows = boundary_rows(n, dim, bool(x_off), moments_grid, sm)
    for i, r in enumerate(rows):                                # a dropped or duplicated boundary row moves M2 a lot
        c = column_of(r, dim)
        x[r, c] = mu[c] + (1e3 if i % 2 else -1e3) * sd[c]
    _, xd = _placed(torch.from_numpy(x).cuda(), x_off)

    tri = ops.batch_moments(xd, dim).clone()
    assert_moments(tri, x)
    assert torch.equal(ops.batch_moments(xd, dim), tri)                            # deterministic
    _, x2 = _placed(xd * 2, x_off)
    tri2 = ops.batch_moments(x2, dim).clone()                                      # exact in every plan
    assert torch.equal(tri2[:dim], 2 * tri[:dim]) and torch.equal(tri2[dim:2 * dim], 4 * tri[dim:2 * dim])

    # every element lands in its own column: a NaN poisons exactly its column, the others keep their bits
    for r in rows:
        c = column_of(r, dim)
        keep = xd[r, c].clone()
        xd[r, c] = float("nan")
        t = ops.batch_moments(xd, dim).clone()
        xd[r, c] = keep
        assert bool(torch.isnan(t[c])) and bool(torch.isnan(t[dim + c])), (r, c)
        others = torch.ones(2 * dim + 1, dtype=torch.bool, device="cuda")
        others[c] = others[dim + c] = False
        assert torch.equal(t[others], tri[others]), (r, c)

    xc = torch.full((n, dim), 0.1, dtype=torch.float32, device="cuda")            # constant columns: M2 exactly 0
    _, xc = _placed(xc, x_off)
    t = ops.batch_moments(xc, dim).cpu().numpy()
    assert np.all(t[:dim] == np.float64(np.float32(0.1))) and np.all(t[dim:2 * dim] == 0.0) and t[2 * dim] == n


@pytest.mark.gpu
@pytest.mark.parametrize("dim,n,x_off", ILL_CASES, ids=[_case_id(c) for c in ILL_CASES])
def test_batch_moments_ill_conditioned(dim, n, x_off):
    """mean / sd = 1e3.  Each fp32 Welford step rounds the running mean by up to u * |mean|, which is u * 1e3 (6e-5) of an
    sd, and every M2 term inherits it; with random signs the sum lands well inside half of that (the worst column of
    these cases measured 1.3e-5 on a B200).  The reference's own float32 np.var reaches 4e-5 on such data."""
    from ppo_and_friends_b200 import ops
    rng = np.random.default_rng(dim + n)
    sd = rng.uniform(0.1, 10, dim)
    x = (rng.standard_normal((n, dim)) * sd + 1e3 * sd).astype(np.float32)
    _, xd = _placed(torch.from_numpy(x).cuda(), x_off)
    assert_moments(ops.batch_moments(xd, dim), x, m2_tol=0.5 * U32 * 1e3)


# ---- stats_merge --------------------------------------------------------------------------------------------------
def _triple64(rows, dim):
    if len(rows) == 0:                            # an empty rank: whatever its mean / M2 slots hold must be ignored
        return np.concatenate([np.full(dim, -7.5), np.full(dim, 3.25), [0.0]])
    mean, m2 = _moments64(rows)
    return np.concatenate([mean, m2, [len(rows)]])


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 257, 1030], ids=lambda d: f"d{d}")
@pytest.mark.parametrize("n_ranks", [1, 3, 8], ids=lambda r: f"R{r}")
def test_stats_merge_pools_ranks_like_the_reference(dim, n_ranks):
    from ppo_and_friends_b200 import ops
    from ppo_and_friends_b200.utils.stats import RunningMeanStd
    rng = np.random.default_rng(dim * 10 + n_ranks)
    counts = rng.integers(1, 400, n_ranks)
    if n_ranks > 1:
        counts[n_ranks // 2] = 0
    base = rng.uniform(-3, 3, dim)
    datas = [(base + r + rng.standard_normal((int(k), dim)) * (1 + r)).astype(np.float32) for r, k in enumerate(counts)]
    loaded = (rng.uniform(-1, 1, dim), rng.uniform(0.5, 2, dim), 12345.0)
    for init in ("fresh", "loaded"):
        rms = RunningMeanStd(shape=(dim,))
        ref = oracle64((dim,))
        if init == "loaded":
            rms.load_reference(*loaded)
            ref.mean, ref.variance, ref.count = loaded[0].copy(), loaded[1].copy(), loaded[2]
        before = rms.state.clone()
        # float64 triples of the same rows: the merge itself is checked at fp64 precision
        tr = np.concatenate([_triple64(d.astype(np.float64), dim) for d in datas])
        ops.stats_merge(rms.state, torch.tensor(tr, device="cuda"), dim)
        ref.update(datas[0].astype(np.float64), other_ranks=[d.astype(np.float64) for d in datas[1:]])
        st = rms.state.cpu().numpy()
        scale = np.sqrt(ref.variance) + np.abs(ref.mean)
        assert _rel_ok(st[:dim], ref.mean, 1e-12, scale), init
        assert _rel_ok(st[dim:2 * dim], ref.variance, 1e-12), init
        assert st[2 * dim] == ref.count, init
        # the same pooling from batch_moments triples (fp32 Welford: the batch-moments bounds)
        rms.state.copy_(before)
        tri = torch.cat([ops.batch_moments(torch.from_numpy(d).cuda(), dim).clone() if len(d) else
                         torch.tensor(_triple64(d, dim), device="cuda") for d in datas])
        ops.stats_merge(rms.state, tri, dim)
        st = rms.state.cpu().numpy()
        assert _rel_ok(st[:dim], ref.mean, 1e-6, scale) and _rel_ok(st[dim:2 * dim], ref.variance, 1e-5), init
        assert st[2 * dim] == ref.count
    # a lone empty triple changes nothing, not even the count
    before = rms.state.clone()
    ops.stats_merge(rms.state, torch.tensor(_triple64(np.zeros((0, dim)), dim), device="cuda"), dim)
    assert torch.equal(rms.state, before)


# ---- normalize_clip / denormalize ---------------------------------------------------------------------------------
SENTINEL = -12345.5
CLIPS = {"clip": (-5.0, 5.0), "noclip": (1.0, -1.0), "lo-eq-hi": (2.0, 2.0)}


def _norm_state(dim, rng):
    """mean | var | count.  Every third column has a dyadic mean and a power-of-4 variance, so that sd is a power of two
    and mean + sd * 5 normalises to exactly 5."""
    mean = rng.uniform(-3, 3, dim)
    var = rng.uniform(0.01, 100, dim)
    c = np.arange(0, dim, 3)
    mean[c] = 0.75 * ((c // 3) % 5 - 2)
    var[c] = 4.0 ** ((c // 3) % 3 - 1)
    return mean, var


@pytest.mark.gpu
@pytest.mark.parametrize("dim,n,x_off,y_off", NORMALIZE_CASES, ids=[_case_id(c) for c in NORMALIZE_CASES])
def test_normalize_and_denormalize_vs_float64(dim, n, x_off, y_off):
    from ppo_and_friends_b200 import ops
    sm = _sm_count()
    n = _resolve_n(n, dim, sm)
    eps = 1e-8
    rng = np.random.default_rng(dim * 31 + n)
    mean, var = _norm_state(dim, rng)
    state = torch.tensor(np.concatenate([mean, var, [77.0]]), device="cuda")
    mu32 = mean.astype(np.float32)
    sd32 = np.sqrt(var.astype(np.float32) + np.float32(eps))                # float32, as the kernel computes it
    mu_d, sd_d = torch.tensor(mu32, device="cuda").double(), torch.tensor(sd32, device="cuda").double()
    g = torch.Generator(device="cuda")
    g.manual_seed(dim * 31 + n)
    x = torch.randn((n, dim), generator=g, device="cuda") * (3 * sd_d.float()) + mu_d.float()
    exact = {}
    for i, r in enumerate(boundary_rows(n, dim, bool(x_off or y_off), normalize_grid, sm)):
        c = column_of(r, dim) // 3 * 3
        v = 5.0 if i % 2 else -5.0
        x[r, c] = float(mu32[c]) + float(sd32[c]) * v                       # exact: dyadic mean, power-of-two sd
        exact[(r, c)] = v
    _, xd = _placed(x, x_off)
    total = n * dim
    ref = (xd.double() - mu_d) / sd_d

    def run(fn, src, *args):
        """fn(src) into an output view at y_off floats past an aligned buffer filled with a sentinel."""
        buf = torch.full((total + y_off + 64,), SENTINEL, dtype=torch.float32, device="cuda")
        y = buf[y_off:y_off + total].view(n, dim)
        fn(src, state, dim, eps, *args, out=y)
        assert bool((buf[:y_off] == SENTINEL).all()) and bool((buf[y_off + total:] == SENTINEL).all()), \
            "write outside the output"
        return y

    for mode, (lo, hi) in CLIPS.items():
        y = run(ops.normalize_clip, xd, lo, hi)
        want = ref.clamp(lo, hi) if lo < hi else ref          # clipping cannot widen the gap to the reference
        err = (y.double() - want).abs()
        assert bool((err <= 3.0001 * U32 * want.abs()).all()), (mode, float((err / want.abs()).max()))
        for (r, c), v in exact.items():
            assert float(y[r, c]) == (min(max(v, lo), hi) if lo < hi else v), (mode, r, c)

    # denormalize the unclipped output, read from the same alignment as x
    _, yd = _placed(run(ops.normalize_clip, xd, 1.0, -1.0), x_off)
    z = run(ops.denormalize, yd)
    want = yd.double() * sd_d + mu_d
    assert bool(((z.double() - want).abs() <= 1.0001 * U32 * want.abs()).all())
    # the round trip returns x: ((x - mu)(1 + 3u) / sd) * sd + mu, rounded once more
    x64 = xd.double()
    assert bool(((z.double() - x64).abs() <= 3.001 * U32 * (x64 - mu_d).abs() + 1.001 * U32 * x64.abs()).all())
    for (r, c) in exact:
        assert float(z[r, c]) == float(x[r, c])


# ---- epoch_prepare ------------------------------------------------------------------------------------------------
def _epoch_prepare(perm, adv, rtg, batch_size, n_mb, guard=3):
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200._lib import check, ptr, stream_ptr
    stats = torch.full((n_mb + guard, 2), SENTINEL, dtype=torch.float32, device="cuda")
    triples = torch.full((n_mb + guard, 3), SENTINEL, dtype=torch.float64, device="cuda")
    check(_lib.load().ppoaf_epoch_prepare(ptr(perm), ptr(adv), ptr(rtg), perm.numel(), batch_size, ptr(stats),
                                          ptr(triples), stream_ptr()), "ppoaf_epoch_prepare")
    assert bool((stats[n_mb:] == SENTINEL).all()) and bool((triples[n_mb:] == SENTINEL).all()), "past n_mb"
    return stats[:n_mb].cpu().numpy(), triples[:n_mb].cpu().numpy()


def _check_epoch_prepare(n, batch_size, rng):
    perm = rng.permutation(n).astype(np.int64)
    scale = 10.0 ** rng.uniform(-3, 3, n)
    adv = (rng.standard_normal(n) * scale + 0.1 * scale).astype(np.float32)
    rtg = (rng.standard_normal(n) * 10.0 ** rng.uniform(-2, 2, n) + 5.0).astype(np.float32)
    n_mb = -(-n // batch_size)
    stats, triples = _epoch_prepare(torch.tensor(perm, device="cuda"), torch.tensor(adv, device="cuda"),
                                    torch.tensor(rtg, device="cuda"), batch_size, n_mb)
    for k in range(n_mb):
        idx = perm[k * batch_size:(k + 1) * batch_size]
        a, v = adv[idx].astype(np.float64), rtg[idx].astype(np.float64)
        m32 = np.float32(a.mean())
        assert abs(stats[k, 0] - m32) <= np.spacing(abs(m32)), (k, stats[k, 0], m32)
        if len(idx) == 1:                                      # torch.std of one row is NaN
            assert np.isnan(stats[k, 1]), k
        else:
            s32 = np.float32(np.float32(a.std(ddof=1)) + np.float32(1e-8))
            assert abs(stats[k, 1] - s32) <= 2 * np.spacing(s32), (k, stats[k, 1], s32)
        vm, vm2 = v.mean(), np.square(v - v.mean()).sum()
        assert triples[k, 2] == len(idx), k
        assert abs(triples[k, 0] - vm) <= 1e-10 * (math.sqrt(vm2 / len(idx)) + abs(vm)), k
        assert abs(triples[k, 1] - vm2) <= 1e-10 * vm2, k


@pytest.mark.gpu
@pytest.mark.parametrize("batch_size", EPOCH_BATCH_SIZES, ids=[f"B{b}-t{epoch_threads(b)}" for b in EPOCH_BATCH_SIZES])
def test_epoch_prepare_vs_float64(batch_size):
    rng = np.random.default_rng(batch_size)
    for rem in sorted({0, 1 % batch_size, batch_size - 1}):
        _check_epoch_prepare(7 * batch_size + rem, batch_size, rng)


@pytest.mark.gpu
def test_epoch_prepare_large():
    _check_epoch_prepare(1 << 20, 512, np.random.default_rng(20))


# ---- value_stats_sequence -----------------------------------------------------------------------------------------
def _value_stats_sequence(state, triples, n_ranks, n_mb, eps, guard=2):
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200._lib import check, ptr, stream_ptr
    out = torch.full((n_mb + guard, 2), SENTINEL, dtype=torch.float32, device="cuda")
    check(_lib.load().ppoaf_value_stats_sequence(ptr(state), ptr(triples), n_ranks, n_mb, eps, ptr(out), stream_ptr()),
          "ppoaf_value_stats_sequence")
    assert bool((out[n_mb:] == SENTINEL).all()), "past n_mb"
    return out[:n_mb].cpu().numpy()


def _assert_sequence_state(state, ref, tol):
    st = state.cpu().numpy()
    sd = math.sqrt(float(ref.variance))
    assert abs(st[0] - float(ref.mean)) <= tol * (sd + abs(float(ref.mean))), (st[0], float(ref.mean))
    assert abs(st[1] - float(ref.variance)) <= tol * float(ref.variance), (st[1], float(ref.variance))
    assert st[2] == ref.count


def _assert_within_ulps(got, want, ulps):
    want = np.asarray(want, dtype=np.float32)
    assert np.all(np.abs(got.astype(np.float64) - want) <= ulps * np.spacing(np.abs(want)).astype(np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("n_mb", [1, 7, 2048], ids=lambda m: f"mb{m}")
@pytest.mark.parametrize("n_ranks", [1, 2, 3, 8], ids=lambda r: f"R{r}")
def test_value_stats_sequence_vs_sequential_updates(n_ranks, n_mb):
    """One RunningMeanStd.update per minibatch on the rank-order concatenation of its rows."""
    eps = 1e-8
    rng = np.random.default_rng(n_ranks * 10_000 + n_mb)
    rows = [[2.0 + 0.01 * k + rng.standard_normal(int(rng.integers(1, 40))) * (1 + r) for k in range(n_mb)]
            for r in range(n_ranks)]
    rows[n_ranks - 1][n_mb // 2] = np.zeros(0)
    triples = np.array([[[-7.5, 3.25, 0.0] if len(d) == 0 else [d.mean(), np.square(d - d.mean()).sum(), len(d)]
                         for d in rk] for rk in rows])
    for init in ((0.0, 1.0, 1e-4), (1.7, 0.3, 5000.0)):
        state = torch.tensor(init, dtype=torch.float64, device="cuda")
        got = _value_stats_sequence(state, torch.tensor(triples, device="cuda"), n_ranks, n_mb, eps)
        ref = OracleRunningMeanStd(shape=())
        ref.mean, ref.variance, ref.count = np.float64(init[0]), np.float64(init[1]), init[2]
        want = np.empty((n_mb, 2), dtype=np.float32)
        for k in range(n_mb):
            batch = np.concatenate([rows[r][k] for r in range(n_ranks)])
            if len(batch):                                  # an empty pool leaves the statistics alone
                ref.update(batch)
            want[k] = np.float32(ref.mean), np.sqrt(np.float32(ref.variance) + np.float32(eps))
        _assert_sequence_state(state, ref, 1e-12)
        _assert_within_ulps(got[:, 0], want[:, 0], 1)
        _assert_within_ulps(got[:, 1], want[:, 1], 1)


# ---- reward filters -----------------------------------------------------------------------------------------------
def _reward_scale_clip(r, state, eps, lo, hi, guard=64):
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200._lib import check, ptr, stream_ptr
    buf = torch.full((r.numel() + guard,), SENTINEL, dtype=torch.float32, device="cuda")
    check(_lib.load().ppoaf_reward_scale_clip(ptr(r), ptr(state), eps, lo, hi, ptr(buf), r.numel(), stream_ptr()),
          "ppoaf_reward_scale_clip")
    assert bool((buf[r.numel():] == SENTINEL).all()), "past n"
    return buf[:r.numel()].cpu().numpy()


def _scale_clip64(r, var, eps, lo, hi):
    y = (np.asarray(r, dtype=np.float64) / np.sqrt(var + np.float64(np.float32(eps)))).astype(np.float32)
    return np.clip(y, np.float32(lo), np.float32(hi)) if lo < hi else y


REWARD_CASES = [(e, g, False) for e in (1, 7, 64, 1000) for g in (0.0, 0.99)] + [(1000, 0.99, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_envs,gamma,ill", REWARD_CASES,
                         ids=[f"E{e}-g{g}" + ("-ill-conditioned" if ill else "") for e, g, ill in REWARD_CASES])
def test_reward_normalizer_steps_vs_oracle(n_envs, gamma, ill):
    """reward_norm_triples then value_stats_sequence with n_mb = E, step after step, as RewardNormalizer.step does."""
    from ppo_and_friends_b200 import _lib
    from ppo_and_friends_b200._lib import check, ptr, stream_ptr
    eps, lo, hi = 1e-8, -10.0, 10.0
    lib = _lib.load()
    rng = np.random.default_rng(n_envs + int(gamma * 100) + ill)
    oracle = OracleFilterStack(("a",), 1, 1, n_envs, gamma=gamma, eps=eps, reward_clip=(lo, hi))
    oracle.reward["a"] = oracle64()
    running = torch.zeros(n_envs, dtype=torch.float64, device="cuda")
    state = torch.tensor([0.0, 1.0, 1e-4], dtype=torch.float64, device="cuda")
    triples = torch.empty((n_envs, 3), dtype=torch.float64, device="cuda")
    tol = 1e-5 if ill else 1e-9
    for step in range(24):
        if ill:      # every environment within 1e-5 relative of the others: the O(1) M2 update is ill-conditioned
            r = (1.0 + 1e-6 * rng.standard_normal(n_envs)).astype(np.float32)
            done = np.zeros(n_envs, dtype=bool)
        else:
            r = (rng.standard_normal(n_envs) * 2.0 + 0.3).astype(np.float32)
            done = rng.random(n_envs) < 0.05
        rd = torch.tensor(r, device="cuda")
        check(lib.ppoaf_reward_norm_triples(ptr(rd), ptr(torch.tensor(done.astype(np.uint8), device="cuda")),
                                            ptr(running), n_envs, float(gamma), ptr(triples), stream_ptr()),
              "ppoaf_reward_norm_triples")
        _value_stats_sequence(state, triples, 1, n_envs, eps)
        out = _reward_scale_clip(rd, state, eps, lo, hi)
        want = oracle.filter_reward({"a": r.astype(np.float64)}, {"a": done}, {"a": np.zeros(n_envs, dtype=bool)})["a"]
        assert np.array_equal(running.cpu().numpy(), oracle.running_reward["a"]), step
        _assert_sequence_state(state, oracle.reward["a"], tol)
        assert np.array_equal(out, _scale_clip64(r, state[1].item(), eps, lo, hi)), step
        assert _rel_ok(out, want, tol + 2 * U32, np.maximum(np.abs(want), 1e-30)), step


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 100_000], ids=lambda n: f"n{n}")
def test_reward_scale_clip_is_the_float64_quotient_rounded_once(n):
    rng = np.random.default_rng(n)
    r = (rng.standard_normal(n) * 20).astype(np.float32)
    r[::17] = rng.uniform(-1e4, 1e4, r[::17].shape).astype(np.float32)
    var = 3.7
    state = torch.tensor([0.25, var, 99.0], dtype=torch.float64, device="cuda")
    for lo, hi in ((-10.0, 10.0), (1.0, -1.0), (3.0, 3.0)):
        got = _reward_scale_clip(torch.tensor(r, device="cuda"), state, 1e-8, lo, hi)
        assert np.array_equal(got, _scale_clip64(r, var, 1e-8, lo, hi)), (lo, hi)


# ---- the user-visible path ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_running_mean_std_over_three_agents_of_128_wide_observations():
    """A MAPPO critic normalising the concatenation of three agents' 128-wide observations: 384-float rows."""
    from ppo_and_friends_b200.utils.stats import RunningMeanStd
    rng = np.random.default_rng(384)
    mu, sd = rng.uniform(-3, 3, (3, 128)), rng.uniform(0.1, 10, (3, 128))
    rms, ref = RunningMeanStd(shape=(3, 128)), oracle64((3, 128))
    for n in (1000, 4096, 77):
        x = (rng.standard_normal((n, 3, 128)) * sd + mu).astype(np.float32)
        rms.update(x)
        ref.update(x.astype(np.float64))
        assert _rel_ok(rms.mean, ref.mean, 1e-6, np.sqrt(ref.variance) + np.abs(ref.mean))
        assert _rel_ok(rms.variance, ref.variance, 1e-5)
        assert rms.count == ref.count
