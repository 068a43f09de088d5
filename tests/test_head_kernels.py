"""
The stand-alone action heads of csrc/loss.cu -- ppoaf_head_evaluate, ppoaf_head_sample,
ppoaf_multi_categorical_evaluate and ppoaf_multi_categorical_sample -- through `ops` and the C ABI, against a float64
restatement of the oracle's formulas (oracle/update.py gaussian_std, gaussian_tanh_log_prob, categorical_from_probs;
torch's Bernoulli(probs = sigmoid(z)) as tests/test_multi_binary.py restates it), at every launch plan the entry points
choose among.

`head_is_wide`, `head_max_width` and `plan` restate the host-side choice (128 rows per block on the one-thread-per-row
kernels; a warp per row, kWideRowsPerCta = 8 rows per CTA, above 64 outputs).  They name the cases and place rows at
grid edges; no result is compared with anything they compute.  The float32 constants are kept as written: eps = 2^-23,
1e-6f, +-100, 0.91893853f, min_std = 0.01f.

Bounds, with u = 2^-24, gamma(n) = n u / (1 - n u), and the CUDA single-precision libm errors under the build's flags
(-O3, no fast-math): expf 2 ulp, logf 1 ulp, log1pf 1 ulp, tanhf 2 ulp, where k ulp <= 2 k u relative; `/` and the
arithmetic operators round correctly.  A monotone step f whose input carries an absolute error e is bounded by the
interval f(x + e) - f(x - e); this is how every clamp and every log enters, so a clamp that binds on both ends of
the interval contributes nothing and an ill-conditioned term carries its own condition number.
  summation depth   thread plan: sequential over the d terms of a row (gamma(d)); warp plan: ceil(d / 32) terms per
                    lane then a 5-level butterfly (gamma(ceil(d / 32) + 5)); multi-categorical log-prob: sequential over
                    the K sections (gamma(K)).  Each sum adds gamma(depth) times the sum of its terms' magnitudes.
  Gaussian          std = max(softplus(ls), min_std): expf 4u, log1pf 2u: 6u relative (0 above 20, where softplus is the
                    identity; the max is 1-Lipschitz, so the min_std tie is covered).  log std: 6u + 2u |log std|.
                    Q = z^2 / (2 std^2): z rounded (u, twice in z^2), z z, std std (2 * 6u + u), the division:
                    5u + 12u relative.  Normal term: Q err + log std err + u (Q + |log std|) + u |term|, then clamped.
                    1 - tanh^2: tanhf 4u |th|, so th^2 carries 8u th^2 + its rounding u th^2, the subtraction u (1 -
                    th^2): e_t = 9u th^2 + u (1 - th^2).  Near the 1e-6 clamp this is ~5e-7 against a value of 1e-6,
                    so log max(1 - th^2, 1e-6) is bounded by the interval log max(t + e_t, 1e-6) - log max(t - e_t,
                    1e-6): large only for the dimensions whose 1 - tanh^2 sits just above the clamp, 0 where both ends
                    clamp (|x| = 12), ~9u elsewhere.
  Gaussian sample   raw = fl(fl(noise std) + mean): |noise| std 6u + u |noise std| + u |raw|.  tanh(raw): the raw error
                    times 1 - th^2, + 4u |th|.  Range map ((th + 1) / 2) (hi - lo) + lo: th's error |hi - lo| / 2 +
                    3u |th + 1| |hi - lo| / 2 + u |a|.  The log-prob is checked at the kernel's own raw action.
  Categorical       e_j = expf(z_j - mx): u |z_j - mx| + 4u relative; se = sum e: gamma(depth) + max rel e; p = e / se:
                    + u; S = sum p: gamma(depth) + max rel p; pn = p / S: + u.  log clamp(pn): the interval over
                    pn (1 +- rel pn), + 2u |lg|.  Entropy: pn e_lg + |lg| pn rel_pn + u pn |lg| per column, summed.
  Bernoulli         p = 1 / (1 + expf(-z)): 6u relative.  l = log q - log1p(-q), q = clamp(p): the interval over
                    p (1 +- 6u) -- at q near 1 - eps this carries 1 / (1 - q) ~ 8e6, which is the float32 head's real
                    conditioning -- + 2u (|log q| + |log1p(-q)|) + u |l|.  logsigmoid(l) is 1-Lipschitz in l:
                    + 6u log1p(e^-|l|) + u |ls|.  Log-prob and entropy columns add one or two roundings each.
  sampled actions   Categorical: the kernel's v_j = (p_j / S) / q_j and torch's each carry gamma(n) + 2u relative; a
                    row is exempt from bit equality with torch.distributions when its two largest float64 v lie within
                    2 (gamma(n) + 2u) of each other.  Bernoulli: p carries 6u in the kernel, torch's sigmoid is allowed
                    4u; a row is exempt when some |u - p| <= 10u p.  Exempt rows are counted and printed.

Non-finite inputs follow the C header: torch.clamp keeps a NaN, so the positions of NaN and of non-finite values in
the kernel's outputs equal the float64 restatement's (numpy's maximum / clip keep NaN as torch.clamp does).
"""
import ctypes as C
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

from ppo_and_friends_b200 import _lib

GAUSS, CAT, BERN = _lib.HEAD_GAUSSIAN_TANH, _lib.HEAD_CATEGORICAL, _lib.HEAD_BERNOULLI
U = 2.0 ** -24
EPS = 2.0 ** -23
ONE_M_EPS = 1.0 - EPS
TINY = float(np.float32(1e-6))
LOG_SQRT_2PI = float(np.float32(0.91893853320467274178))
MIN_STD = float(np.float32(0.01))
ULP = dict(exp=2, log=1, log1p=1, tanh=2)             # CUDA single-precision libm, maximum error in ulp


def rel(fn):
    return 2 * ULP[fn] * U


# ---- restated launch plans ----------------------------------------------------------------------------------------
ROW_BLOCK, WIDE_ROWS_PER_CTA, MAX_NARROW = 128, 8, 64
MAX_WIDTH = {GAUSS: 4096, CAT: 65536, BERN: 64}


def cdiv(a, b):
    return -(-a // b)


def head_max_width(head):
    return MAX_WIDTH[head]


def head_is_wide(head, pred_dim, act_dim):
    return act_dim > MAX_NARROW if head == GAUSS else head == CAT and pred_dim > MAX_NARROW


def plan(head, pred_dim, act_dim, rows):
    """(plan name, blocks): 'thread' = one thread per row, 128 rows per block; 'warp' = one warp per row, 8 per CTA."""
    if head_is_wide(head, pred_dim, act_dim):
        return "warp", cdiv(rows, WIDE_ROWS_PER_CTA)
    return "thread", cdiv(rows, ROW_BLOCK)


def kernel(family, op, pred_dim, act_dim):
    """The kernel an entry point launches (family: gauss, cat, bern, mcat; op: evaluate, sample)."""
    if family == "mcat":
        return f"multi_categorical_{op}_kernel"
    if family == "bern":
        return f"bernoulli_{op}_kernel"
    head = GAUSS if family == "gauss" else CAT
    wide = head_is_wide(head, pred_dim, act_dim)
    if family == "gauss":
        return f"gaussian_{op}_wide_kernel" if wide else f"head_{op}_kernel"
    return f"categorical_{op}_wide_kernel" if wide else f"multi_categorical_{op}_kernel"


ALL_KERNELS = {f"head_{o}_kernel" for o in ("evaluate", "sample")} | \
              {f"{f}_{o}_wide_kernel" for f in ("gaussian", "categorical") for o in ("evaluate", "sample")} | \
              {f"{f}_{o}_kernel" for f in ("multi_categorical", "bernoulli") for o in ("evaluate", "sample")}

# ---- cases --------------------------------------------------------------------------------------------------------
Case = namedtuple("Case", "id family pred act rows")
GAUSS_THREAD_D, GAUSS_WARP_D = (1, 63, 64), (65, 96, 97, 4095, 4096)
THREAD_ROWS, WARP_ROWS = (1, 127, 128, 129, 1000), (1, 7, 8, 9, 1000)
CAT_THREAD_P, CAT_WARP_P = (1, 2, 63, 64), (65, 96, 97, 4672)
BERN_K = (1, 63, 64)


def _gauss_cases():
    out = []
    for d in GAUSS_THREAD_D + GAUSS_WARP_D:
        p = plan(GAUSS, d, d, 1)[0]
        for r in (THREAD_ROWS if p == "thread" else WARP_ROWS):
            out.append(Case(f"gauss-{p}-d{d}-rows{r}", "gauss", d, d, r))
    out.append(Case("gauss-thread-d63-ld70-rows129", "gauss", 70, 63, 129))      # row stride wider than act_dim
    out.append(Case("gauss-warp-d97-ld130-rows9", "gauss", 130, 97, 9))
    return out


def _cat_cases():
    out = []
    for P in CAT_THREAD_P + CAT_WARP_P:
        p = plan(CAT, P, 1, 1)[0]
        for r in (THREAD_ROWS if p == "thread" else WARP_ROWS):
            out.append(Case(f"cat-{p}-P{P}-rows{r}", "cat", P, 1, r))
    out.append(Case("cat-warp-P65536-rows64", "cat", 65536, 1, 64))
    out.append(Case("cat-thread-P63-ld3-rows129", "cat", 63, 3, 129))            # int64 actions at act_ld = 3
    out.append(Case("cat-warp-P97-ld3-rows9", "cat", 97, 3, 9))
    return out


def _bern_cases():
    return [Case(f"bern-thread-k{k}-rows{r}", "bern", k, k, r) for k in BERN_K for r in THREAD_ROWS]


def ends_of(sizes):
    e, o = 0, 0
    for n in sizes:
        o += n
        e |= 1 << (o - 1)
    return e


MCAT_TABLES = {
    "64x1": [1] * 64,                 # 64 sections of one output
    "1x64": [64],                     # one section of 64
    "straddle": [30, 4, 30],          # section 1 covers outputs 30..33, across 31 / 32
    "first1": [1, 20, 10],            # a first section of one output
    "last63": [7, 25, 32],            # sections end at 31 and at the last bit, 63
}


def _mcat_cases():
    return [Case(f"mcat-thread-{name}-rows{r}", "mcat", sum(s), len(s), r) for name, s in MCAT_TABLES.items()
            for r in (1, 128, 129)]


GAUSS_CASES, CAT_CASES, BERN_CASES, MCAT_CASES = _gauss_cases(), _cat_cases(), _bern_cases(), _mcat_cases()


def test_cases_reach_every_kernel_and_edge():
    reached = set()
    for c in GAUSS_CASES + CAT_CASES + BERN_CASES + MCAT_CASES:
        head = {"gauss": GAUSS, "cat": CAT, "bern": BERN, "mcat": None}[c.family]
        if head is not None:
            assert 1 <= c.pred <= head_max_width(head) and c.act <= head_max_width(head)
            assert c.id.startswith(f"{c.family}-{plan(head, c.pred, c.act, c.rows)[0]}-"), c.id
        for op in ("evaluate", "sample"):
            reached.add(kernel(c.family, op, c.pred, c.act))
    assert reached == ALL_KERNELS and len(ALL_KERNELS) == 10

    g = [(c.act, c.rows) for c in GAUSS_CASES if c.pred == c.act]
    assert {(d, r) for d in GAUSS_THREAD_D for r in (1, 127, 128, 129, 1000)} <= set(g)
    assert {(d, r) for d in GAUSS_WARP_D for r in (1, 7, 8, 9, 1000)} <= set(g)
    assert {plan(GAUSS, c.pred, c.act, 1)[0] for c in GAUSS_CASES if c.pred > c.act} == {"thread", "warp"}
    # warp plan: one partial lane stride, whole strides, one column past a stride, 16 KB of staged std
    assert {d % 32 for d in GAUSS_WARP_D} >= {0, 1} and 4 * max(GAUSS_WARP_D) == 16 * 1024
    blocks = {plan(GAUSS, 1, 1, r)[1] for r in THREAD_ROWS} | {plan(GAUSS, 65, 65, r)[1] for r in WARP_ROWS}
    assert {1, 2, 8, 125} <= blocks
    cats = {(c.pred, c.rows) for c in CAT_CASES}
    assert {P for P, _ in cats} == set(CAT_THREAD_P + CAT_WARP_P + (65536,)) and (65536, 64) in cats
    assert {plan(CAT, c.pred, 1, 1)[0] for c in CAT_CASES if c.act > 1} == {"thread", "warp"}
    assert {(c.pred, c.rows) for c in BERN_CASES} == {(k, r) for k in BERN_K for r in THREAD_ROWS}
    ends = {name: ends_of(s) for name, s in MCAT_TABLES.items()}
    assert ends["64x1"] == (1 << 64) - 1 and ends["1x64"] == 1 << 63 and ends["first1"] & 1
    assert ends["straddle"] & ((1 << 31) | (1 << 32)) == 0 and ends["last63"] >> 63 == 1 and ends["last63"] >> 31 & 1


# ---- float64 restatements and bounds -------------------------------------------------------------------------------
def gamma(n):
    return n * U / (1 - n * U)


def depth(p, n):
    return n if p == "thread" else cdiv(n, 32) + 5


def clamp(x, lo, hi):
    return np.minimum(np.maximum(x, lo), hi)                          # torch.clamp: NaN stays NaN


def interval(f, x, e):
    """|f(x') - f(x)| for |x' - x| <= e, f monotone non-decreasing."""
    return f(x + e) - f(x - e)


def gauss_std64(log_std, min_std=MIN_STD):
    ls = np.asarray(log_std, np.float64)
    with np.errstate(over="ignore"):
        sp = np.where(ls > 20, ls, np.log1p(np.exp(ls)))
    return clamp(sp, min_std, np.inf), np.where(ls > 20, 0.0, rel("exp") + rel("log1p"))


def _tanh_term(x):
    """log max(1 - tanh(x)^2, 1e-6) and its bound."""
    with np.errstate(over="ignore"):
        t = 1.0 / np.cosh(x) ** 2
    th2 = np.tanh(x) ** 2
    e_t = (2 * rel("tanh") + U) * th2 + U * t
    lg = lambda v: np.log(np.maximum(v, TINY))
    val = lg(t)
    return val, interval(lg, t, e_t) + rel("log") * np.abs(val)


def _normal_term(z, sd, rel_sd):
    lsd = np.log(sd)
    e_lsd = rel_sd + rel("log") * np.abs(lsd)
    with np.errstate(over="ignore", invalid="ignore"):
        Q = z * z / (2 * sd * sd)
        nl = -Q - lsd - LOG_SQRT_2PI
        e_nl = (5 * U + 2 * rel_sd) * Q + e_lsd + U * (Q + np.abs(lsd)) + U * np.abs(nl)
        nle = -lsd - LOG_SQRT_2PI
        e_nle = e_lsd + U * np.abs(nle)
    cl = lambda v: clamp(v, -100.0, 100.0)
    return cl(nl), interval(cl, nl, e_nl), cl(nle), interval(cl, nle, e_nle)


def gauss_ref(mean, log_std, x, p):
    """float64 (lp, ent, bound_lp, bound_ent) per row; mean [n, d] (the first act_dim columns), x [n, d]."""
    mu, x = np.asarray(mean, np.float64), np.asarray(x, np.float64)
    d = x.shape[1]
    sd, rel_sd = gauss_std64(log_std)
    with np.errstate(all="ignore"):
        cl, e_cl, cle, e_cle = _normal_term(x - mu, sd, rel_sd)
        cle, e_cle = np.broadcast_to(cle, x.shape), np.broadcast_to(e_cle, x.shape)
        tl, e_tl = _tanh_term(x)
        tm, e_tm = _tanh_term(mu)
        g = gamma(depth(p, d))
        lp = cl.sum(1) - tl.sum(1)
        ent = -(cle.sum(1) - tm.sum(1))
        b_lp = (e_cl + e_tl).sum(1) + g * (np.abs(cl).sum(1) + np.abs(tl).sum(1)) + U * np.abs(lp)
        b_ent = (e_cle + e_tm).sum(1) + g * (np.abs(cle).sum(1) + np.abs(tm).sum(1)) + U * np.abs(ent)
    return lp, ent, b_lp, b_ent


def softmax_parts(z, p):
    """e, se, p = e / se and the relative errors of the kernel's float32 e and p (Categorical bound)."""
    z = np.asarray(z, np.float64)
    with np.errstate(invalid="ignore"):
        mx = np.max(z, axis=1, keepdims=True)
        e = np.exp(z - mx)
        se = e.sum(1, keepdims=True)
        rel_e = U * np.abs(z - mx) + rel("exp")
        rel_se = gamma(depth(p, z.shape[1])) + np.max(rel_e, axis=1, keepdims=True)
    return e / se, rel_e + rel_se + U


def cat_columns(probs, rel_p, sections, p):
    """pn, lg, rel_pn, e_lg per column: one Categorical(probs) per section (a list of (start, size))."""
    pn = np.empty_like(probs)
    rel_pn = np.empty_like(probs)
    with np.errstate(invalid="ignore", divide="ignore"):
        for o, n in sections:
            blk = probs[:, o:o + n]
            S = blk.sum(1, keepdims=True)
            pn[:, o:o + n] = blk / S
            rel_S = gamma(depth(p, n)) + np.max(rel_p[:, o:o + n], axis=1, keepdims=True)
            rel_pn[:, o:o + n] = rel_p[:, o:o + n] + rel_S + U
        lgf = lambda v: np.log(clamp(v, EPS, ONE_M_EPS))
        lg = lgf(pn)
        e_lg = interval(lgf, pn, pn * rel_pn) + rel("log") * np.abs(lg)
    return pn, lg, rel_pn, e_lg


def sections_of(sizes):
    out, o = [], 0
    for n in sizes:
        out.append((o, n))
        o += n
    return out


def cat_eval_ref(logits, actions, sizes, p):
    """float64 (lp, ent, b_lp, b_ent): softmax over the row, one Categorical per section, actions [n, K] in-section."""
    probs, rel_p = softmax_parts(logits, p)
    secs = sections_of(sizes)
    pn, lg, rel_pn, e_lg = cat_columns(probs, rel_p, secs, p)
    rows = np.arange(probs.shape[0])
    lp_cols = np.stack([lg[rows, o + actions[:, k]] for k, (o, _) in enumerate(secs)], 1)
    e_cols = np.stack([e_lg[rows, o + actions[:, k]] for k, (o, _) in enumerate(secs)], 1)
    with np.errstate(invalid="ignore"):
        lp = lp_cols.sum(1)
        b_lp = e_cols.sum(1) + gamma(len(secs)) * np.abs(lp_cols).sum(1)
        t = pn * lg
        ent = -t.sum(1)
        b_ent = (pn * e_lg + np.abs(lg) * pn * rel_pn + U * np.abs(t)).sum(1) + \
            gamma(depth(p, probs.shape[1])) * np.abs(t).sum(1) + 1e-37
    return lp, ent, b_lp, b_ent


def bern_ref(logits, actions):
    """float64 (lp, ent, b_lp, b_ent) of fp32 0/1 actions under Bernoulli(sigmoid(z)), summed over the columns."""
    z, x = np.asarray(logits, np.float64), np.asarray(actions, np.float64)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        pr = 1.0 / (1.0 + np.exp(-z))
        rp = 6 * U
        lf = lambda q: (lambda c: np.log(c) - np.log1p(-c))(clamp(q, EPS, ONE_M_EPS))
        q = clamp(pr, EPS, ONE_M_EPS)
        l = lf(pr)
        e_l = interval(lf, pr, rp * pr) + rel("log") * np.abs(np.log(q)) + rel("log1p") * np.abs(np.log1p(-q)) + \
            U * np.abs(l)
        L = np.log1p(np.exp(-np.abs(l)))
        ls = np.minimum(l, 0) - L
        e_ls = e_l + 6 * U * L + U * np.abs(ls)
        lpc = ls - (1 - x) * l
        e_lpc = e_ls + (1 - x) * e_l + U * np.abs(lpc)
        hc = (1 - pr) * l - ls
        e_hc = np.abs(l) * (rp * pr + U * (1 - pr)) + (1 - pr) * e_l + U * np.abs((1 - pr) * l) + e_ls + U * np.abs(hc)
        g = gamma(z.shape[1])
        lp, ent = lpc.sum(1), hc.sum(1)
        b_lp = e_lpc.sum(1) + g * np.abs(lpc).sum(1) + U * np.abs(lp)
        b_ent = e_hc.sum(1) + g * np.abs(hc).sum(1) + U * np.abs(ent)
    return lp, ent, b_lp, b_ent, pr


SHARES = {}


@pytest.fixture(scope="module", autouse=True)
def report_shares():
    """Prints the worst error of each family as a share of its bound once the module's tests ran."""
    yield
    if SHARES:
        print("\nworst error / bound:", {k: round(v, 4) for k, v in sorted(SHARES.items())})


def check_within(name, got, ref, bound):
    """Finite rows: |got - ref| <= bound; records the worst share of the bound per family."""
    got = np.asarray(got, np.float64)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin), name
    err = np.abs(got[fin] - ref[fin])
    share = err / np.maximum(bound[fin], 1e-300)
    worst = float(share.max()) if share.size else 0.0
    fam = name.split("-")[0]
    SHARES[fam] = max(SHARES.get(fam, 0.0), worst)
    assert worst <= 1.0, (name, worst, int(np.argmax(share)))


def same_bits(a, b):
    return torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                       b.view(torch.int32) if b.dtype == torch.float32 else b)


# ---- inputs --------------------------------------------------------------------------------------------------------
def gauss_inputs(c, seed):
    g = np.random.default_rng(seed)
    n, d = c.rows, c.act
    mean = (g.standard_normal((n, c.pred)) * 2).astype(np.float32)
    ls = (g.uniform(-3, 1, d)).astype(np.float32)
    specials = [-10.0, 25.0, float(np.float32(math.log(math.expm1(MIN_STD))))]   # min_std binds, identity, the tie
    for k, v in enumerate(specials[:d]):
        ls[(k * 7) % d] = v
    x = (mean[:, :d] + g.standard_normal((n, d)) * 1.5).astype(np.float32)
    x[::5, (3 % d)] = 12.0                                            # tanh saturates
    x[1::5, (5 % d)] = -12.0
    x[2::7] = np.arctanh(1 - g.uniform(1e-7, 2e-6, (len(x[2::7]), d))).astype(np.float32)   # 1 - tanh^2 near 1e-6
    mean[3::11, :d] = np.where(g.random((len(mean[3::11]), d)) < 0.5, 12.0, -12.0)
    return mean, ls, x


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


# ---- GPU: Gaussian --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", GAUSS_CASES, ids=lambda c: c.id)
def test_gaussian_evaluate(c):
    from ppo_and_friends_b200 import ops
    mean, ls, x = gauss_inputs(c, c.act * 1009 + c.rows)
    p = plan(GAUSS, c.pred, c.act, c.rows)[0]
    lp, ent = ops.head_evaluate(GAUSS, dev(mean), dev(ls), dev(x))
    lp2, none = ops.head_evaluate(GAUSS, dev(mean), dev(ls), dev(x), want_entropy=False)   # ent_out NULL
    assert none is None and same_bits(lp, lp2)
    r_lp, r_ent, b_lp, b_ent = gauss_ref(mean[:, :c.act], ls, x, p)
    check_within(c.id, host(lp), r_lp, b_lp)
    check_within(c.id, host(ent), r_ent, b_ent)


def gauss_sample_ref(mean, ls, noise, lo, hi):
    """float64 raw = noise std + mean, action, and bounds (module docstring)."""
    sd, rel_sd = gauss_std64(ls)
    mu, z = np.asarray(mean, np.float64), np.asarray(noise, np.float64)
    with np.errstate(all="ignore"):
        raw = z * sd + mu
        e_raw = np.abs(z) * sd * rel_sd + U * np.abs(z * sd) + U * np.abs(raw)
        th = np.tanh(raw)
        e_th = e_raw / np.cosh(raw) ** 2 + rel("tanh") * np.abs(th)
        if lo is None:
            return raw, e_raw, th, e_th
        w = (hi - lo).astype(np.float64)
        a = (th + 1) / 2 * w + lo
        return raw, e_raw, a, e_th * np.abs(w) / 2 + 1.5 * U * np.abs(th + 1) * np.abs(w) + U * np.abs(a)


@pytest.mark.gpu
@pytest.mark.parametrize("c", GAUSS_CASES, ids=lambda c: c.id)
def test_gaussian_sample(c):
    from ppo_and_friends_b200 import ops
    mean, ls, _ = gauss_inputs(c, c.act * 1013 + c.rows)
    d, p = c.act, plan(GAUSS, c.pred, c.act, c.rows)[0]
    torch.manual_seed(c.rows)
    noise = torch.randn(c.rows, d)                                    # the policy's draw: torch.normal's N(0, 1)
    g = np.random.default_rng(d)
    lo = g.uniform(-3, 0, d).astype(np.float32)
    hi = (lo + g.uniform(0.5, 4, d)).astype(np.float32)
    for rng in (None, (lo, hi)):
        args = (dev(rng[0]), dev(rng[1])) if rng else (None, None)
        raw, act, lp = ops.head_sample(GAUSS, dev(mean), dev(ls), noise.cuda(), MIN_STD, *args, act_dim=d)
        raw2, act2, lp2 = ops.head_sample(GAUSS, dev(mean), dev(ls), noise.cuda(), MIN_STD, *args, act_dim=d)
        assert same_bits(raw, raw2) and same_bits(act, act2) and same_bits(lp, lp2)
        r_raw, e_raw, r_act, e_act = gauss_sample_ref(mean[:, :d], ls, noise.numpy(), *(rng or (None, None)))
        name = f"{c.id}-{'range' if rng else 'tanh'}"
        check_within("gauss_raw-" + name, host(raw).ravel(), r_raw.ravel(), e_raw.ravel())
        check_within("gauss_act-" + name, host(act).ravel(), r_act.ravel(), e_act.ravel())
        r_lp, _, b_lp, _ = gauss_ref(mean[:, :d], ls, host(raw), p)
        check_within("gauss-sample-" + name, host(lp), r_lp, b_lp)


# ---- GPU: Categorical and multi-categorical evaluation -------------------------------------------------------------
def cat_logits(n, P, seed):
    g = np.random.default_rng(seed)
    z = (g.standard_normal((n, P)) * 3).astype(np.float32)
    z[1::4] += np.float32(1e4)                                        # offset by 1e4
    dom = np.arange(2, n, 4)
    z[dom, g.integers(0, P, len(dom))] += np.float32(60.0)            # one dominant logit: the rest's pn < eps
    return z


@pytest.mark.gpu
@pytest.mark.parametrize("c", CAT_CASES, ids=lambda c: c.id)
def test_categorical_evaluate(c):
    from ppo_and_friends_b200 import ops
    z = cat_logits(c.rows, c.pred, c.pred * 31 + c.rows)
    g = np.random.default_rng(c.rows)
    acts = g.integers(0, c.pred, (c.rows, c.act)).astype(np.int64)
    acts[2::4, 0] = np.argmax(z[2::4], 1)                             # the dominant class: pn > 1 - eps
    lp, ent = ops.head_evaluate(CAT, dev(z), None, dev(acts))
    lp2, ent2 = ops.head_evaluate(CAT, dev(z), None, dev(acts))
    assert same_bits(lp, lp2) and same_bits(ent, ent2)
    p = plan(CAT, c.pred, c.act, c.rows)[0]
    r_lp, r_ent, b_lp, b_ent = cat_eval_ref(z, acts[:, :1], [c.pred], p)
    check_within(c.id, host(lp), r_lp, b_lp)
    check_within(c.id, host(ent), r_ent, b_ent)


@pytest.mark.gpu
@pytest.mark.parametrize("c", MCAT_CASES, ids=lambda c: c.id)
def test_multi_categorical_evaluate(c):
    from ppo_and_friends_b200 import ops
    sizes = MCAT_TABLES[c.id.split("-")[2]]
    z = cat_logits(c.rows, c.pred, c.rows + len(sizes))
    g = np.random.default_rng(c.rows)
    acts = np.stack([g.integers(0, n, c.rows) for n in sizes], 1).astype(np.int64)
    lp, ent = ops.multi_categorical_evaluate(dev(z), ends_of(sizes), dev(acts))
    r_lp, r_ent, b_lp, b_ent = cat_eval_ref(z, acts, sizes, "thread")
    check_within(c.id, host(lp), r_lp, b_lp)
    check_within(c.id, host(ent), r_ent, b_ent)


@pytest.mark.gpu
def test_multi_categorical_underflowed_section_is_nan():
    """A section whose probabilities all underflow to 0 (another section's logit 200 above) has no distribution:
    torch's Categorical normalises 0 / 0; the log-prob and the entropy are NaN, in evaluation and in sampling."""
    from ppo_and_friends_b200 import ops
    sizes = [3, 4]
    z = np.zeros((9, 7), np.float32)
    z[4, 1] = 200.0
    acts = np.zeros((9, 2), np.int64)
    from oracle.update import categorical_from_probs
    lp, ent = ops.multi_categorical_evaluate(dev(z), ends_of(sizes), dev(acts))
    probs = torch.softmax(torch.as_tensor(z), 1)
    assert float(probs[4, 3:].sum()) == 0.0
    want = torch.isnan(categorical_from_probs(probs[:, 3:])[1]).any(1).numpy()    # torch in float32
    assert want.tolist() == [i == 4 for i in range(9)]
    assert np.isnan(host(lp)).tolist() == want.tolist() and np.isnan(host(ent)).tolist() == want.tolist()
    act, lp = ops.multi_categorical_sample(probs.cuda(), ends_of(sizes), torch.ones(9 * 7).cuda(), 2)
    assert np.isnan(host(lp)).tolist() == [i == 4 for i in range(9)] and host(act)[4].tolist() == [1, 0]


# ---- GPU: Bernoulli ------------------------------------------------------------------------------------------------
BERN_SPECIAL = np.array([0, 1e-3, 15, 17, 20, 88, 100, 1e30, np.inf], np.float32)


def bern_logits(n, k, seed):
    g = np.random.default_rng(seed)
    z = (g.standard_normal((n, k)) * 4).astype(np.float32)
    sp = np.concatenate([BERN_SPECIAL, -BERN_SPECIAL])
    z[::3] = sp[g.integers(0, len(sp), (len(z[::3]), k))]
    return z


@pytest.mark.gpu
@pytest.mark.parametrize("c", BERN_CASES, ids=lambda c: c.id)
def test_bernoulli_evaluate(c):
    from ppo_and_friends_b200 import ops
    z = bern_logits(c.rows, c.act, c.act * 7 + c.rows)
    x = np.random.default_rng(c.rows).integers(0, 2, z.shape).astype(np.float32)
    lp, ent = ops.head_evaluate(BERN, dev(z), None, dev(x))
    lp2, ent2 = ops.head_evaluate(BERN, dev(z), None, dev(x))
    assert same_bits(lp, lp2) and same_bits(ent, ent2)
    r_lp, r_ent, b_lp, b_ent, _ = bern_ref(z, x)
    check_within(c.id, host(lp), r_lp, b_lp)
    check_within(c.id, host(ent), r_ent, b_ent)


@pytest.mark.gpu
@pytest.mark.parametrize("c", BERN_CASES, ids=lambda c: c.id)
def test_bernoulli_sample_matches_torch(c):
    from torch.distributions import Bernoulli
    from ppo_and_friends_b200 import ops
    z = bern_logits(c.rows, c.act, c.act * 5 + c.rows)
    torch.manual_seed(c.rows)
    want = Bernoulli(probs=torch.sigmoid(torch.as_tensor(z))).sample()
    torch.manual_seed(c.rows)
    u = torch.rand(z.shape, dtype=torch.float32)                      # the policy's draw: torch.rand
    raw, act, lp = ops.head_sample(BERN, dev(z), None, u.cuda(), act_dim=c.act)
    assert same_bits(raw, act)
    _, _, _, _, pr = bern_ref(z, np.zeros_like(z))
    exempt = (np.abs(u.numpy().astype(np.float64) - pr) <= 10 * U * pr).any(1)
    got = host(act)
    assert np.array_equal(got[~exempt], want.numpy()[~exempt]), c.id
    print(f"{c.id}: {int(exempt.sum())} of {c.rows} rows within the bound of a draw")
    assert exempt.sum() <= max(1, c.rows // 100)
    r_lp, _, b_lp, _, _ = bern_ref(z, got)
    check_within(c.id, host(lp), r_lp, b_lp)


@pytest.mark.gpu
def test_bernoulli_null_outputs_and_exact_ties():
    """Each output of the Bernoulli sampler may be NULL; the draw is strict: logit 0 (p = 0.5 exactly) with u = 0.5
    gives 0, u = nextafter(0.5, 0) gives 1."""
    from ppo_and_friends_b200 import ops
    from ppo_and_friends_b200._lib import load, ptr, stream_ptr
    n, k = 129, 3
    z = bern_logits(n, k, 3)
    z[127] = 0.0
    z[128] = 0.0
    u = np.random.default_rng(3).random((n, k)).astype(np.float32)
    u[127] = 0.5
    u[128] = np.nextafter(np.float32(0.5), np.float32(0))
    zd, ud = dev(z), dev(u)
    raw, act, lp = ops.head_sample(BERN, zd, None, ud, act_dim=k)
    assert host(act)[127].tolist() == [0, 0, 0] and host(act)[128].tolist() == [1, 1, 1]
    for keep in ("raw", "act", "none"):
        o_raw = torch.full((n, k), 7.0, device="cuda")
        o_act = torch.full((n, k), 7.0, device="cuda")
        o_lp = torch.empty(n, device="cuda")
        _lib.check(load().ppoaf_head_sample(BERN, ptr(zd), k, None, MIN_STD, ptr(ud), None, None, k, n,
                                            ptr(o_raw) if keep == "raw" else None,
                                            ptr(o_act) if keep == "act" else None, ptr(o_lp), stream_ptr()))
        assert same_bits(o_lp, lp)
        assert torch.equal(o_raw, raw) if keep == "raw" else bool((o_raw == 7).all())
        assert torch.equal(o_act, act) if keep == "act" else bool((o_act == 7).all())
    lp_e = torch.empty(n, device="cuda")
    _lib.check(load().ppoaf_head_evaluate(BERN, ptr(zd), k, None, MIN_STD, ptr(act), k, n, ptr(lp_e), None,
                                          stream_ptr()))
    assert same_bits(lp_e, ops.head_evaluate(BERN, zd, None, act)[0])


# ---- GPU: Categorical and multi-categorical sampling ---------------------------------------------------------------
def draw_sections(probs, sizes, seed):
    """torch.distributions' actions (one Categorical per section, in order) and the same draws as section-major noise."""
    from torch.distributions import Categorical
    t = torch.as_tensor(probs)
    torch.manual_seed(seed)
    want = torch.stack([Categorical(probs=t[:, o:o + n]).sample() for o, n in sections_of(sizes)], 1)
    torch.manual_seed(seed)
    noise = torch.cat([torch.empty(t.shape[0], n).exponential_(1).reshape(-1) for n in sizes])
    return want.numpy(), noise


def sample_exempt(probs, noise, sizes):
    """Rows whose two largest float64 p~/q in some section lie within 2 (gamma(n) + 2u) of each other."""
    n_rows = probs.shape[0]
    q = noise.numpy().astype(np.float64)
    ex = np.zeros(n_rows, bool)
    for o, n in sections_of(sizes):
        blk = probs[:, o:o + n].astype(np.float64)
        v = blk / blk.sum(1, keepdims=True) / q[n_rows * o:n_rows * (o + n)].reshape(n_rows, n)
        if n > 1:
            top = -np.sort(-v, 1)[:, :2]
            ex |= top[:, 0] - top[:, 1] <= 2 * (gamma(n) + 2 * U) * top[:, 0]
    return ex


def sample_lp_ref(probs, acts, sizes, p):
    pr = probs.astype(np.float64)
    pn, lg, _, e_lg = cat_columns(pr, np.zeros_like(pr), sections_of(sizes), p)
    rows = np.arange(pr.shape[0])
    cols = np.stack([lg[rows, o + acts[:, k]] for k, (o, _) in enumerate(sections_of(sizes))], 1)
    errs = np.stack([e_lg[rows, o + acts[:, k]] for k, (o, _) in enumerate(sections_of(sizes))], 1)
    with np.errstate(invalid="ignore"):
        return cols.sum(1), errs.sum(1) + gamma(len(sizes)) * np.abs(cols).sum(1)


def _check_sampled(name, probs, sizes, want, noise, act, lp, p):
    exempt = sample_exempt(probs, noise, sizes)
    assert np.array_equal(act[~exempt], want[~exempt]), name
    print(f"{name}: {int(exempt.sum())} of {len(act)} rows within the bound of a draw")
    assert exempt.sum() <= max(1, len(act) // 100)
    r_lp, b_lp = sample_lp_ref(probs, act, sizes, p)
    check_within(name, lp, r_lp, b_lp)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CAT_CASES, ids=lambda c: c.id)
def test_categorical_sample_matches_torch(c):
    from ppo_and_friends_b200 import ops
    probs = torch.softmax(torch.as_tensor(cat_logits(c.rows, c.pred, c.pred * 17 + c.rows)), 1).numpy()
    want, noise = draw_sections(probs, [c.pred], c.rows)
    raw, act, lp = ops.head_sample(CAT, dev(probs), None, noise.cuda())
    raw2, act2, lp2 = ops.head_sample(CAT, dev(probs), None, noise.cuda())
    assert torch.equal(raw, act) and torch.equal(act, act2) and same_bits(lp, lp2)
    _check_sampled(c.id, probs, [c.pred], want, noise, host(act), host(lp), plan(CAT, c.pred, 1, c.rows)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("c", MCAT_CASES, ids=lambda c: c.id)
def test_multi_categorical_sample_matches_torch(c):
    from ppo_and_friends_b200 import ops
    sizes = MCAT_TABLES[c.id.split("-")[2]]
    probs = torch.softmax(torch.as_tensor(cat_logits(c.rows, c.pred, c.rows * 3 + len(sizes))), 1).numpy()
    want, noise = draw_sections(probs, sizes, c.rows + 1)
    act, lp = ops.multi_categorical_sample(dev(probs), ends_of(sizes), noise.cuda(), len(sizes))
    _check_sampled(c.id, probs, sizes, want, noise, host(act), host(lp), "thread")


TIES = {"cat-thread-P64": (64, [(3, 35), (10, 11)]),                  # in one thread: columns 3 / 35, 10 / 11
        "cat-warp-P97": (97, [(40, 72), (40, 70)])}                   # one lane (40 / 72), two lanes (40 / 70)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TIES) + ["mcat-thread-straddle"])
def test_sampling_exact_ties_take_the_first_column(name):
    """Equal p~/q at two columns, and q = 0 at two columns with p > 0 (+inf twice): the lower column wins."""
    from ppo_and_friends_b200 import ops
    if name.startswith("mcat"):
        sizes, pairs = MCAT_TABLES["straddle"], [(30, 33), (31, 32)]
    else:
        sizes, pairs = [TIES[name][0]], TIES[name][1]
    P, rows = sum(sizes), 2 * len(pairs)
    probs = np.full((rows, P), 0.1 / P, np.float32)
    q = np.ones((rows, P), np.float32)
    for r, (a, b) in enumerate(pairs * 2):
        probs[r, [a, b]] = 0.3
        q[r, [a, b]] = 0.5 if r < len(pairs) else 0.0
    ends = ends_of(sizes)
    noise = torch.cat([torch.as_tensor(q[:, o:o + n]).reshape(-1) for o, n in sections_of(sizes)])
    if name.startswith("mcat"):
        act, lp = ops.multi_categorical_sample(dev(probs), ends, noise.cuda(), len(sizes))
        got = [int(host(act)[r, 1]) + 30 for r in range(rows)]
    else:
        _, act, lp = ops.head_sample(CAT, dev(probs), None, noise.cuda())
        got = host(act)[:, 0].tolist()
    assert got == [min(a, b) for a, b in pairs * 2]
    assert np.isfinite(host(lp)).all()


# ---- GPU: non-finite plants ----------------------------------------------------------------------------------------
KINDS = {"nan": np.nan, "inf": np.inf, "-inf": -np.inf}


def plant_rows(p):
    """Rows just before and just after three block (thread plan) or CTA (warp plan) edges, and the row count."""
    E = ROW_BLOCK if p == "thread" else WIDE_ROWS_PER_CTA
    return [E - 1, E, 2 * E - 1, 2 * E, 3 * E - 1, 3 * E], 3 * E + 5


def plant(a, rows, value, ncol):
    a = a.copy()
    cols = [0, ncol // 2, ncol - 1]
    for k, r in enumerate(rows):
        a[r, cols[k % 3]] = value
    return a


def check_planted(name, got, ref, clean, rows):
    got = np.asarray(got)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), (name, np.flatnonzero(np.isnan(got)), np.flatnonzero(np.isnan(ref)))
    assert np.array_equal(np.isfinite(got), np.isfinite(ref)), name
    other = np.setdiff1d(np.arange(len(got)), rows)
    assert np.array_equal(got[other].view(np.int32), np.asarray(clean)[other].view(np.int32)), name


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 97], ids=["thread", "warp"])
@pytest.mark.parametrize("site", ["mean", "action", "log_std"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_gaussian_nonfinite_plants(kind, site, d):
    from ppo_and_friends_b200 import ops
    p = plan(GAUSS, d, d, 1)[0]
    rows, n = plant_rows(p)
    mean, ls, x = gauss_inputs(Case("", "gauss", d, d, n), 5)
    torch.manual_seed(0)
    noise = torch.randn(n, d)
    clean_e = ops.head_evaluate(GAUSS, dev(mean), dev(ls), dev(x))
    clean_s = ops.head_sample(GAUSS, dev(mean), dev(ls), noise.cuda(), act_dim=d)
    v = KINDS[kind]
    if site == "log_std":
        ls = ls.copy()
        ls[[0, d // 2, d - 1]] = v
        rows = list(range(n))
    elif site == "mean":
        mean = plant(mean, rows, v, d)
    else:
        x = plant(x, rows, v, d)
    lp, ent = ops.head_evaluate(GAUSS, dev(mean), dev(ls), dev(x))
    r_lp, r_ent, _, _ = gauss_ref(mean, ls, x, p)
    check_planted(f"eval-{site}", host(lp), r_lp, host(clean_e[0]), rows)
    check_planted(f"ent-{site}", host(ent), r_ent, host(clean_e[1]), rows)
    if site == "action":
        return
    raw, act, lps = ops.head_sample(GAUSS, dev(mean), dev(ls), noise.cuda(), act_dim=d)
    r_raw, _, r_act, _ = gauss_sample_ref(mean, ls, noise.numpy(), None, None)
    assert np.array_equal(np.isnan(host(raw)), np.isnan(r_raw)) and np.array_equal(np.isnan(host(act)), np.isnan(r_act))
    assert np.array_equal(np.isfinite(host(raw)), np.isfinite(r_raw))
    r_lps, _, _, _ = gauss_ref(mean, ls, host(raw), p)
    check_planted(f"sample-{site}", host(lps), r_lps, host(clean_s[2]), rows)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [64, 97], ids=["thread", "warp"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_categorical_nonfinite_plants(kind, P):
    """Logits planted for evaluation, probabilities for sampling (the noise stays finite).  A sampled row with a NaN
    takes column 0 and a NaN log-prob."""
    from ppo_and_friends_b200 import ops
    p = plan(CAT, P, 1, 1)[0]
    rows, n = plant_rows(p)
    z = cat_logits(n, P, 9)
    acts = np.random.default_rng(1).integers(0, P, (n, 1)).astype(np.int64)
    clean = ops.head_evaluate(CAT, dev(z), None, dev(acts))
    zp = plant(z, rows, KINDS[kind], P)
    lp, ent = ops.head_evaluate(CAT, dev(zp), None, dev(acts))
    r_lp, r_ent, _, _ = cat_eval_ref(zp, acts, [P], p)
    check_planted("eval", host(lp), r_lp, host(clean[0]), rows)
    check_planted("ent", host(ent), r_ent, host(clean[1]), rows)

    probs = torch.softmax(torch.as_tensor(z), 1).numpy()
    _, noise = draw_sections(probs, [P], 2)
    _, clean_a, clean_lp = ops.head_sample(CAT, dev(probs), None, noise.cuda())
    pp = plant(probs, rows, KINDS[kind], P)
    _, act, lps = ops.head_sample(CAT, dev(pp), None, noise.cuda())
    act, lps = host(act)[:, 0], host(lps)
    q = noise.numpy().reshape(n, P).astype(np.float64)
    with np.errstate(invalid="ignore"):
        v = pp / pp.astype(np.float64).sum(1, keepdims=True) / q
    for r in rows:                                                    # first maximum of the comparable p~/q, else 0
        ok = ~np.isnan(v[r])
        assert act[r] == (int(np.flatnonzero(ok & (v[r] == v[r][ok].max()))[0]) if ok.any() else 0), r
    if kind == "nan":
        assert (act[rows] == 0).all()
    r_lp, _ = sample_lp_ref(pp, act.reshape(-1, 1), [P], p)
    check_planted("sample", lps, r_lp, host(clean_lp), rows)
    other = np.setdiff1d(np.arange(n), rows)
    assert np.array_equal(act[other], host(clean_a)[other, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_bernoulli_and_multi_categorical_nonfinite_plants(kind):
    from ppo_and_friends_b200 import ops
    rows, n = plant_rows("thread")
    k = 64
    z = bern_logits(n, k, 4)
    x = np.random.default_rng(4).integers(0, 2, z.shape).astype(np.float32)
    clean = ops.head_evaluate(BERN, dev(z), None, dev(x))
    zp = plant(z, rows, KINDS[kind], k)
    lp, ent = ops.head_evaluate(BERN, dev(zp), None, dev(x))
    r_lp, r_ent, _, _, _ = bern_ref(zp, x)
    check_planted("bern-eval", host(lp), r_lp, host(clean[0]), rows)
    check_planted("bern-ent", host(ent), r_ent, host(clean[1]), rows)
    u = torch.rand(n, k)
    _, ca, clp = ops.head_sample(BERN, dev(z), None, u.cuda(), act_dim=k)
    _, act, lps = ops.head_sample(BERN, dev(zp), None, u.cuda(), act_dim=k)
    r_lps, _, _, _, _ = bern_ref(zp, host(act))
    check_planted("bern-sample", host(lps), r_lps, host(clp), rows)

    sizes = MCAT_TABLES["straddle"]
    zm = cat_logits(n, sum(sizes), 6)
    am = np.stack([np.random.default_rng(6).integers(0, s, n) for s in sizes], 1).astype(np.int64)
    clean = ops.multi_categorical_evaluate(dev(zm), ends_of(sizes), dev(am))
    zmp = plant(zm, rows, KINDS[kind], sum(sizes))
    lp, ent = ops.multi_categorical_evaluate(dev(zmp), ends_of(sizes), dev(am))
    r_lp, r_ent, _, _ = cat_eval_ref(zmp, am, sizes, "thread")
    check_planted("mcat-eval", host(lp), r_lp, host(clean[0]), rows)
    check_planted("mcat-ent", host(ent), r_ent, host(clean[1]), rows)
    probs = torch.softmax(torch.as_tensor(zm), 1).numpy()
    _, noise = draw_sections(probs, sizes, 3)
    _, clp = ops.multi_categorical_sample(dev(probs), ends_of(sizes), noise.cuda(), len(sizes))
    pp = plant(probs, rows, KINDS[kind], sum(sizes))
    act, lps = ops.multi_categorical_sample(dev(pp), ends_of(sizes), noise.cuda(), len(sizes))
    r_lps, _ = sample_lp_ref(pp, host(act), sizes, "thread")
    check_planted("mcat-sample", host(lps), r_lps, host(clp), rows)
    if kind == "nan":
        for k_, r in enumerate(rows):                                 # the planted column's section takes column 0
            col = [0, sum(sizes) // 2, sum(sizes) - 1][k_ % 3]
            sec = next(i for i, (o, s) in enumerate(sections_of(sizes)) if o <= col < o + s)
            assert host(act)[r, sec] == 0


# ---- argument refusals (zero rows: nothing is launched) -------------------------------------------------------------
def test_missing_arguments_are_refused_before_the_zero_row_return():
    from ppo_and_friends_b200.build import build
    build()
    lib = _lib.load()
    msg = lambda: lib.ppoaf_last_error().decode()
    f = C.c_void_p(16)                                                # never dereferenced: zero rows
    ev = lambda head, log_std, lp, pred=4, act=4: lib.ppoaf_head_evaluate(head, f, pred, log_std, MIN_STD, f, act, 0,
                                                                         lp, None, None)
    assert ev(GAUSS, f, f) == 0 and ev(CAT, None, f, 70, 1) == 0 and ev(BERN, None, f) == 0
    assert ev(GAUSS, None, f) != 0 and "log_std" in msg()
    assert ev(GAUSS, None, f, 65, 65) != 0 and "log_std" in msg()
    for head, ls, pred, act in ((GAUSS, f, 4, 4), (CAT, None, 4, 1), (CAT, None, 70, 1), (BERN, None, 4, 4)):
        assert ev(head, ls, None, pred, act) != 0 and "log_prob_out" in msg()

    sm = lambda head, log_std, raw, act, lp, pred=4, ad=4: lib.ppoaf_head_sample(
        head, f, pred, log_std, MIN_STD, f, None, None, ad, 0, raw, act, lp, None)
    assert sm(GAUSS, f, f, f, f) == 0 and sm(CAT, None, None, f, f, 4, 1) == 0
    assert sm(BERN, None, None, None, f) == 0                         # Bernoulli outputs stay nullable
    for pred in (4, 65):
        assert sm(GAUSS, None, f, f, f, pred, pred) != 0 and "log_std" in msg()
        assert sm(GAUSS, f, None, f, f, pred, pred) != 0 and "raw_action_out" in msg()
        assert sm(GAUSS, f, f, None, f, pred, pred) != 0 and "action_out" in msg()
        assert sm(GAUSS, f, f, f, None, pred, pred) != 0 and "log_prob_out" in msg()
    for pred in (4, 70):
        assert sm(CAT, None, f, None, f, pred, 1) != 0 and "action_out" in msg()
        assert sm(CAT, None, f, f, None, pred, 1) != 0 and "log_prob_out" in msg()
    assert sm(BERN, None, f, f, None) != 0 and "log_prob_out" in msg()

    ends = ends_of([3, 4])
    assert lib.ppoaf_multi_categorical_evaluate(f, 7, ends, 0, f, 2, 0, f, None, None) == 0
    assert lib.ppoaf_multi_categorical_evaluate(f, 7, ends, 0, f, 2, 0, None, None, None) != 0
    assert "log_prob_out" in msg()
    assert lib.ppoaf_multi_categorical_sample(f, 7, ends, 0, f, 2, 0, f, f, None) == 0
    for noise, act, lp in ((None, f, f), (f, None, f), (f, f, None)):
        assert lib.ppoaf_multi_categorical_sample(f, 7, ends, 0, noise, 2, 0, act, lp, None) != 0
        assert "required" in msg()


# ---- GPU: a NaN log_std through the update ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["chain", "fused"])
def test_update_counts_a_nan_log_std_as_a_bad_ratio(engine, monkeypatch):
    """A NaN in a Gaussian actor's log_std gives every sample a NaN std, log-prob and ratio, which the step's
    bad-ratio counter records for every sample of the epoch (ppo_batch_train then aborts, as the reference's NaN check
    does)."""
    from helpers import make_policy, run_device_rollout
    from ppo_and_friends_b200.ppo import PPOUpdateState, _get_engine
    from ppo_and_friends_b200.synthetic import make_rollout
    monkeypatch.setenv("PPOAF_STEP", engine)
    ro = make_rollout(seed=3, T=48, E=8, obs_dim=8, act_dim=2, max_ts_per_ep=16, obs_scale=False)
    torch.manual_seed(0)
    pol = make_policy(ro, act="leaky_relu", actor_hidden=64, critic_hidden=64, lr=3e-4)
    ds = run_device_rollout(pol, ro)
    pol.actor.state_dict()["distribution.log_std"][1] = float("nan")
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    eng = _get_engine(state, "pol", 128)
    st = eng.run_epoch(ds).numpy()
    assert eng.fused == (engine == "fused")
    assert st[_lib.ST["BAD_RATIO"]] == ds.observations.shape[0]


