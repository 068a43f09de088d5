"""
The forward GEMMs and softmax of ppoaf_mlp_forward (csrc/mlp.cuh, csrc/umma.cuh, csrc/mlp.cu) and the clip + Adam step
of ppoaf_clip_adam_step (csrc/optim.cu), each through the C ABI against a float64 restatement, at the launch plans the
host code picks among.

`ffma_plan`, `tc_plan` and `adam_plan` restate the host-side plan choice (tile counts of mlp.cu, the K rounds and
per-warp K slices of mlp.cuh, the chunk ring of umma.cuh, the grids of optim.cu).  They name the cases, choose shapes
at plan edges and give the number of float32 roundings on a path; no result is compared with anything they compute.

Bounds, with u = 2^-24 (the unit roundoff of float32) and gamma(d) = d u / (1 - d u):
  FFMA forward      Integer-valued operands (|x|, |w|, |b| <= 8, every partial sum < 2^24): bit-exact.  Random
                    operands: |y - ref| <= gamma(d) (|x| |W|^T + |b|), d = the FMAs of one warp's K slices over all
                    rounds + 16 for the split-K fold and the bias add.
  tcgen05 forward   Integer-valued operands: bit-exact (tf32 holds them, the lo parts are 0).  Random operands: every
                    product misses lo*lo and the tf32 rounding of the two lo parts, <= 3 * 2^-22 |x| |w|; the tensor
                    core accumulates the 3 K_pad products in float32 without a stated rounding mode, so each addition
                    is allowed 2u: |y - ref| <= (3 * 2^-22 + 2u (3 K_pad + 2)) (|x| |W|^T + |b|).
  fast_tanh         __expf within 2 + 1.173 |2x| ulp of t = e^2x (at most 2^-22 on tanh, whose slope in ln t is
                    <= 1/2), t + 1 rounded (<= 2^-22 on 2 / (t + 1) <= 2), __fdividef within 2 ulp (<= 2^-22),
                    the final subtraction <= 2^-24: |fast_tanh(z) - tanh(z)| <= 2^-20 absolute.
  activation sweep  FFMA: the pre-activation is exactly z and the identity layer is exact, so the error is the
                    activation's alone (tanh: 2^-20; leaky relu: 0.01f z, one rounding, within 2u of 0.01 z; relu:
                    exact).  tcgen05: the hi/lo split of z and of h loses <= 2^-22 each, so add
                    2^-22 (|act(z)| + |z act'(z)|).
  depth             the GEMM bound of each layer plus the propagated input error |W| e_in, then + 2^-20 after a
                    tanh and + 2u |y| after a leaky relu.
  softmax           e_j = expf(l_j - mx): the subtraction rounds (u |l_j - mx|), expf <= 2 ulp (4u); the row sum
                    adds n_add u (n - 1 sequential additions in the narrow kernel, ceil(n / 32) + 5 in the wide one's
                    lanes and shuffles) plus the weighted errors of its terms; the division 1u.  Underflowed terms:
                    + 2^-126 absolute.
  clip + Adam       per step, from the kernel's own float32 (p, m, v) and with the kernel's float32 scalars:
                    coefficient within 7u of float64 when clipping binds (four float32 roundings of the squares,
                    the float conversion, + 1e-6f, the division), exactly 1 otherwise; g' = g inv_world coef
                    within e_g = (2u + that) |g'|; m = m + w1 (g' - m) within 4u (|m| + w1 |g'|) + w1 e_g;
                    v = v b2 + (w2 g') g' within 3u (b2 |v| + w2 g'^2) + 2 w2 |g'| e_g; the step
                    p + (-lr / bc1) m / (sqrt(v) / sqrt(bc2) + eps) within |lr / bc1| e_m / denom +
                    (18u + e_v / 2v) |step| + u |p| (sqrt.approx and the two __fdividef within 2 ulp each, the
                    bias corrections one float32 ulp each from a chained versus a pow() beta^t).
                    Trajectories against torch.optim.Adam(foreach=False) in float32: the project's 2e-6 relative,
                    1e-7 absolute (15 steps of at most u |p| + 30u |step| apart each).
"""
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

U = 2.0 ** -24
TANH_ABS = 2.0 ** -20
TF32_SPLIT = 3 * 2.0 ** -22

# ---- restated launch plans ----------------------------------------------------------------------------------------
KBM, KBN, KROUND, KGROUPS = 32, 64, 512, 16          # mlp.cuh
KUM, KUN, KUK, KUSTAGES = 128, 64, 32, 3              # umma.cuh
ADAM_THREADS, ADAM_SLOTS = 1024, 2                   # optim.cu


def cdiv(a, b):
    return -(-a // b)


FfmaPlan = namedtuple("FfmaPlan", "tiles rounds kw_total warps_last flavour")
TcPlan = namedtuple("TcPlan", "tiles chunks wraps ragged flavour")


def flavour(K, x_off, p_off, w_off_floats):
    """mlp.cu add_forward: bit 1 = x rows take 16-byte loads, bit 0 = W rows do."""
    x_vec = x_off == 0 and K % 4 == 0
    w_vec = (p_off + w_off_floats) % 4 == 0 and K % 4 == 0
    return 2 * int(x_vec) + int(w_vec)


def ffma_plan(rows, K, N, flav=None):
    kw_total, warps_last = 0, 0
    for r in range(cdiv(K, KROUND)):
        Kr = min(K - r * KROUND, KROUND)
        Kr4 = (Kr + 3) & ~3
        Kw = (cdiv(Kr, KGROUPS) + 3) & ~3
        kw_total += Kw
        warps_last = cdiv(Kr4, Kw)
    return FfmaPlan(cdiv(rows, KBM) * cdiv(N, KBN), cdiv(K, KROUND), kw_total, warps_last, flav)


def tc_plan(rows, K, N, flav=None):
    chunks = cdiv(K, KUK)
    return TcPlan(cdiv(rows, KUM) * cdiv(N, KUN), chunks, chunks > KUSTAGES, K % KUK != 0, flav)


def ffma_depth(K):
    return ffma_plan(1, K, 1).kw_total + KGROUPS


def gamma(d):
    return d * U / (1 - d * U)


def gemm_bound(backend, K, absprod):
    if backend == "ffma":
        return gamma(ffma_depth(K)) * absprod
    k_pad = cdiv(K, KUK) * KUK
    return (TF32_SPLIT + 2 * U * (3 * k_pad + 2)) * absprod


def adam_plan(nv, sm):
    grid = max(1, min(cdiv(nv, ADAM_THREADS), sm))
    stride = grid * ADAM_THREADS
    passes = cdiv(nv, stride)
    return grid, ("1slot" if passes == 1 else "2slot" if passes == 2 else f"tail{passes - ADAM_SLOTS}")


# ---- float64 restatements -----------------------------------------------------------------------------------------
def act64(z, act):
    if act == "tanh":
        return np.tanh(z)
    if act == "relu":
        return np.where(z > 0, z, 0.0)
    if act == "leaky_relu":
        return np.where(z > 0, z, 0.01 * z)
    return z


def forward64(layers, x, act):
    """layers: [(W [out, in], b [out])] as float32 arrays; float64 forward, identity after the last layer."""
    h = np.asarray(x, np.float64)
    for l, (W, b) in enumerate(layers):
        h = h @ W.astype(np.float64).T + b.astype(np.float64)
        if l + 1 < len(layers):
            h = act64(h, act)
    return h


def softmax64(logits):
    z = np.asarray(logits, np.float64)
    e = np.exp(z - z.max(-1, keepdims=True))
    return e / e.sum(-1, keepdims=True)


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


def adam_step64(p, g, m, v, t, hp, n_actor, f32_scalars=True):
    """One clip + Adam step in float64 -> (p, m, v, coef_a, coef_c, bounds dict)."""
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
        e_m = 4 * U * (np.abs(m) + s["w1"] * np.abs(gk)) + s["w1"] * gk_err
        e_v = 3 * U * (s["b2"] * np.abs(v) + s["w2"] * gk * gk) + 2 * s["w2"] * np.abs(gk) * gk_err
        rel_v = np.divide(e_v, v1, out=np.zeros_like(v1), where=v1 > 0)
        e_p = abs(s["neg_step"]) * e_m / denom + (18 * U + rel_v / 2) * np.abs(step) + U * np.abs(p1)
    return p1, m1, v1, coefs, dict(p=e_p, m=e_m, v=e_v)


# ---- cases --------------------------------------------------------------------------------------------------------
FFMA_K = (1, 2, 3, 4, 5, 63, 64, 65, 511, 512, 513, 1029, 2051)
FFMA_N = (1, 3, 63, 64, 65, 130)
FFMA_ROWS = (1, 31, 32, 33, 513)
TC_K = (1, 31, 32, 33, 96, 97, 128, 1025)
TC_ROWS = (1, 127, 128, 129, 300)
TC_N = (1, 63, 64, 65)
WAVE = -1            # rows whose FFMA tile count exceeds two CTAs per SM: derived from the SM count


def gemm_cases():
    cases = [("ffma", 33, K, N) for K in FFMA_K for N in FFMA_N]
    cases += [("ffma", rows, K, N) for rows in FFMA_ROWS for K, N in ((5, 65), (513, 64), (64, 130)) if rows != 33]
    cases += [("ffma", WAVE, 64, 64)]
    cases += [("tcgen05", 129, K, N) for K in TC_K for N in TC_N]
    cases += [("tcgen05", rows, K, N) for rows in TC_ROWS for K, N in ((97, 65), (33, 1), (128, 64)) if rows != 129]
    return cases


def gemm_id(c):
    backend, rows, K, N = c
    if rows == WAVE:
        return f"ffma-wave-beyond-2-ctas-per-sm-K{K}-N{N}"
    if backend == "ffma":
        p = ffma_plan(rows, K, N)
        return f"ffma-t{p.tiles}-r{p.rounds}-w{p.warps_last}-rows{rows}-K{K}-N{N}"
    p = tc_plan(rows, K, N)
    return (f"tcgen05-t{p.tiles}-c{p.chunks}{'-wrap' if p.wraps else ''}{'-ragged' if p.ragged else ''}"
            f"-rows{rows}-K{K}-N{N}")


GEMM_CASES = gemm_cases()

# (backend, K, x offset, params offset, y offset) in floats; flavour per mlp.cu add_forward
ALIGN_CASES = [(b, K, xo, po, yo) for b in ("ffma", "tcgen05") for K in (64, 65) for xo in (0, 1, 3) for po in (0, 1)
               for yo in (0, 1)] + [(b, 64, 2, 0, 0) for b in ("ffma", "tcgen05")]


def align_id(c):
    b, K, xo, po, yo = c
    return f"{b}-flavour{flavour(K, xo, po, 0)}-K{K}-xoff{xo}-poff{po}-yoff{yo}"


# Z values of the activation sweep
Z_MAG = (0.0, 1e-30, 1e-6, 0.01, 0.5, 1.0, 10.0, 43.0, 44.5, 89.0, 1e30)
Z_SWEEP = np.array([s * z for z in Z_MAG for s in (1.0, -1.0)], dtype=np.float32)

SOFTMAX_CASES = [(n, rows) for n in (1, 2, 63, 64) for rows in (127, 128, 129)] + \
                [(n, rows) for n in (65, 4672, 65536) for rows in (7, 8, 9)]

# Adam plans: nv = a * S + b float4 slots (S = SM count); n_actor likewise in float4 slots
ADAM_NV = [(0, 1), (0, 1023), (0, 1024), (0, 1025), (1024, -1), (1024, 0), (1024, 1), (2048, 0), (2048, 1), (5120, 3)]
ADAM_SPLITS = [(0, 0), (5120, 3), (0, 100), (0, 1024), (1024, 37), (2048, 1000)]   # n_actor on nv = 5120 S + 3


def sym(ab):
    a, b = ab
    return f"{a}S{b:+d}" if a else str(b)


def resolve(ab, sm):
    return ab[0] * sm + ab[1]


def adam_cases():
    cases = [(nv, (0, -2)) for nv in ADAM_NV]          # (0, -2): n_actor = half of the slots
    cases += [((5120, 3), na) for na in ADAM_SPLITS]
    return cases


def adam_id(c):
    nv, na = c
    return f"nv{sym(nv)}-na{'half' if na == (0, -2) else sym(na)}"


def resolve_split(nv, na, sm):
    return nv // 2 if na == (0, -2) else resolve(na, sm)


# ---- CPU checks of the restatements and case tables ---------------------------------------------------------------
@pytest.mark.parametrize("sm", [132, 148, 160])
def test_case_tables_reach_every_launch_plan(sm):
    """(CPU) the case tables reach every plan the host code can pick, for any SM count."""
    flavours = {flavour(K, xo, po, 0) for b, K, xo, po, yo in ALIGN_CASES}
    assert flavours == {0, 1, 2, 3}
    assert {(flavour(K, xo, po, 0), K % 4 == 0) for b, K, xo, po, yo in ALIGN_CASES} >= {(0, True), (0, False)}
    ffma = [ffma_plan(r, K, N) for b, r, K, N in GEMM_CASES if b == "ffma" and r != WAVE]
    assert {p.rounds for p in ffma} >= {1, 2, 3, 5}
    assert {p.warps_last for p in ffma} >= {1, 2, 16}
    wave_rows = KBM * (2 * sm + 1)
    assert ffma_plan(wave_rows, 64, 64).tiles > 2 * sm
    tc = [tc_plan(r, K, N) for b, r, K, N in GEMM_CASES if b == "tcgen05"]
    assert {(p.wraps, p.ragged) for p in tc} == {(False, False), (False, True), (True, False), (True, True)}
    assert {p.chunks for p in tc} >= {1, 2, 3, 4, 33}
    plans = {adam_plan(resolve(nv, sm), sm)[1] for nv, _ in adam_cases()}
    assert {"1slot", "2slot", "tail1", "tail4"} <= plans
    grids = {adam_plan(resolve(nv, sm), sm)[0] for nv, _ in adam_cases()}
    assert {1, 2, sm} <= grids
    nv = resolve((5120, 3), sm)
    stride = sm * ADAM_THREADS
    where = set()
    for na in ADAM_SPLITS:
        i = resolve(na, sm)
        where.add("none" if i == 0 else "all" if i == nv else "cta0" if i < ADAM_THREADS else
                  "cta-edge" if i % ADAM_THREADS == 0 and i < stride else "slot2" if i < 2 * stride else "tail")
    assert where == {"none", "all", "cta0", "cta-edge", "slot2", "tail"}


def test_forward_restatement_matches_torch_float64():
    """(CPU) forward64 / act64 / softmax64 against torch in float64."""
    rng = np.random.default_rng(0)
    dims = [7, 33, 20, 5]
    layers = [(rng.standard_normal((dims[l + 1], dims[l])).astype(np.float32),
               rng.standard_normal(dims[l + 1]).astype(np.float32)) for l in range(3)]
    x = rng.standard_normal((11, 7)).astype(np.float32)
    mods = {"tanh": torch.tanh, "relu": torch.relu, "leaky_relu": torch.nn.functional.leaky_relu}
    for act, fn in mods.items():
        h = torch.from_numpy(x).double()
        for l, (W, b) in enumerate(layers):
            h = torch.nn.functional.linear(h, torch.from_numpy(W).double(), torch.from_numpy(b).double())
            if l + 1 < len(layers):
                h = fn(h)
        np.testing.assert_allclose(forward64(layers, x, act), h.numpy(), rtol=1e-13, atol=1e-13)
        z = torch.from_numpy(Z_SWEEP.astype(np.float64))
        np.testing.assert_allclose(act64(Z_SWEEP.astype(np.float64), act), fn(z).numpy(), rtol=1e-15, atol=0)
    logits = np.concatenate([rng.standard_normal((3, 70)) * 30, np.full((1, 70), 5.0), 1e4 + rng.standard_normal((1, 70))])
    np.testing.assert_allclose(softmax64(logits), torch.softmax(torch.from_numpy(logits), -1).numpy(), rtol=1e-13,
                               atol=1e-300)


def _torch_step(params, grads, opts, max_norm):
    for p, g, o in zip(params, grads, opts):
        p.grad = g.clone()
        if max_norm >= 0:
            torch.nn.utils.clip_grad_norm_([p], max_norm, foreach=False)
        o.step()


def test_adam_restatement_matches_torch_float64():
    """(CPU) adam_step64 with exact scalars against torch clip_grad_norm_ + Adam(foreach=False) in float64, through a
    betas change, a binding and a non-binding clip, and a NaN gradient under clipping."""
    rng = np.random.default_rng(1)
    n_a, n = 40, 64
    p = rng.standard_normal(n)
    m, v = np.zeros(n), np.zeros(n)
    hp = dict(LR=1e-3, GRAD_CLIP=0.5, BETA1=0.9, BETA2=0.999, ADAM_EPS=1e-5, INV_WORLD=1.0)
    tp = [torch.tensor(p[:n_a], requires_grad=True), torch.tensor(p[n_a:], requires_grad=True)]
    opts = [torch.optim.Adam([t], lr=hp["LR"], eps=hp["ADAM_EPS"], foreach=False) for t in tp]
    for t in range(1, 9):
        if t == 5:
            hp.update(BETA1=0.5, BETA2=0.9)
            for o in opts:
                o.param_groups[0]["betas"] = (0.5, 0.9)
        g = rng.standard_normal(n) * (3.0 if t % 2 else 0.01)
        if t == 8:
            g[3] = np.nan
        p, m, v, _, _ = adam_step64(p, g, m, v, t, hp, n_a, f32_scalars=False)
        _torch_step(tp, [torch.tensor(g[:n_a]), torch.tensor(g[n_a:])], opts, hp["GRAD_CLIP"])
        ref = torch.cat([x.detach() for x in tp]).numpy()
        assert np.array_equal(np.isnan(p), np.isnan(ref))
        np.testing.assert_allclose(p, ref, rtol=1e-13, atol=1e-15)
        st = [o.state[x] for o, x in zip(opts, tp)]
        np.testing.assert_allclose(m, np.concatenate([s["exp_avg"].numpy() for s in st]), rtol=1e-13, atol=1e-300)
        np.testing.assert_allclose(v, np.concatenate([s["exp_avg_sq"].numpy() for s in st]), rtol=1e-13, atol=1e-300)
    assert np.isnan(p[:n_a]).all() and np.isfinite(p[n_a:]).all()


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _sm_count():
    from ppo_and_friends_b200 import ops
    return ops.device_info()["sm_count"]


def _placed(x, off, pad=4, dtype=torch.float32):
    """A contiguous copy of x whose base is `off` elements past a 16-byte aligned allocation."""
    buf = torch.full((x.numel() + off + pad,), float("nan"), dtype=dtype, device="cuda")
    view = buf[off:off + x.numel()].view(x.shape)
    view.copy_(x)
    assert view.data_ptr() % 16 == off * buf.element_size() % 16
    return buf, view


class _Backend:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        from ppo_and_friends_b200 import ops
        ops.set_gemm_backend(self.name)

    def __exit__(self, *exc):
        from ppo_and_friends_b200 import ops
        ops.set_gemm_backend("ffma")


def _net(dims, act, layers, p_off=0):
    """Descriptor and flat parameter buffer (at a p_off-float offset) of float32 layers [(W, b)]."""
    from ppo_and_friends_b200 import _lib
    desc = _lib.MlpDesc.make(dims, act)
    offs, total = _lib.param_layout(desc)
    flat = torch.zeros(total)
    for l, (W, b) in enumerate(layers):
        flat[offs[2 * l]:offs[2 * l] + W.size] = torch.from_numpy(W.reshape(-1))
        flat[offs[2 * l + 1]:offs[2 * l + 1] + b.size] = torch.from_numpy(b)
    buf, params = _placed(flat.cuda(), p_off)
    return desc, (buf, params)


def _forward(desc, params, x, idx=None, softmax=False, y_off=None, rows=None):
    """ppoaf_mlp_forward twice (the second launch must be bit-identical); y at a y_off-float offset when given."""
    from ppo_and_friends_b200 import ops
    n = rows if rows is not None else (idx.numel() if idx is not None else x.shape[0])
    outs = []
    for _ in range(2):
        out = None
        if y_off is not None:
            _, out = _placed(torch.zeros(n, desc.dims[desc.n_layers], device="cuda"), y_off)
        outs.append(ops.mlp_forward(desc, params, x, idx=idx, n_rows=n, softmax_out=softmax, out=out))
    torch.cuda.synchronize()
    a, b = (o.cpu().numpy() for o in outs)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "second launch differs"
    return a


def _layers(rng, dims, integer):
    out = []
    for l in range(len(dims) - 1):
        if integer:
            W = rng.integers(-8, 9, (dims[l + 1], dims[l])).astype(np.float32)
            b = rng.integers(-8, 9, dims[l + 1]).astype(np.float32)
        else:
            W = (rng.standard_normal((dims[l + 1], dims[l])) / np.sqrt(dims[l])).astype(np.float32)
            b = (rng.standard_normal(dims[l + 1]) * 0.1).astype(np.float32)
        out.append((W, b))
    return out


def _inputs(rng, rows, K, integer):
    if integer:
        return rng.integers(-8, 9, (rows, K)).astype(np.float32)
    return rng.standard_normal((rows, K)).astype(np.float32)


def _check_gemm(backend, rows, K, N, x_off=0, p_off=0, y_off=None, idx=None, n_src=None, seed=0):
    """One-layer [K, N] net: integer operands bit-exact, random operands within the GEMM bound."""
    rng = np.random.default_rng(seed + 7 * K + N)
    n_src = rows if n_src is None else n_src
    worst = 0.0
    for integer in (True, False):
        layers = _layers(rng, [K, N], integer)
        x = _inputs(rng, n_src, K, integer)
        desc, (pbuf, params) = _net([K, N], "identity", layers, p_off)
        xbuf, xd = _placed(torch.from_numpy(x).cuda(), x_off)
        idx_d = None if idx is None else torch.as_tensor(idx, dtype=torch.int64, device="cuda")
        with _Backend(backend):
            y = _forward(desc, params, xd, idx=idx_d, y_off=y_off, rows=rows)
        xs = x if idx is None else x[np.asarray(idx)]
        ref = forward64(layers, xs, "identity")
        if integer:
            np.testing.assert_array_equal(y.astype(np.float64), ref)
        else:
            W, b = layers[0]
            bound = gemm_bound(backend, K, np.abs(xs.astype(np.float64)) @ np.abs(W.astype(np.float64)).T
                               + np.abs(b.astype(np.float64)))
            err = np.abs(y - ref)
            assert (err <= bound).all(), f"max err {err.max():.3e}, max err/bound {np.max(err / bound):.3f}"
            worst = max(worst, float(np.max(err / bound)))
    return worst


# ---- GPU: forward GEMM --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", GEMM_CASES, ids=gemm_id)
def test_forward_gemm_vs_float64(case):
    backend, rows, K, N = case
    if rows == WAVE:
        rows = KBM * (2 * _sm_count() + 1)
        assert ffma_plan(rows, K, N).tiles > 2 * _sm_count()
    _check_gemm(backend, rows, K, N)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ALIGN_CASES, ids=align_id)
def test_forward_gemm_operand_alignment(case):
    """x at a 1-3 float offset, params at a 1-float offset (W and the bias lose their 16-byte alignment), y through
    out= at a 1-float offset: every operand flavour, for K % 4 == 0 and K % 4 != 0."""
    backend, K, x_off, p_off, y_off = case
    rows = 129 if backend == "tcgen05" else 33
    _check_gemm(backend, rows, K, 64, x_off=x_off, p_off=p_off, y_off=y_off)   # N % 4 == 0: 16-byte stores when y allows


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["ffma", "tcgen05"])
@pytest.mark.parametrize("kind", ["repeats", "reversed"])
@pytest.mark.parametrize("K", [3, 64, 97])
def test_forward_gemm_row_gather(backend, kind, K):
    """An int64 row index with repeats, and a reversed one (no index: every other case)."""
    rng = np.random.default_rng(K)
    n_src, rows = 300, 257
    idx = rng.integers(0, 40, rows) if kind == "repeats" else np.arange(n_src - 1, n_src - 1 - rows, -1)
    _check_gemm(backend, rows, K, 65, idx=idx, n_src=n_src)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["ffma", "tcgen05"])
@pytest.mark.parametrize("act", ["tanh", "relu", "leaky_relu"])
def test_activation_epilogue_sweep(backend, act):
    """[1, H, H] nets: layer 1 makes the pre-activation exactly z, layer 2 is the identity with zero bias."""
    _check_activation(backend, act)


def _check_activation(backend, act):
    H = Z_SWEEP.size
    layers = [(Z_SWEEP.reshape(H, 1).copy(), np.zeros(H, np.float32)), (np.eye(H, dtype=np.float32), np.zeros(H, np.float32))]
    desc, (_, params) = _net([1, H, H], act, layers)
    rows = 5
    with _Backend(backend):
        y = _forward(desc, params, torch.ones(rows, 1, device="cuda"))
    z = Z_SWEEP.astype(np.float64)
    ref = act64(z, act)
    bound = {"tanh": np.full_like(z, TANH_ABS), "relu": np.zeros_like(z), "leaky_relu": 2 * U * np.abs(ref)}[act]
    if backend == "tcgen05":
        slope = {"tanh": 1.0 / np.cosh(np.minimum(np.abs(z), 300.0)) ** 2, "relu": (z > 0).astype(np.float64),
                 "leaky_relu": np.where(z > 0, 1.0, 0.01)}[act]
        bound = bound + 2.0 ** -22 * (np.abs(ref) + np.abs(z) * slope)
    err = np.abs(y - ref)
    assert (err <= bound).all(), [(float(z[j]), float(y[0, j]), float(ref[j])) for j in np.nonzero((err > bound).any(0))[0]]
    if act == "tanh" and backend == "ffma":
        assert np.array_equal(y[:, z == 0], np.zeros((rows, 2), np.float32))
        assert (np.abs(y[:, np.abs(z) >= 44.5]) == 1.0).all()
    return float(np.max(np.divide(err, bound, out=np.zeros_like(err), where=bound > 0))), float(err.max())


DEPTH_NETS = [([24, 96, 40, 7], "tanh"), ([5, 130, 64, 64, 33, 3], "leaky_relu"), ([64, 200, 17, 150, 1], "relu"),
              ([33, 64, 65, 130, 64, 40, 31, 20, 9], "tanh")]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["ffma", "tcgen05"])
@pytest.mark.parametrize("dims,act", DEPTH_NETS, ids=lambda v: "x".join(map(str, v)) if isinstance(v, list) else v)
def test_forward_depth_workspace_ping_pong(backend, dims, act):
    """Nets of depth 3-8 whose widest layer is not the last: the hidden activations alternate between the two halves
    of the workspace.  Bound propagated layer by layer."""
    _check_depth(backend, dims, act)


def _check_depth(backend, dims, act):
    rng = np.random.default_rng(len(dims))
    layers = _layers(rng, dims, integer=False)
    rows = 300
    x = _inputs(rng, rows, dims[0], integer=False)
    desc, (_, params) = _net(dims, act, layers)
    with _Backend(backend):
        y = _forward(desc, params, torch.from_numpy(x).cuda())
    h, e = x.astype(np.float64), np.zeros((rows, dims[0]))
    for l, (W, b) in enumerate(layers):
        W64, b64 = np.abs(W.astype(np.float64)), np.abs(b.astype(np.float64))
        pre = h @ W.astype(np.float64).T + b.astype(np.float64)
        e = gemm_bound(backend, dims[l], (np.abs(h) + e) @ W64.T + b64) + e @ W64.T
        if l + 1 < len(layers):
            h = act64(pre, act)
            e = e + (TANH_ABS if act == "tanh" else 2 * U * (np.abs(h) + e) if act == "leaky_relu" else 0.0)
        else:
            h = pre
    err = np.abs(y - h)
    assert (err <= e).all(), f"max err/bound {np.max(err / e):.3f}"
    return float(np.max(err / e))


# ---- GPU: softmax -------------------------------------------------------------------------------------------------
def _softmax_rows(n, rows, rng):
    """x for a [3, n] net whose logits are a*w0 (ordinary rows), c (all equal), 0.01*w0 + 1000*onehot (one dominant
    logit, the others underflow to exactly 0), and a*w0 + 1e4 (offset rows)."""
    block = 128 if n <= 64 else 8
    x = np.zeros((rows, 3), np.float32)
    x[:, 0] = rng.standard_normal(rows) * 2
    special = {0: "equal", block - 1: "dominant", block: "offset", rows - 1: "dominant"}
    for r, kind in special.items():
        if r >= rows:
            continue
        if kind == "equal":
            x[r] = (0.0, 0.0, 3.0)
        elif kind == "dominant":
            x[r] = (0.01, 1.0, 0.0)
        else:
            x[r, 2] = 1e4
    W = np.zeros((n, 3), np.float32)
    W[:, 0] = rng.standard_normal(n) * 3
    W[n // 2, 1] = 1000.0
    W[:, 2] = 1.0
    return x, [(W, np.zeros(n, np.float32))], special


@pytest.mark.gpu
@pytest.mark.parametrize("n,rows", SOFTMAX_CASES,
                         ids=[f"{'narrow' if n <= 64 else 'wide'}-n{n}-rows{rows}" for n, rows in SOFTMAX_CASES])
def test_softmax_vs_float64(n, rows):
    _check_softmax(n, rows)


def _check_softmax(n, rows):
    rng = np.random.default_rng(n + rows)
    x, layers, special = _softmax_rows(n, rows, rng)
    desc, (_, params) = _net([3, n], "identity", layers)
    xd = torch.from_numpy(x).cuda()
    logits = _forward(desc, params, xd)
    probs = _forward(desc, params, xd, softmax=True)
    ref = softmax64(logits)
    l64 = logits.astype(np.float64)
    d = np.abs(l64 - l64.max(-1, keepdims=True))
    n_add = n - 1 if n <= 64 else cdiv(n, 32) + 5
    sum_rel = (n_add + 4) * U + U * (ref * d).sum(-1, keepdims=True)
    bound = (U * d + 4 * U + sum_rel + U) * ref + 2.0 ** -126
    err = np.abs(probs - ref)
    assert (err <= bound).all(), f"max err/bound {np.max(err / bound):.3f}"
    for r, kind in special.items():
        if r >= rows:
            continue
        if kind == "equal":
            assert np.allclose(probs[r], 1.0 / n, rtol=4 * U * (n_add + 4), atol=0)
        elif kind == "dominant" and n > 1:
            assert probs[r, n // 2] == 1.0 and np.count_nonzero(probs[r]) == 1
    assert np.isfinite(probs).all()
    return float(np.max(err / bound))


# ---- GPU: clip + Adam ---------------------------------------------------------------------------------------------
HP_BASE = dict(LR=3e-4, GRAD_CLIP=0.5, BETA1=0.9, BETA2=0.999, ADAM_EPS=1e-5, INV_WORLD=1.0)


class AdamRun:
    """Device buffers of one parameter set and its own zeroed optimizer workspace (the beta-power cache lives there)."""

    def __init__(self, n_total, n_actor, rng, workspace=None, t0=0, moments=False):
        self.n, self.na = n_total, n_actor
        self.p = torch.from_numpy(rng.standard_normal(n_total).astype(np.float32)).cuda()
        m = rng.standard_normal(n_total).astype(np.float32) * 0.01 if moments else np.zeros(n_total, np.float32)
        v = np.square(rng.standard_normal(n_total)).astype(np.float32) * 1e-4 if moments else np.zeros(n_total, np.float32)
        self.m, self.v = torch.from_numpy(m).cuda(), torch.from_numpy(v).cuda()
        self.step = torch.full((1,), t0, dtype=torch.int64, device="cuda")
        self.ws = workspace if workspace is not None else torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")

    def state(self):
        return self.p.cpu().numpy(), self.m.cpu().numpy(), self.v.cpu().numpy(), int(self.step.item())

    def launch(self, g, hp):
        from ppo_and_friends_b200 import _lib
        from ppo_and_friends_b200._lib import HP, check, ptr, stream_ptr
        h = torch.zeros(HP["COUNT"], dtype=torch.float64)
        for k, val in hp.items():
            h[HP[k]] = val
        hd, gd = h.cuda(), torch.from_numpy(np.ascontiguousarray(g, np.float32)).cuda()
        check(_lib.load().ppoaf_clip_adam_step(ptr(self.p), ptr(gd), ptr(self.m), ptr(self.v), ptr(self.step), ptr(hd),
                                               self.na, self.n - self.na, ptr(self.ws), self.ws.numel(), stream_ptr()),
              "ppoaf_clip_adam_step")
        torch.cuda.synchronize()

    def step_and_check(self, g, hp, nan_ok=False):
        """One kernel step checked against adam_step64 from the kernel's own state before it; returns the coefficients
        and the worst error / bound ratio."""
        p0, m0, v0, t0 = self.state()
        self.launch(g, hp)
        p1, m1, v1, t1 = self.state()
        assert t1 == t0 + 1
        rp, rm, rv, coefs, bnd = adam_step64(p0, g, m0, v0, t0 + 1, hp, self.na)
        worst = 0.0
        for name, got, ref in (("p", p1, rp), ("m", m1, rm), ("v", v1, rv)):
            nan_ref = np.isnan(ref)
            assert np.array_equal(np.isnan(got), nan_ref), f"{name}: NaN pattern differs"
            ok = ~nan_ref
            if not nan_ok:
                assert ok.all()
            err = np.abs(got[ok].astype(np.float64) - ref[ok])
            b = bnd[name][ok]
            assert (err <= b).all(), f"{name}: max err {err.max():.3e}, max err/bound {np.max(err / np.maximum(b, 1e-300)):.3f}"
            if err.size:
                worst = max(worst, float(np.max(np.divide(err, b, out=np.zeros_like(err), where=b > 0))))
        return coefs, worst


def _grads(rng, n, na, actor_scale, critic_scale):
    g = rng.standard_normal(n)
    g[:na] *= actor_scale
    g[na:] *= critic_scale
    return g.astype(np.float32)


def _scale_for(norm_target, count):
    """Per-element scale that gives a network of `count` normal entries about this norm."""
    return norm_target / math.sqrt(max(count, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("case", adam_cases(), ids=adam_id)
def test_clip_adam_plans(case):
    """Two steps from zero moments on every plan: the first shows the clip coefficient directly
    (m = (1 - b1) coef g), the second runs from the kernel's own state; adam_step advances by one each time (the second
    call on a multi-CTA grid needs the ticket reset)."""
    sm = _sm_count()
    nv = resolve(case[0], sm)
    na = resolve_split(nv, case[1], sm)
    n, n_a = 4 * nv, 4 * na
    rng = np.random.default_rng(nv + na)
    run = AdamRun(n, n_a, rng)
    hp = dict(HP_BASE)
    # actor clipped (norm ~ 4 x 0.5), critic not (norm ~ 0.1)
    g = _grads(rng, n, n_a, _scale_for(2.0, n_a), _scale_for(0.1, n - n_a))
    coefs, _ = run.step_and_check(g, hp)
    _, m1, _, _ = run.state()
    w1 = f32(1 - hp["BETA1"])
    nz = g != 0
    observed = m1[nz].astype(np.float64) / (w1 * g[nz].astype(np.float64))
    expect = np.where(np.arange(n)[nz] < n_a, coefs[0], coefs[1])
    assert np.all(np.abs(observed - expect) <= 11 * U * expect)
    if n_a:
        assert coefs[0] < 0.5
    if n - n_a:
        assert coefs[1] == 1.0
    g2 = _grads(rng, n, n_a, _scale_for(0.2, n_a), _scale_for(3.0, n - n_a))
    run.step_and_check(g2, hp)
    assert run.state()[3] == 2


def _mid_run(rng, **kw):
    sm = _sm_count()
    nv = 1024 * sm + 1
    return AdamRun(4 * nv, 4 * (nv // 3), rng, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("clip", [-1.0, 0.0, "actor-only"])
@pytest.mark.parametrize("inv_world", [1.0, 0.5, 0.125])
def test_clip_adam_clip_and_world_scale(clip, inv_world):
    rng = np.random.default_rng(int(inv_world * 8) + (3 if clip == "actor-only" else int(clip) + 1))
    run = _mid_run(rng)
    hp = dict(HP_BASE, INV_WORLD=inv_world, GRAD_CLIP=0.5 if clip == "actor-only" else clip)
    for t in range(3):
        # summed gradients of 1 / inv_world ranks: actor norm ~ 3 (binding), critic ~ 0.05 (not), after averaging
        g = _grads(rng, run.n, run.na, _scale_for(3.0 / inv_world, run.na), _scale_for(0.05 / inv_world, run.n - run.na))
        coefs, _ = run.step_and_check(g, hp)
        if clip == -1.0:
            assert coefs == [1.0, 1.0]
        elif clip == 0.0:
            assert coefs == [0.0, 0.0]
        else:
            assert coefs[0] < 0.25 and coefs[1] == 1.0
    if clip == 0.0:             # zero coefficient: the moments decay, no gradient enters them
        _, m, v, _ = run.state()
        assert not m.any() and not v.any()


@pytest.mark.gpu
def test_clip_adam_lr_changes_between_steps():
    rng = np.random.default_rng(5)
    run = _mid_run(rng)
    for t, lr in enumerate((3e-4, 1e-3, 1e-4, 2.5e-4)):
        g = _grads(rng, run.n, run.na, _scale_for(2.0, run.na), _scale_for(0.1, run.n - run.na))
        run.step_and_check(g, dict(HP_BASE, LR=lr))


@pytest.mark.gpu
def test_clip_adam_resume_at_large_step_with_empty_cache():
    """adam_step restored as 10^4 with a fresh workspace: beta^t from pow(), moments carried in."""
    rng = np.random.default_rng(6)
    run = _mid_run(rng, t0=10 ** 4, moments=True)
    for _ in range(3):
        g = _grads(rng, run.n, run.na, _scale_for(2.0, run.na), _scale_for(0.1, run.n - run.na))
        run.step_and_check(g, HP_BASE)
    assert run.state()[3] == 10 ** 4 + 3


@pytest.mark.gpu
def test_clip_adam_betas_change_between_steps():
    """torch's Adam uses the current betas with beta^t of the step count; a cache of beta^(t-1) built under the old
    betas must not be chained with the new ones."""
    rng = np.random.default_rng(7)
    run = _mid_run(rng)
    hp = dict(HP_BASE)
    for t in range(1, 8):
        if t == 4:
            hp.update(BETA1=0.5, BETA2=0.9)
        if t == 6:
            hp.update(BETA1=0.8, BETA2=0.99)
        g = _grads(rng, run.n, run.na, _scale_for(2.0, run.na), _scale_for(0.1, run.n - run.na))
        run.step_and_check(g, hp)


@pytest.mark.gpu
def test_clip_adam_two_parameter_sets_share_a_workspace():
    """Interleaved steps of two parameter sets with different betas on one workspace (as every caller of
    ops.clip_adam_step does): each must see its own beta^t."""
    rng = np.random.default_rng(8)
    a = _mid_run(rng)
    b = AdamRun(4 * 1027, 4 * 300, rng, workspace=a.ws)
    hp_a, hp_b = dict(HP_BASE), dict(HP_BASE, BETA1=0.8, BETA2=0.99)
    for _ in range(4):
        for run, hp in ((a, hp_a), (b, hp_b)):
            g = _grads(rng, run.n, run.na, _scale_for(2.0, run.na), _scale_for(0.1, run.n - run.na))
            run.step_and_check(g, hp)


def _torch_trajectory(run, grads_hps):
    """The same steps through torch clip_grad_norm_ + Adam(foreach=False) in float32 from the run's initial state."""
    p0 = run.p.cpu()
    ta, tc = p0[:run.na].clone().requires_grad_(True), p0[run.na:].clone().requires_grad_(True)
    hp0 = grads_hps[0][1]
    opts = [torch.optim.Adam([t], lr=hp0["LR"], eps=hp0["ADAM_EPS"], betas=(hp0["BETA1"], hp0["BETA2"]), foreach=False)
            for t in (ta, tc)]
    for g, hp in grads_hps:
        for o in opts:
            o.param_groups[0]["betas"] = (hp["BETA1"], hp["BETA2"])
            o.param_groups[0]["lr"] = hp["LR"]
        gt = torch.from_numpy(g) * hp["INV_WORLD"]
        _torch_step([ta, tc], [gt[:run.na], gt[run.na:]], opts, hp["GRAD_CLIP"])
    return torch.cat([ta.detach(), tc.detach()]).numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("nv", [(0, 1025), (2048, 1)], ids=sym)
@pytest.mark.parametrize("betas_change", [False, True])
def test_clip_adam_trajectory_vs_torch(nv, betas_change):
    sm = _sm_count()
    n = 4 * resolve(nv, sm)
    rng = np.random.default_rng(n)
    run = AdamRun(n, 4 * (n // 8), rng)
    steps = []
    for t in range(15):
        hp = dict(HP_BASE, BETA1=0.5, BETA2=0.9) if betas_change and t >= 7 else dict(HP_BASE)
        scale = 3.0 if t % 2 == 0 else 0.01
        g = (rng.standard_normal(n) * scale).astype(np.float32)
        run.launch(g, hp)
        steps.append((g, hp))
    assert run.state()[3] == 15
    init = AdamRun(n, 4 * (n // 8), np.random.default_rng(n))     # the same initial parameters
    ref = _torch_trajectory(init, steps)
    np.testing.assert_allclose(run.p.cpu().numpy(), ref, rtol=2e-6, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("clip", [0.5, -1.0], ids=["clip-on", "clip-off"])
def test_clip_adam_nan_gradient(clip):
    """torch clip_grad_norm_: a NaN norm gives a NaN coefficient, so with clipping on every parameter of that network
    goes NaN and the other network is untouched; with clipping off only the NaN element's parameter does."""
    rng = np.random.default_rng(9)
    run = _mid_run(rng)
    hp = dict(HP_BASE, GRAD_CLIP=clip)
    g = _grads(rng, run.n, run.na, _scale_for(2.0, run.na), _scale_for(0.1, run.n - run.na))
    g[run.na // 2] = np.nan
    coefs, _ = run.step_and_check(g, hp, nan_ok=True)
    p, m, v, _ = run.state()
    if clip >= 0:
        assert math.isnan(coefs[0])
        assert np.isnan(p[:run.na]).all() and np.isnan(m[:run.na]).all() and np.isnan(v[:run.na]).all()
    else:
        assert np.flatnonzero(np.isnan(p)).tolist() == [run.na // 2]
    assert np.isfinite(p[run.na:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("value", [np.inf, 1e20], ids=["inf", "1e20"])
def test_clip_adam_nonfinite_norm_matches_torch(value):
    """Pinned cases that already match torch: an Inf element gives an Inf norm and a zero coefficient (the Inf entry
    becomes NaN, the others 0); a 1e20 element's square overflows float32 in both, with the same result."""
    rng = np.random.default_rng(10)
    n, na = 4 * 3001, 4 * 1000
    run = AdamRun(n, na, rng)
    init = AdamRun(n, na, np.random.default_rng(10))
    g = _grads(rng, n, na, _scale_for(2.0, na), _scale_for(0.1, n - na))
    g[17] = value
    coefs, _ = run.step_and_check(g, HP_BASE, nan_ok=True)
    assert coefs[0] == 0.0
    ref = _torch_trajectory(init, [(g, HP_BASE)])
    got = run.p.cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    np.testing.assert_allclose(got, ref, rtol=2e-6, atol=1e-7)


# ---- GPU: both step engines after a betas change ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["chain", "fused"])
def test_update_engines_after_betas_change(engine, monkeypatch):
    """Train one iteration, change pol.actor_optim's betas, train again: the launch chain and the fused step kernel
    must both agree with the oracle run with the same betas."""
    from helpers import make_policy, run_device_rollout
    from oracle.update import OracleUpdater
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    from ppo_and_friends_b200.synthetic import make_rollout
    monkeypatch.setenv("PPOAF_STEP", engine)
    ro = make_rollout(seed=3, T=48, E=8, obs_dim=8, act_dim=2, max_ts_per_ep=16, obs_scale=False)
    torch.manual_seed(0)
    pol = make_policy(ro, act="leaky_relu", actor_hidden=64, critic_hidden=64, lr=3e-4)
    ds = run_device_rollout(pol, ro)
    host = {k: getattr(ds, k).cpu().numpy().copy() for k in
            ("critic_observations", "observations", "raw_actions", "advantages", "log_probs", "rewards_to_go", "values")}
    oracle = OracleUpdater({k: v.cpu().numpy() for k, v in pol.actor.state_dict().items()},
                           {k: v.cpu().numpy() for k, v in pol.critic.state_dict().items()}, "leaky_relu", False)
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    for it, betas in enumerate(((0.9, 0.999), (0.5, 0.9))):
        pol.actor_optim.param_groups[0]["betas"] = betas
        oracle.betas = betas
        torch.manual_seed(1 + it)
        ppo_batch_train(state, _Loader(ds, 128), "pol")
        assert pol._engine.fused == (engine == "fused")
        oracle.batch_train([host], [pol._engine._perm_dev.cpu().numpy()], 128)
    ref = oracle.state()
    for net, obj in (("actor", pol.actor), ("critic", pol.critic)):
        for k, v in obj.state_dict().items():
            np.testing.assert_allclose(v.cpu().numpy(), ref[f"{net}/param/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
