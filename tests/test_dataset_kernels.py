"""
The dataset-build kernels (csrc/gather.cu, csrc/segscan.cu), each through `ops` or the C ABI against an exact or float64
restatement of the reference, at the launch plans the host code picks among:

  gather_rows      bit-exact against numpy fancy indexing over the raw bytes (NaN payloads included); bytes around the
                   destination rows stay untouched.
  build_flat_map   src_row and seg_flag bit-exact against a numpy restatement; entries around the outputs untouched.
  gae_rtg_segscan  |got - ref| <= 2^-24 |ref| + 2^-30 S, where ref is the float64 reference (oracle/segments.py:
                   segment_returns) and S the same discounted sum over absolute values (slack for the kernel's fp64
                   reassociation); a second launch is bit-identical.  A NaN or Inf in a reward, in a value at a segment's
                   first step or in a bootstrap value stays inside its own segment: the kernel's NaN positions equal the
                   reference's, and so do its non-finite positions.

`gather_plan`, `scan_plan_id` and the grid formulas below restate the host-side plan selection of gather.cu and
segscan.cu.  They only choose sizes and place segment ends at plan boundaries and name the cases; no result is compared
with anything they compute, so if they drift from the C code the placement weakens but no comparison becomes wrong.
"""
import ctypes as C

import numpy as np
import pytest
import torch

U32 = 2.0 ** -24
SLACK = 2.0 ** -30

# ---- restated launch plans (gather.cu: launch_gather; segscan.cu: ppoaf_build_flat_map, ppoaf_gae_rtg_segscan) -----
GATHER_THREADS, GATHER_CAP_PER_SM = 256, 8          # grid <= 8 * SMs CTAs of 256 threads
FLAT_MAP_THREADS, FLAT_MAP_CAP_PER_SM = 256, 16     # one warp per segment, grid <= 16 * SMs CTAs
SCAN_TILE, SCAN_ITEMS, SCAN_WARP = 1024, 8, 256     # 128 threads x 8 items per tile; a warp covers 256 items
MAX_CTAS_PER_SM = 16                                # 2048 threads / 128: no resident grid of the scan exceeds 16 * SMs


def gather_plan(row_bytes, stride_bytes, src_off, dst_off):
    """Vector width in bytes: the widest of 16/8/4/1 that divides both base addresses, the row and the stride."""
    al = src_off | dst_off | row_bytes | (stride_bytes or row_bytes)
    return next(w for w in (16, 8, 4, 1) if al % w == 0)


def scan_plan_id(n):
    """Tiles of the scan for n steps that are not persistent (every tile has its own CTA)."""
    tiles, last = -(-n // SCAN_TILE), n % SCAN_TILE
    if tiles == 1 and last:
        return f"one-ragged-tile-{last}"
    return f"{tiles}-tiles-" + (f"ragged-tile-{last}" if last else "full-last-tile-no-halo")


# ---- cases --------------------------------------------------------------------------------------------------------
PERSISTENT_FULL = -2        # n derived from the SM count: more tiles than any resident grid, full last tile
PERSISTENT_RAGGED = -3      # the same with a ragged last tile of one element
FLAT_MAP_CAPPED = -4        # segment count derived from the SM count so that the flat-map grid is capped

GATHER_GEOMETRIES = [       # (row_bytes, src_stride_bytes (0 = row), src field offset, destination offset)
    (16, 48, 16, 0), (1504, 1600, 32, 0),                       # 16-byte vectors
    (16, 0, 0, 8), (8, 24, 8, 0), (1504, 1512, 8, 0),           # 8-byte: misaligned destination, 8-byte rows
    (12, 20, 4, 0), (4, 12, 4, 0), (16, 20, 0, 0),              # 4-byte: the stride demotes a 16-byte row
    (3, 7, 1, 0), (1, 5, 3, 0), (1504, 1505, 3, 1),             # bytes
]
GATHER_CASES = ([(g, idx, pat) for g in GATHER_GEOMETRIES for idx in (32, 64)
                 for pat in ("random-repeats", "reversed", "one-row")]
                + [(g, idx, "grid-stride") for g in ((16, 48, 16, 0), (8, 24, 8, 0), (4, 12, 4, 0), (3, 7, 1, 0))
                   for idx in (32, 64)])


def _gather_id(c):
    (row, stride, src_off, dst_off), idx, pat = c
    return f"vec{gather_plan(row, stride, src_off, dst_off)}-idx{idx}-row{row}-stride{stride or row}-off{src_off}" \
           f"-dst{dst_off}-{pat}"


FLAT_MAP_CASES = [(lens, n_cols) for lens in ("len1", "len31", "len32", "len33", "len1000", "mixed", FLAT_MAP_CAPPED)
                  for n_cols in (1, 4099)]


def _flat_map_id(c):
    lens, n_cols = c
    return f"{'grid-capped' if lens == FLAT_MAP_CAPPED else lens}-cols{n_cols}"


GL_PAIRS = [(0.99, 0.95), (1.0, 1.0), (0.99, 0.0), (0.0, 0.95)]
EDGES_N = 16 * SCAN_TILE + 100
SCAN_CASES = (
    [("random40", n, 0.99, 0.95, True) for n in (1, 7, 1023, 1024, 1025, 2048, 2049)]
    + [("random40", n, 0.99, 0.95, False) for n in (7, 1025, 2049)]
    + [("edges", EDGES_N, g, lam, gae) for g, lam in GL_PAIRS + [(0.5, 0.5)] for gae in (True, False)]
    + [("random300", 50_001, g, lam, gae) for g, lam in GL_PAIRS for gae in (True, False)]
    + [("one-segment", 5000, 0.99, 0.95, True), ("one-segment", 5000, 1.0, 1.0, False),
       ("one-segment", PERSISTENT_RAGGED, 0.99, 0.95, True)]
    + [("all-length-1", 5000, 0.99, 0.95, True), ("all-length-1", PERSISTENT_FULL, 0.99, 0.95, True)]
    + [("random64", PERSISTENT_FULL, 0.99, 0.95, True), ("random64", PERSISTENT_RAGGED, 0.99, 0.95, False),
       ("random64", PERSISTENT_RAGGED, 1.0, 1.0, True), ("edges", PERSISTENT_FULL, 0.99, 0.95, True)]
    + [("long2000", 10_000, 0.5, 0.5, gae) for gae in (True, False)]
)


def _scan_id(c):
    layout, n, g, lam, gae = c
    size = {PERSISTENT_FULL: "persistent-2plus-tiles-full", PERSISTENT_RAGGED: "persistent-2plus-tiles-ragged-tile-1"}
    return f"{size.get(n) or scan_plan_id(n)}-{layout}-g{g}-l{lam}-{'gae' if gae else 'nogae'}"


PLANT_KINDS = ("reward", "value-at-first-step", "v_boot")
PLANT_CASES = ([("edges", EDGES_N, kind, val, g, lam, gae) for kind in PLANT_KINDS for val in ("nan", "inf", "-inf")
                for g, lam in GL_PAIRS + [(0.5, 0.5)] for gae in (True, False)
                if gae or kind != "v_boot"]                  # without GAE the bootstrap value is not read
               + [("edges", PERSISTENT_RAGGED, kind, "nan", 0.99, 0.95, True) for kind in PLANT_KINDS])


def _plant_id(c):
    layout, n, kind, val, g, lam, gae = c
    return f"{_scan_id((layout, n, g, lam, gae))}-{val}-in-{kind}"


def test_case_tables_reach_every_launch_plan():
    """(CPU) the parametrisations cover every plan the host code can pick and every edge the scan has."""
    plans = {(gather_plan(*g), idx) for g, idx, _ in GATHER_CASES}
    assert plans == {(w, i) for w in (16, 8, 4, 1) for i in (32, 64)}
    assert {gather_plan(*g) for g, _, pat in GATHER_CASES if pat == "grid-stride"} == {16, 8, 4, 1}
    assert {g[0] for g in GATHER_GEOMETRIES} >= {1, 3, 4, 8, 12, 16, 1504}
    assert any(g[1] > g[0] and g[2] for g in GATHER_GEOMETRIES if gather_plan(*g) == 16)
    assert {lens for lens, _ in FLAT_MAP_CASES} >= {"len1", "len31", "len32", "len33", "len1000", FLAT_MAP_CAPPED}
    ids = [_scan_id(c) for c in SCAN_CASES]
    for want in ("one-ragged-tile-1", "one-ragged-tile-7", "one-ragged-tile-1023", "1-tiles-full-last-tile-no-halo",
                 "2-tiles-ragged-tile-1", "2-tiles-full-last-tile-no-halo", "3-tiles-ragged-tile-1",
                 "persistent-2plus-tiles-full", "persistent-2plus-tiles-ragged-tile-1"):
        assert any(i.startswith(want + "-") for i in ids), want
    assert {(g, lam) for _, _, g, lam, _ in SCAN_CASES} >= set(GL_PAIRS) | {(0.5, 0.5)}
    assert {(layout, gae) for layout, *_, gae in SCAN_CASES} >= {("edges", True), ("edges", False)}
    assert {layout for layout, n, *_ in SCAN_CASES if n == PERSISTENT_RAGGED} >= {"one-segment", "random64"}
    # the edge layout puts segment ends at a tile's first and last element, on both sides of thread and warp edges, and
    # leaves a tile without an end
    ends = np.flatnonzero(_edge_ends(EDGES_N))
    assert {0, SCAN_TILE - 1} <= set(ends % SCAN_TILE)
    assert {SCAN_WARP - 1, 0} <= set(ends % SCAN_WARP) and {SCAN_ITEMS - 1, 0} <= set(ends % SCAN_ITEMS)
    assert set(range(-(-EDGES_N // SCAN_TILE))) - set(ends // SCAN_TILE)
    lens = np.diff(np.concatenate([[-1], ends]))
    assert lens.max() > SCAN_TILE and (0.25 ** np.arange(lens.max()))[-1] == 0.0  # (gamma lambda)^k underflows inside
    # every plant kind lands on a tile, a warp and a thread edge
    lens = _lens_from_ends(_edge_ends(EDGES_N))
    for kind in PLANT_KINDS:
        pos = _plant_positions(lens, kind)
        edge = pos if kind != "v_boot" else np.cumsum(lens)[pos] - 1
        for mod in (SCAN_TILE, SCAN_WARP, SCAN_ITEMS):          # a value planted at a first step: one side suffices
            assert any(edge % mod == 0) and (kind == "value-at-first-step" or any(edge % mod == mod - 1)), (kind, mod)


# ---- float64 reference --------------------------------------------------------------------------------------------
def _sweep(x, lens, g, seed):
    """out[i] = x[i] + g * out[i + 1] inside a segment and x[end] + g * seed[s] at its last element, in float64 and in
    the order of oracle.segments.discounted_sums.  One vectorised step per distance from the segment ends; the last few
    long segments finish in a scalar loop."""
    x = np.asarray(x, dtype=np.float64)
    lens = np.asarray(lens, dtype=np.int64)
    g = float(g)
    ends = np.cumsum(lens) - 1
    out = np.empty(len(x))
    out[ends] = x[ends] + g * np.asarray(seed, dtype=np.float64)
    act_end, act_len = ends, lens
    d = 1
    while act_end.size:
        keep = act_len > d
        act_end, act_len = act_end[keep], act_len[keep]
        if act_end.size <= 4:
            for e, L in zip(act_end.tolist(), act_len.tolist()):
                lo, hi = e - L + 1, e - d + 1
                xs, acc = x[lo:hi].tolist(), float(out[hi])
                res = [0.0] * len(xs)
                for i in range(len(xs) - 1, -1, -1):
                    acc = xs[i] + g * acc
                    res[i] = acc
                out[lo:hi] = res
            break
        p = act_end - d
        out[p] = x[p] + g * out[p + 1]
        d += 1
    return out


def segscan_reference(rewards, values, lens, v_boot, r_boot, gamma, lambd, use_gae):
    """(adv, rtg, S_adv, S_rtg) in float64: the flat restatement of segment_returns and the same sums over |terms|."""
    with np.errstate(invalid="ignore", over="ignore"):
        return _segscan_reference(rewards, values, lens, v_boot, r_boot, gamma, lambd, use_gae)


def _segscan_reference(rewards, values, lens, v_boot, r_boot, gamma, lambd, use_gae):
    lens = np.asarray(lens, dtype=np.int64)
    ends = np.cumsum(lens) - 1
    r64 = rewards.astype(np.float64)
    rb = r_boot.astype(np.float64) + 0.0            # the reference's accumulator starts at 0.0 + r_boot
    rtg = _sweep(r64, lens, gamma, rb)
    s_rtg = _sweep(np.abs(r64), lens, gamma, np.abs(rb))
    v64 = values.astype(np.float64)
    if use_gae:
        vnext = np.empty_like(values)
        vnext[:-1] = values[1:]
        vnext[ends] = v_boot
        gv = (np.float32(gamma) * vnext).astype(np.float32)
        delta = r64 + gv.astype(np.float64) - v64
        zero = np.zeros(len(lens))
        adv = _sweep(delta, lens, gamma * lambd, zero)
        s_adv = _sweep(np.abs(delta), lens, gamma * lambd, zero)
    else:
        adv = rtg - v64
        s_adv = s_rtg + np.abs(v64)
    return adv, rtg, s_adv, s_rtg


# ---- inputs -------------------------------------------------------------------------------------------------------
def _lens_from_ends(end_mask):
    ends = np.flatnonzero(end_mask)
    return np.diff(np.concatenate([[-1], ends])).astype(np.int64)


def _edge_ends(n):
    """Segment ends by tile, cycling four patterns: a tile's last element and a thread edge; a tile's first element and
    both sides of two warp edges; no end at all; both sides of three thread edges and of a warp edge."""
    end = np.zeros(n, dtype=bool)
    for t in range(-(-n // SCAN_TILE)):
        b = t * SCAN_TILE
        pattern = {0: [SCAN_TILE - 1, 8 * 3 - 1, 8 * 3],
                   1: [0, SCAN_WARP - 1, SCAN_WARP, 3 * SCAN_WARP - 1, 3 * SCAN_WARP],
                   2: [],
                   3: [8 - 1, 8, 8 * 17 - 1, 8 * 17, 8 * 100 - 1, 8 * 100, 2 * SCAN_WARP - 1, 2 * SCAN_WARP]}[t % 4]
        for k in pattern:
            if b + k < n:
                end[b + k] = True
    end[n - 1] = True
    return end


def _cut(lens, n):
    """The leading segments of `lens` that cover exactly n steps (the last one shortened)."""
    c = np.cumsum(lens)
    k = int(np.searchsorted(c, n))
    lens = np.array(lens[:k + 1], dtype=np.int64)
    lens[-1] -= int(c[k] - n)
    return lens


def _random_lens(rng, n, max_len):
    return _cut(rng.integers(1, max_len + 1, size=n // max(1, (max_len + 1) // 2) + 16), n)


def _scan_n(n, sm):
    tiles = MAX_CTAS_PER_SM * sm + 3
    if n == PERSISTENT_FULL:
        return tiles * SCAN_TILE
    if n == PERSISTENT_RAGGED:
        return (tiles - 1) * SCAN_TILE + 1
    return n


def _layout(layout, n, rng):
    if layout.startswith("random"):
        return _random_lens(rng, n, int(layout[len("random"):]))
    if layout == "edges":
        return _lens_from_ends(_edge_ends(n))
    if layout == "one-segment":
        return np.array([n], dtype=np.int64)
    if layout == "all-length-1":
        return np.ones(n, dtype=np.int64)
    if layout == "long2000":                         # 2000-step segments starting mid-tile, short ones between
        return _cut([37, 2000, 5] * (n // 2042 + 1), n)
    raise ValueError(layout)


def _scan_inputs(rng, lens):
    n, n_seg = int(lens.sum()), len(lens)
    rewards = rng.standard_normal(n).astype(np.float32)
    values = rng.standard_normal(n).astype(np.float32)
    terminal = rng.random(n_seg) < 0.5
    v_boot = np.where(terminal, 0.0, rng.standard_normal(n_seg) * 3).astype(np.float32)
    r_boot = np.clip(v_boot, -2.0, 2.0).astype(np.float32)
    return rewards, values, terminal, v_boot, r_boot


def _plant_positions(lens, kind):
    """Where a non-finite value goes, at most one per segment: for rewards, positions at a tile's first and last element
    and on both sides of warp and thread edges (the tile-first one inside a segment that spans a tile without an end);
    for values, the first step of segments that start at such edges; for bootstrap values, segments that end there.
    Positions (segment indices for v_boot) are returned sorted."""
    off = np.concatenate([[0], np.cumsum(lens)])
    n = int(off[-1])
    seg_of = np.repeat(np.arange(len(lens)), lens)
    if kind == "reward":
        cand = [3 * SCAN_TILE, 4 * SCAN_TILE + SCAN_TILE - 1, 5 * SCAN_TILE + SCAN_WARP - 1, 9 * SCAN_TILE + SCAN_WARP,
                8 * SCAN_TILE + 8 * 3 - 1, 11 * SCAN_TILE + 8 * 17, 7 * SCAN_TILE + 8 * 50]
        chosen, used = [], set()
        for p in cand:
            if p < n and seg_of[p] not in used:
                chosen.append(p)
                used.add(seg_of[p])
        return np.array(sorted(chosen), dtype=np.int64)
    starts, ends = off[:-1], off[1:] - 1
    pick = starts if kind == "value-at-first-step" else ends
    chosen = []
    for mod, r in ((SCAN_TILE, 0), (SCAN_TILE, SCAN_TILE - 1), (SCAN_WARP, 0), (SCAN_WARP, SCAN_WARP - 1),
                   (SCAN_ITEMS, 0), (SCAN_ITEMS, SCAN_ITEMS - 1)):
        hits = np.flatnonzero((pick % mod == r) & (pick > 2 * SCAN_TILE))
        hits = [h for h in hits if h not in chosen and all(abs(int(pick[h]) - int(pick[c])) > 600 for c in chosen)]
        if hits:
            chosen.append(hits[len(hits) // 2])
    segs = np.array(sorted(chosen), dtype=np.int64)
    return segs if kind == "v_boot" else starts[segs]


def test_sweep_reference_restates_the_oracle():
    """(CPU) the vectorised float64 reference equals oracle.segments.flat_segscan_reference bit for bit (NaN positions
    included) on small inputs, for every (gamma, lambda) and both advantage kinds, with and without planted NaN/Inf."""
    from oracle.segments import flat_segscan_reference
    rng = np.random.default_rng(7)
    for trial in range(6):
        lens = _random_lens(rng, 2000, [1, 8, 40, 300, 2000, 64][trial])
        rewards, values, _, v_boot, r_boot = _scan_inputs(rng, lens)
        v_boot[0] = -0.0
        r_boot[0] = -0.0
        if trial >= 2:
            bad = [np.nan, np.inf, -np.inf][trial % 3]
            rewards[rng.integers(0, len(rewards), 3)] = bad
            values[np.concatenate([[0], np.cumsum(lens)[:-1]])[rng.integers(0, len(lens), 2)]] = bad
            v_boot[rng.integers(0, len(lens), 2)] = bad
        for g, lam in GL_PAIRS + [(0.5, 0.5)]:
            for gae in (True, False):
                adv, rtg, *_ = segscan_reference(rewards, values, lens, v_boot, r_boot, g, lam, gae)
                with np.errstate(invalid="ignore", over="ignore"):
                    ref_adv, ref_rtg = flat_segscan_reference(rewards, values, lens, v_boot, r_boot, g, lam, gae)
                for got, ref in ((adv, ref_adv), (rtg, ref_rtg)):
                    assert np.array_equal(got, ref, equal_nan=True), (trial, g, lam, gae)
                    fin = np.isfinite(ref)
                    assert np.array_equal(np.signbit(got[fin]), np.signbit(ref[fin]))


def test_refused_arguments_without_gpu():
    """(CPU) argument checks that run before anything touches the device: code 1 and a message naming the problem."""
    from ppo_and_friends_b200 import _lib
    lib = _lib.load()
    for stride, row in ((7, 8), (1, 1504), (15, 16)):
        assert lib.ppoaf_gather_rows(None, stride, None, 0, None, 4, row, None) == 1
        assert b"stride smaller than the row" in lib.ppoaf_last_error()
    for row in (0, -1, -16, 1 << 31, (1 << 31) + 16):
        assert lib.ppoaf_gather_rows(None, 0, None, 1, None, 4, row, None) == 1
        assert b"bad sizes" in lib.ppoaf_last_error()
    assert lib.ppoaf_gather_rows(None, 0, None, 1, None, 0, (1 << 31) - 1, None) == 0      # the largest row, no rows
    args = (None, None, None, None, None)
    assert lib.ppoaf_build_flat_map(*args, 1, 0, 1, None, None, None) == 1                 # n_cols = 0
    assert lib.ppoaf_build_flat_map(*args, 1, 4, 1 << 31, None, None, None) == 1           # int32 ring rows
    assert b"2^31" in lib.ppoaf_last_error()


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _sm_count():
    from ppo_and_friends_b200 import ops
    return ops.device_info()["sm_count"]


def _dev(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def _bits(t):
    return t.view(torch.int32)


# ---- gather_rows --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", GATHER_CASES, ids=_gather_id)
def test_gather_rows_bit_exact(case):
    from ppo_and_friends_b200 import ops
    (row, stride, src_off, dst_off), idx_bits, pat = case
    eff_stride = stride or row
    rng = np.random.default_rng(row * 1009 + eff_stride * 31 + src_off + idx_bits)
    n_src = 257
    if pat == "random-repeats":
        idx = rng.integers(0, n_src, 1000)
        idx[:8] = idx[8]                                       # repeated rows
    elif pat == "reversed":
        idx = np.arange(n_src)[::-1]
    elif pat == "one-row":
        idx = np.array([n_src - 1])
    else:
        vpr = row // gather_plan(row, stride, src_off, dst_off)
        cap_vecs = GATHER_CAP_PER_SM * _sm_count() * GATHER_THREADS
        idx = rng.integers(0, n_src, 2 * cap_vecs // vpr + 3)
        assert len(idx) * vpr > cap_vecs
    idx = idx.astype(np.int32 if idx_bits == 32 else np.int64)
    n = len(idx)
    src = rng.integers(0, 256, src_off + n_src * eff_stride + 64, dtype=np.uint8)
    words = src[:len(src) // 4 * 4].view(np.uint32)            # NaN payloads, quiet and signalling, of either sign
    words[::97] = np.array([0x7FC12345, 0xFFA00001, 0x7F800001, 0xFFFFFFFF], dtype=np.uint32)[np.arange(len(words[::97])) % 4]
    src_d = _dev(src)
    margin = 64
    sentinel = 0xA5
    dst_buf = torch.full((margin + n * row + margin,), sentinel, dtype=torch.uint8, device="cuda")
    dst_start = margin + dst_off
    dst = dst_buf[dst_start:dst_start + n * row]
    assert src_d.data_ptr() % 16 == 0 and dst.data_ptr() % 16 == dst_off % 16
    ops.gather_rows(src_d, _dev(idx), out=dst, row_bytes=row, src_stride_bytes=stride, src_offset_bytes=src_off, n_rows=n)
    got = dst_buf.cpu().numpy()
    expect = src[src_off + idx.astype(np.int64)[:, None] * eff_stride + np.arange(row)[None, :]].reshape(-1)
    assert np.array_equal(got[dst_start:dst_start + n * row], expect)
    assert (got[:dst_start] == sentinel).all() and (got[dst_start + n * row:] == sentinel).all()


# ---- build_flat_map -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", FLAT_MAP_CASES, ids=_flat_map_id)
def test_build_flat_map_bit_exact(case):
    from ppo_and_friends_b200 import _lib
    lens_kind, n_cols = case
    rng = np.random.default_rng(n_cols + len(str(lens_kind)))
    if lens_kind == FLAT_MAP_CAPPED:
        n_seg = 2 * FLAT_MAP_CAP_PER_SM * _sm_count() * FLAT_MAP_THREADS // 32 + 5
        assert -(-n_seg * 32 // FLAT_MAP_THREADS) > FLAT_MAP_CAP_PER_SM * _sm_count()
        lens = rng.integers(1, 41, n_seg)
        lens[::997] = 1000
    elif lens_kind == "mixed":
        lens = rng.choice([1, 31, 32, 33, 64, 65, 1000], 400)
    else:
        lens = np.full(300 if lens_kind != "len1000" else 40, int(lens_kind[3:]))
    lens = lens.astype(np.int64)
    n_seg, n = len(lens), int(lens.sum())
    t_max = (2 ** 31 - 1) // n_cols - int(lens.max())
    t0 = rng.integers(0, min(t_max, 50_000), n_seg)
    t0[0] = t_max                                            # the largest source row that still fits in int32
    col = rng.integers(0, n_cols, n_seg)
    col[0] = n_cols - 1
    term = rng.random(n_seg) < 0.5
    off = np.concatenate([[0], np.cumsum(lens)])
    assert (t0[0] + lens[0]) * n_cols - 1 <= 2 ** 31 - 1

    pad = 37
    src_buf = torch.full((n + 2 * pad,), -12345, dtype=torch.int32, device="cuda")
    flag_buf = torch.full((n + 2 * pad,), 0xEE, dtype=torch.uint8, device="cuda")
    lib = _lib.load()
    i32 = lambda a: _dev(np.asarray(a, dtype=np.int32))
    ins = (i32(col), i32(t0), i32(lens), _dev(off.astype(np.int64)), _dev(term.astype(np.uint8)))
    _lib.check(lib.ppoaf_build_flat_map(*(_lib.ptr(t) for t in ins), n_seg, n_cols, n,
                                        C.c_void_p(src_buf.data_ptr() + 4 * pad), C.c_void_p(flag_buf.data_ptr() + pad),
                                        _lib.stream_ptr()), "ppoaf_build_flat_map")
    seg = np.repeat(np.arange(n_seg), lens)
    k = np.arange(n) - off[seg]
    expect_row = (t0[seg] + k) * n_cols + col[seg]
    assert expect_row.max() < 2 ** 31
    expect_flag = np.zeros(n, dtype=np.uint8)
    expect_flag[off[1:] - 1] = 1 + 2 * term.astype(np.uint8)
    got_row, got_flag = src_buf.cpu().numpy(), flag_buf.cpu().numpy()
    assert np.array_equal(got_row[pad:pad + n], expect_row.astype(np.int32))
    assert np.array_equal(got_flag[pad:pad + n], expect_flag)
    assert (got_row[:pad] == -12345).all() and (got_row[pad + n:] == -12345).all()
    assert (got_flag[:pad] == 0xEE).all() and (got_flag[pad + n:] == 0xEE).all()


# ---- gae_rtg_segscan ----------------------------------------------------------------------------------------------
def _run_scan(lens, rewards, values, terminal, v_boot, r_boot, g, lam, gae, adv_out=None, rtg_out=None):
    from ppo_and_friends_b200 import ops
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    flag = np.zeros(len(rewards), dtype=np.uint8)
    flag[off[1:] - 1] = 1 + 2 * terminal.astype(np.uint8)
    args = (_dev(rewards), _dev(values), _dev(flag), _dev(off), _dev(v_boot), _dev(r_boot), g, lam, gae)
    adv, rtg = ops.gae_rtg_segscan(*args, adv_out=adv_out, rtg_out=rtg_out)
    adv2, rtg2 = ops.gae_rtg_segscan(*args)
    assert torch.equal(_bits(adv2), _bits(adv)) and torch.equal(_bits(rtg2), _bits(rtg)), "second launch differs"
    return adv.cpu().numpy().astype(np.float64), rtg.cpu().numpy().astype(np.float64)


def _assert_bound(got, ref, s, what):
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin), f"{what}: non-finite at {np.flatnonzero(np.isfinite(got) != fin)[:10]}"
    err = np.abs(got[fin] - ref[fin])
    lim = U32 * np.abs(ref[fin]) + SLACK * s[fin]
    bad = np.flatnonzero(err > lim)
    assert bad.size == 0, f"{what}: {bad.size} over the bound, first at {np.flatnonzero(fin)[bad[0]]}: " \
                          f"got {got[fin][bad[0]]!r} ref {ref[fin][bad[0]]!r} bound {lim[bad[0]]!r}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", SCAN_CASES, ids=_scan_id)
def test_segscan_matches_float64_reference(case):
    layout, n, g, lam, gae = case
    n = _scan_n(n, _sm_count())
    rng = np.random.default_rng(n + int(100 * g) + int(10 * lam) + len(layout))
    lens = _layout(layout, n, rng)
    assert lens.sum() == n and lens.min() >= 1
    inputs = _scan_inputs(rng, lens)
    adv, rtg = _run_scan(lens, *inputs, g, lam, gae)
    ref_adv, ref_rtg, s_adv, s_rtg = segscan_reference(*inputs[:2], lens, *inputs[3:], g, lam, gae)
    assert np.isfinite(ref_adv).all() and np.isfinite(ref_rtg).all()
    _assert_bound(adv, ref_adv, s_adv, "advantages")
    _assert_bound(rtg, ref_rtg, s_rtg, "rewards-to-go")


@pytest.mark.gpu
@pytest.mark.parametrize("case", PLANT_CASES, ids=_plant_id)
def test_segscan_keeps_non_finite_values_in_their_segment(case):
    layout, n, kind, val, g, lam, gae = case
    n = _scan_n(n, _sm_count())
    rng = np.random.default_rng(n + PLANT_KINDS.index(kind))
    lens = _layout(layout, n, rng)
    rewards, values, terminal, v_boot, r_boot = _scan_inputs(rng, lens)
    pos = _plant_positions(lens, kind)
    assert pos.size >= 3
    bad = np.float32(val)
    if kind == "reward":
        rewards[pos] = bad
    elif kind == "value-at-first-step":
        values[pos] = bad
    else:
        v_boot[pos] = bad
        terminal[pos] = False
    adv, rtg = _run_scan(lens, rewards, values, terminal, v_boot, r_boot, g, lam, gae)
    with np.errstate(invalid="ignore", over="ignore"):
        ref_adv, ref_rtg, s_adv, s_rtg = segscan_reference(rewards, values, lens, v_boot, r_boot, g, lam, gae)
    for got, ref, s, what in ((adv, ref_adv, s_adv, "advantages"), (rtg, ref_rtg, s_rtg, "rewards-to-go")):
        if val == "nan":
            assert np.array_equal(np.isnan(got), np.isnan(ref)), \
                f"{what}: NaN at {np.flatnonzero(np.isnan(got) != np.isnan(ref))[:10]} differs from the reference"
        _assert_bound(got, ref, s, what)                  # same non-finite positions, finite ones within the bound
    assert not np.isfinite(ref_adv).all() and np.isfinite(ref_adv).mean() > 0.5 and np.isfinite(ref_rtg).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2049, PERSISTENT_RAGGED], ids=["3-tiles-ragged-tile-1", "persistent-2plus-tiles"])
def test_segscan_into_recalculate_advantages_buffers(n):
    """The way EpisodeInfo.recalculate_advantages calls the scan: the advantages written into the dataset's existing
    buffer with new values, the returns into a scratch buffer.  Every output element is written, nothing around them,
    and the result is the reference's for the new values."""
    n = _scan_n(n, _sm_count())
    rng = np.random.default_rng(n)
    lens = _layout("random64", n, rng)
    rewards, values, terminal, v_boot, r_boot = _scan_inputs(rng, lens)
    margin = 16                                                 # floats: keeps the outputs 16-byte aligned
    adv_buf = torch.full((n + 2 * margin,), float("nan"), device="cuda")
    rtg_buf = torch.full((n + 2 * margin,), -7.0, device="cuda")
    adv_view, rtg_view = adv_buf[margin:margin + n], rtg_buf[margin:margin + n]
    _run_scan(lens, rewards, values, terminal, v_boot, r_boot, 0.99, 0.95, True, adv_view, rtg_view)
    new_values = rng.standard_normal(n).astype(np.float32)
    scratch = torch.full((n,), float("inf"), device="cuda")
    adv, rtg = _run_scan(lens, rewards, new_values, terminal, v_boot, r_boot, 0.99, 0.95, True, adv_view, scratch)
    got_adv = adv_buf.cpu().numpy().astype(np.float64)
    assert np.array_equal(got_adv[margin:margin + n], adv)
    assert np.isnan(got_adv[:margin]).all() and np.isnan(got_adv[margin + n:]).all()
    got_rtg = rtg_buf.cpu().numpy()
    assert (got_rtg[:margin] == -7.0).all() and (got_rtg[margin + n:] == -7.0).all()
    assert np.array_equal(scratch.cpu().numpy(), got_rtg[margin:margin + n])    # returns do not depend on the values
    ref_adv, ref_rtg, s_adv, s_rtg = segscan_reference(rewards, new_values, lens, v_boot, r_boot, 0.99, 0.95, True)
    _assert_bound(adv, ref_adv, s_adv, "advantages")
    _assert_bound(rtg, ref_rtg, s_rtg, "rewards-to-go")
