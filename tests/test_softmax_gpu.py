"""Block-sparse softmax and its gradient (csrc/softmax.cuh) against a float64 reference, on every dispatch path.

bst_softmax / bst_softmax_grad pick one of two kernel families:
  * the TMA-staged kernels: 16-bit in and out, bs 32/64, rows of <= 16 key blocks (MAXE buckets 4, 8, 12, 16), 16-byte
    aligned tensors;
  * the register kernels: everything else.  A row's first KEEP (4 or 8) blocks stay in registers with an online max, the
    rest are re-read, and LUT entries past the 32nd come from global memory.
Every GPU test asserts which kernel ran (`_lib.last_kernel()`) and that no kernel faulted, and compares elementwise with
the float64 reference below, which follows the NumPy checker's semantics (masked entries are -FLT_MAX, so a fully masked
row comes out uniform).  The reference itself is pinned to the committed fixtures by a CPU test.

Tolerances are elementwise and derived in the comments next to EPS / TINY / GRAD_EPS and in `prob_bound` / `ref_grad`.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests._util import GOLDEN, ROOT, golden_files
from tests.golden.make_golden import causal_callback, checker_callback
from blocksparse_b200 import BlocksparseTransformer, _lib
from oracle.bst_oracle import TransformerOracle

FLT_MAX = float(np.finfo(np.float32).max)
BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
NAME = {BF16: "bf16", F16: "f16", F32: "f32"}
E_ARG = -3                                   # BSMM_E_ARG

# Probabilities, relative part.  16-bit outputs: storing rounds by half an ulp (2^-9 bf16, 2^-12 fp16); the fp32 work
# before it (exp2f <= 2 ulp, one reciprocal, one product, the row sum) adds ~1e-6, so one full ulp bounds both.  fp32
# outputs: the same fp32 work, with the row sum's rounding growing like sqrt(n) * 2^-24 over per-lane sums of at most
# 64 blocks x 8 entries (~1.4e-6); long rows use the worst-case bound in `prob_bound` instead.
EPS = {BF16: 2.0 ** -8, F16: 2.0 ** -11, F32: 1e-5}
# Absolute floor.  fp16: one subnormal spacing (2^-24).  fp32: FLT_MIN -- below it the kernel's exp2f results are
# subnormal and keep fewer bits.  bf16: 2^-20, far below any probability that carries weight in a row.
TINY = {BF16: 2.0 ** -20, F16: 2.0 ** -24, F32: 2.0 ** -126}
# Gradient output rounding (one ulp; fp32: the three roundings of (dy - acc) * y * scale, 2^-24 each, plus margin).
GRAD_EPS = {BF16: 2.0 ** -8, F16: 2.0 ** -11, F32: 2.0 ** -22}
# (explicit significand bits, subnormal step) of each dtype, for ulp()
BITS = {BF16: (7, 2.0 ** -133), F16: (10, 2.0 ** -24), F32: (23, 2.0 ** -149)}

PAIRS = [(F16, F16), (BF16, BF16), (F16, BF16), (BF16, F16), (F32, F32), (F32, BF16), (BF16, F32)]
PAIRS16 = PAIRS[:4]
# key blocks per query row: every MAXE bucket edge (4/5, 8/9, 12/13, 16/17 -- 17 leaves the staged kernel), KEEP (4 or 8)
# of the register kernels, and rows that reload LUT entries past the 32nd
ROW_LENGTHS = [1, 4, 5, 8, 9, 12, 13, 16, 17, 33, 40]


def pair_id(p):
    return "%s-%s" % (NAME[p[0]], NAME[p[1]])


# ---------------------------------------------------------------------------------------------------- float64 reference
def rows(orc):
    """(lut head, head slice, block ids) of every non-empty query row; with one LUT head it serves all heads."""
    for hl in range(orc.lut_heads):
        hs = slice(None) if orc.lut_heads == 1 else slice(hl, hl + 1)
        for row in orc.nn_list[hl]:
            if row:
                yield hl, hs, [b for b, _ in row]


def visibility(orc, autoregress_at_key=None):
    """bool[lut_heads, blocks, bs, bs] (key j of block b visible to its query row r), or None without a mask."""
    if orc.softmax_mask_np is None:
        return None
    return np.stack([np.stack([orc._mask_bits(hl, b, k, autoregress_at_key) for b, (_, k) in enumerate(orc.nt_list[hl])])
                     for hl in range(orc.lut_heads)])


def ref_softmax(orc, x, scale, vis=None):
    """float64 softmax of x (batch, heads, blocks, bs, bs) over each query row's blocks; masked entries are -FLT_MAX.

    Returns (y, mag, hard0): mag = max |x*scale| over the row's visible entries (bounds the kernel's fp32 exponent
    argument, see prob_bound), hard0 = masked entries of rows that have a visible entry (exactly 0 in the kernel too)."""
    x = np.asarray(x, np.float64)
    y = np.zeros_like(x)
    mag = np.zeros_like(x)
    hard0 = np.zeros(x.shape, bool)
    for hl, hs, bids in rows(orc):
        v = x[:, hs][:, :, bids] * scale                     # (batch, heads, L, bs, bs): [.., l, r, j] = row r, key j
        if vis is not None:
            seen = np.broadcast_to(vis[hl, bids], v.shape)
            v = np.where(seen, v, -FLT_MAX)
            some = seen.any(axis=(2, 4), keepdims=True)
            hard0[:, hs, bids] = ~seen & some
            mag[:, hs, bids] = np.where(seen, np.abs(v), 0).max(axis=(2, 4), keepdims=True)
        else:
            mag[:, hs, bids] = np.abs(v).max(axis=(2, 4), keepdims=True)
        e = np.exp(v - v.max(axis=(2, 4), keepdims=True))
        y[:, hs, bids] = e / e.sum(axis=(2, 4), keepdims=True)
    return y, mag, hard0


def ref_grad(orc, dy, y, scale):
    """dx = (dy - sum_row(dy*y)) * y * scale in float64 from the (rounded) inputs, and the kernel's accumulation bound
    gamma * |scale| * |y| * (|dy| + sum_row |dy*y|).  gamma = (n + 8) * 2^-24: the fp32 row sum of n = count*bs products
    (each product and each addition rounds once, at most n terms deep), the subtraction, two products and the lanes'
    xor-tree merge (<= 5 levels, within the + 8)."""
    dy, y = np.asarray(dy, np.float64), np.asarray(y, np.float64)
    dx = np.zeros_like(dy)
    err = np.zeros_like(dy)
    for hl, hs, bids in rows(orc):
        d, p = dy[:, hs][:, :, bids], y[:, hs][:, :, bids]
        acc = (d * p).sum(axis=(2, 4), keepdims=True)
        dx[:, hs, bids] = (d - acc) * p * scale
        gamma = (len(bids) * orc.blk_size + 8) * 2.0 ** -24
        err[:, hs, bids] = gamma * abs(scale) * np.abs(p) * (np.abs(d) + np.abs(d * p).sum(axis=(2, 4), keepdims=True))
    return dx, err


def long_row_rel(row_entries):
    """Worst-case relative error of an fp32 softmax over one row of `row_entries` entries: a lane adds up to
    row_entries/4 terms in sequence (at least 4 lanes share a row), each addition rounding by 2^-24, then a <= 5-level
    merge; exp2f, the reciprocal and the product add 2^-22."""
    return 2.0 ** -22 + (row_entries // 4 + 8) * 2.0 ** -24


def prob_bound(ref, mag, dtype, row_entries=0):
    """Elementwise bound on |kernel - reference| for probabilities.

    EPS/TINY above, plus the exponent argument: the kernel forms x*scale, the max subtraction and the log2(e) product
    in fp32, each rounding by 2^-24 of magnitudes <= mag, and an argument error d moves e^arg (and the row sum) by a
    relative d -- 2^-20 * mag covers the <= 6 such roundings of the element and of the terms that dominate the sum.
    Rows longer than 64 blocks pass `row_entries` and are held to long_row_rel instead of fp32's 1e-5."""
    rel = EPS[dtype]
    if row_entries:
        rel = max(rel, long_row_rel(row_entries))
    return (rel + 2.0 ** -20 * mag) * np.abs(ref) + TINY[dtype]


def assert_within(got, ref, bound, what):
    d = np.abs(got - ref)
    bad = ~(d <= bound)                                  # also catches NaN
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, d / np.maximum(bound, 1e-300), 0)), d.shape)
        raise AssertionError("%s: %d elements out of bound; worst at %s: got %.9g ref %.9g bound %.3g"
                             % (what, int(bad.sum()), i, got[i], ref[i], bound[i]))


def as_f64(t):
    return t.detach().float().cpu().numpy().astype(np.float64) if torch.is_tensor(t) else np.asarray(t, np.float64)


def check_probs(orc, got, ref, mag, hard0, dtype, what, row_entries=0):
    g = as_f64(got)
    assert_within(g, ref, prob_bound(ref, mag, dtype, row_entries), what)
    assert (g[hard0] == 0).all(), "%s: a masked entry is not exactly 0" % what
    # each row's stored probabilities sum to 1 within the half-ulps of its entries and the fp32 arithmetic
    arith = EPS[F32] if not row_entries else long_row_rel(row_entries)
    for hl, hs, bids in rows(orc):
        blk = g[:, hs][:, :, bids]
        s = blk.sum(axis=(2, 4))
        tol = 0.5 * ulp(blk, dtype).sum(axis=(2, 4)) + arith
        assert (np.abs(s - 1) <= tol).all(), "%s: row sums off by %.3g" % (what, float(np.abs(s - 1).max()))


def ulp(v, dtype):
    """One ulp of each value's magnitude in dtype, at least the subnormal step."""
    mant, sub = BITS[dtype]
    _, e = np.frexp(np.abs(np.asarray(v, np.float64)))
    return np.maximum(np.ldexp(1.0, e - 1 - mant), sub)


def check_grad(got, ref, err, dtype, what):
    g = as_f64(got)
    assert_within(g, ref, GRAD_EPS[dtype] * np.abs(ref) + err + TINY[dtype], what)


# ---------------------------------------------------------------------------------------------------- cases
def to_dev(a, dtype):
    """(CUDA tensor of `a` rounded to dtype, float64 copy of the rounded values)."""
    t = torch.as_tensor(np.asarray(a, np.float32)).to(dtype)
    return t.cuda(), t.double().numpy()


def build(layout, bs, heads, cb=None):
    return (BlocksparseTransformer(layout, bs, heads=heads, mask_callback=cb),
            TransformerOracle(layout, bs, heads=heads, mask_callback=cb))


def rand_mask(density, seed):
    """Random visibility bits, fixed per (head, query block, key block): lane groups end up partly masked."""
    def cb(shape, h, q, k, b):
        return np.random.default_rng((seed, h, q, k)).random(shape) < density
    return cb


def mixed_layout(L, lut_heads, seed=0):
    """Query rows of L, 0, ceil(L/2), 1 and L-1 key blocks over L + 2 key blocks: nn_max = L (which picks MAXE) while
    most rows are shorter, and one row is empty.  Head h holds the same rows rotated by h (equal block counts)."""
    lens = [L, 0, (L + 1) // 2, 1, max(L - 1, 0)]
    ctx_k = L + 2
    rng = np.random.default_rng((seed, L))
    base = np.zeros((len(lens), ctx_k), np.int32)
    for q, n in enumerate(lens):
        base[q, rng.choice(ctx_k, n, replace=False)] = 1
    return np.stack([np.roll(base, h, axis=0) for h in range(lut_heads)])


def staged_expected(bs, xdt, ydt, nn_max):
    return bs in (32, 64) and xdt != F32 and ydt != F32 and 1 <= nn_max <= 16


def kernel_names(staged):
    return ("bst_softmax_staged", "bst_softmax_grad_staged") if staged else ("bst_softmax", "bst_softmax_grad")


def grad_call(bst, dy, y, scale, dx_dtype):
    """The wrapper when dx has y's dtype; the C ABI directly for the mixed 16-bit / fp32 pairs it also accepts."""
    if dx_dtype == y.dtype:
        return bst._softmax_grad(dy, y, scale)
    lib = _lib.load()
    d = bst._device_luts(y.device)
    dx = torch.empty(y.shape, dtype=dx_dtype, device=y.device)
    rc = lib.bst_softmax_grad(_lib.dtype_code(y.dtype), _lib.dtype_code(dx_dtype), bst.blk_size,
                              d["nn"].data_ptr(), bst.lut_heads, bst.blocks, bst.nn_max,
                              dy.data_ptr(), y.data_ptr(), dx.data_ptr(), float(scale),
                              y.shape[0], bst.heads, bst.ctx_blks_q, _lib.stream_ptr())
    _lib.check(rc, "bst_softmax_grad")
    return dx


def run_softmax(bst, x, scale, use_mask, ak, ydt, kernel, what):
    y = bst._softmax(x, scale, use_mask, ak, ydt)
    assert _lib.last_kernel() == kernel, "%s: ran %s, expected %s" % (what, _lib.last_kernel(), kernel)
    assert _lib.device_error() == 0, _lib.device_error_text()
    return y


def run_grad(bst, dy, y, scale, dxt, kernel, what):
    dx = grad_call(bst, dy, y, scale, dxt)
    assert _lib.last_kernel() == kernel, "%s: ran %s, expected %s" % (what, _lib.last_kernel(), kernel)
    assert _lib.device_error() == 0, _lib.device_error_text()
    return dx


SWEEP_SCALE = 0.25


def sweep_case(bs, xdt, L, variant, seed=1):
    """batch 2, heads 3; 'plain': one shared LUT, no mask; 'perhead': a LUT and random mask bits per head."""
    heads, batch = 3, 2
    lut_heads = heads if variant == "perhead" else 1
    cb = rand_mask(0.7, bs) if variant == "perhead" else None
    bst, orc = build(mixed_layout(L, lut_heads), bs, heads, cb)
    rng = np.random.default_rng((seed, bs, L))
    x, xh = to_dev(rng.normal(0, 4, (batch, heads, orc.blocks, bs, bs)), xdt)
    return bst, orc, x, xh, rng


def grad_inputs(orc, xh, vis, dt, rng, scale=SWEEP_SCALE):
    """y = the float64 softmax rounded to dt, dy random."""
    yr, _, _ = ref_softmax(orc, xh, scale, vis)
    y, yh = to_dev(yr, dt)
    dy, dyh = to_dev(rng.normal(0, 1, yr.shape), dt)
    return y, yh, dy, dyh


# ---------------------------------------------------------------------------------------------------- CPU: the reference
def _callback_for(name, has_mask):
    if not has_mask:
        return None
    return checker_callback if "perhead" in name else causal_callback


@pytest.mark.parametrize("fname", golden_files("bst_"))
def test_reference_matches_fixtures(fname):
    """The float64 reference reproduces the reference checkers' fp32 outputs P, P_auto and DS within fp32 rounding."""
    g = np.load(os.path.join(GOLDEN, fname))
    orc = TransformerOracle(g["layout"], int(g["bs"]), heads=int(g["heads"]),
                            mask_callback=_callback_for(fname, bool(g["has_mask"])))
    scale = float(g["scale"])
    P, mag, _ = ref_softmax(orc, g["S"], scale, visibility(orc))
    # the fixtures were computed in fp32: the bound of an fp32 kernel applies to them as well
    assert_within(g["P"].astype(np.float64), P, prob_bound(P, mag, F32), "P")
    DS, err = ref_grad(orc, g["DP"], g["P"], scale)
    assert_within(g["DS"].astype(np.float64), DS, GRAD_EPS[F32] * np.abs(DS) + err + TINY[F32], "DS")
    if bool(g["has_mask"]):
        Pa, mag, _ = ref_softmax(orc, g["S"], scale, visibility(orc, int(g["autoregress_at_key"])))
        assert_within(g["P_auto"].astype(np.float64), Pa, prob_bound(Pa, mag, F32), "P_auto")


def test_reference_edge_semantics():
    """Fully masked rows are uniform over the row's entries, scale 0 is uniform over the visible ones, and a
    negative scale flips the order."""
    lay = np.ones((1, 2, 3), np.int32)
    bs = 8
    masked_row = lambda shape, h, q, k, b: np.tile((np.arange(bs) != 2)[:, None], (1, bs))   # row 2 of every block off
    orc = TransformerOracle(lay, bs, heads=1, mask_callback=masked_row)
    x = np.random.default_rng(0).normal(0, 3, (1, 1, orc.blocks, bs, bs))
    y, _, hard0 = ref_softmax(orc, x, 0.5, visibility(orc))
    assert np.all(y[:, :, :, 2, :] == 1.0 / (3 * bs)) and not hard0[:, :, :, 2, :].any()
    y0, _, _ = ref_softmax(orc, x, 0.0, visibility(orc))
    assert np.allclose(y0[:, :, :, 0, :], 1.0 / (3 * bs))
    yn, _, _ = ref_softmax(orc, x, -1.0, None)
    assert np.argmax(yn[0, 0, :3, 0, :].reshape(-1)) == np.argmin(x[0, 0, :3, 0, :].reshape(-1))


# ---------------------------------------------------------------------------------------------------- host checks
def _shape_cases(bs=32, heads=2):
    bst = BlocksparseTransformer(np.tril(np.ones((3, 3), np.int32)), bs, heads=heads)
    n = bst.blocks
    # every wrong shape holds MORE elements than the right one: even an unchecked launch would stay inside the tensor
    wrong = {"heads": (2, heads + 1, n, bs, bs), "blocks": (2, heads, n + 1, bs, bs),
             "bs": (2, heads, n, 2 * bs, 2 * bs), "rank": (2 * heads, n, bs, bs, 1)}
    return bst, (2, heads, n, bs, bs), wrong


@pytest.mark.parametrize("device", ["cpu", pytest.param("cuda", marks=pytest.mark.gpu)])
@pytest.mark.parametrize("which", ["heads", "blocks", "bs", "rank"])
def test_softmax_rejects_wrong_shapes(device, which):
    bst, good, wrong = _shape_cases()
    ok = torch.rand(good, device=device).half()
    bad = torch.rand(wrong[which], device=device).half()
    if device == "cuda":
        bst._softmax_grad(ok, ok, 1.0)                 # a known last kernel: a launch by the calls below would replace it
        before = _lib.last_kernel()
    with pytest.raises(ValueError, match="shape"):
        bst._softmax(bad, 1.0, False, None, torch.float16)
    with pytest.raises(ValueError, match="shape"):
        bst._softmax_grad(bad, ok, 1.0)
    with pytest.raises(ValueError, match="shape"):
        bst._softmax_grad(ok, bad, 1.0)
    with pytest.raises(ValueError, match="shape"):
        bst.softmax(bad)
    if device == "cuda":
        assert _lib.last_kernel() == before
        assert _lib.device_error() == 0


def _misaligned(t):
    """A copy of t that starts one element (2 or 4 bytes) past an aligned address."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0 and v.is_contiguous()
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("bs,L,dtype", [(64, 12, BF16), (64, 20, BF16), (8, 12, BF16), (16, 12, F16), (32, 20, F32)])
def test_misaligned_inputs(bs, L, dtype):
    """A view that starts inside its storage: the public ops copy it and give bit-identical results; the C ABI refuses
    it (BSMM_E_ARG) instead of handing it to a kernel whose vector accesses need alignment."""
    bst, orc = build(mixed_layout(L, 1), bs, 2, rand_mask(0.7, 3))
    rng = np.random.default_rng(5)
    x, _ = to_dev(rng.normal(0, 3, (2, 2, orc.blocks, bs, bs)), dtype)
    dy, _ = to_dev(rng.normal(0, 1, x.shape), dtype)
    xm, dym = _misaligned(x), _misaligned(dy)
    y = bst.masked_softmax(x, scale=0.5)
    ym = bst.masked_softmax(xm, scale=0.5)
    assert torch.equal(y, ym)
    assert torch.equal(bst._softmax_grad(dy, y, 0.5), bst._softmax_grad(dym, _misaligned(y), 0.5))
    assert _lib.device_error() == 0

    lib = _lib.load()
    d = bst._device_luts(x.device)
    out = torch.empty_like(x)
    code = _lib.dtype_code(dtype)
    rc = lib.bst_softmax(code, code, bs, d["nn"].data_ptr(), d["nt"].data_ptr(), bst.lut_heads, bst.blocks, bst.nn_max,
                         d["mask"].data_ptr(), bst.lut_heads, -1, xm.data_ptr(), out.data_ptr(), 0.5,
                         2, 2, bst.ctx_blks_q, _lib.stream_ptr())
    assert rc == E_ARG, (rc, _lib.device_error_text())
    rc = lib.bst_softmax_grad(code, code, bs, d["nn"].data_ptr(), bst.lut_heads, bst.blocks, bst.nn_max,
                              dym.data_ptr(), y.data_ptr(), out.data_ptr(), 0.5, 2, 2, bst.ctx_blks_q, _lib.stream_ptr())
    assert rc == E_ARG, (rc, _lib.device_error_text())
    assert _lib.device_error() == 0


# ---------------------------------------------------------------------------------------------------- dispatch sweep
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "perhead"])
@pytest.mark.parametrize("L", ROW_LENGTHS)
@pytest.mark.parametrize("xdt,ydt", PAIRS, ids=[pair_id(p) for p in PAIRS])
@pytest.mark.parametrize("bs", [8, 16, 32, 64])
def test_softmax_dispatch(bs, xdt, ydt, L, variant):
    bst, orc, x, xh, _ = sweep_case(bs, xdt, L, variant)
    assert bst.nn_max == L
    kernel = kernel_names(staged_expected(bs, xdt, ydt, L))[0]
    y = run_softmax(bst, x, SWEEP_SCALE, variant == "perhead", None, ydt, kernel, "forward")
    assert y.dtype == ydt
    ref, mag, hard0 = ref_softmax(orc, xh, SWEEP_SCALE, visibility(orc))
    check_probs(orc, y, ref, mag, hard0, ydt, "%s bs%d L%d" % (kernel, bs, L))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "perhead"])
@pytest.mark.parametrize("L", ROW_LENGTHS)
@pytest.mark.parametrize("dt,dxt", PAIRS, ids=[pair_id(p) for p in PAIRS])
@pytest.mark.parametrize("bs", [8, 16, 32, 64])
def test_softmax_grad_dispatch(bs, dt, dxt, L, variant):
    bst, orc, _, xh, rng = sweep_case(bs, F32, L, variant)
    y, yh, dy, dyh = grad_inputs(orc, xh, visibility(orc), dt, rng)
    kernel = kernel_names(staged_expected(bs, dt, dxt, L))[1]
    dx = run_grad(bst, dy, y, SWEEP_SCALE, dxt, kernel, "grad")
    assert dx.dtype == dxt
    ref, err = ref_grad(orc, dyh, yh, SWEEP_SCALE)
    check_grad(dx, ref, err, dxt, "%s bs%d L%d" % (kernel, bs, L))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, BF16], ids=NAME.get)
@pytest.mark.parametrize("bs", [8, 16, 32, 64])
def test_softmax_row_at_limit(bs, dtype):
    """A row of max_lut * bs = 32768 entries (512 blocks at bs 64, 4096 at bs 8), next to a short and an empty row."""
    L = 32768 // bs
    lay = np.zeros((3, L), np.int32)
    lay[0] = 1
    lay[2, [0, L // 2, L - 1]] = 1
    bst, orc = build(lay, bs, 2)
    assert bst.nn_max * bs == 32768
    rng = np.random.default_rng(bs)
    x, xh = to_dev(rng.normal(0, 4, (2, 2, orc.blocks, bs, bs)), dtype)
    y = run_softmax(bst, x, SWEEP_SCALE, False, None, dtype, "bst_softmax", "limit")
    ref, mag, hard0 = ref_softmax(orc, xh, SWEEP_SCALE)
    check_probs(orc, y, ref, mag, hard0, dtype, "limit bs%d" % bs, row_entries=32768)
    if dtype == F32:
        g = y.double().cpu().numpy()
        assert np.linalg.norm(g - ref) <= 1e-5 * np.linalg.norm(ref)
    yg, yh, dy, dyh = grad_inputs(orc, xh, None, dtype, rng)
    dx = run_grad(bst, dy, yg, SWEEP_SCALE, dtype, "bst_softmax_grad", "limit grad")
    ref, err = ref_grad(orc, dyh, yh, SWEEP_SCALE)
    check_grad(dx, ref, err, dtype, "limit grad bs%d" % bs)


# ---------------------------------------------------------------------------------------------------- masks
# (x dtype, y dtype, row length) per kernel path; staged exists for bs 32/64 only
PATHS = {"staged_f16": (F16, F16, 12), "staged_bf16": (BF16, BF16, 16), "reg_bf16": (BF16, BF16, 40), "reg_f32": (F32, F32, 40)}
PATH_BS = [(p, bs) for p in PATHS for bs in ((32, 64) if p.startswith("staged") else (8, 16, 32, 64))]


def path_case(path, bs, cb, lut_heads=1, heads=2, seed=0, x_sd=3.0):
    xdt, ydt, L = PATHS[path]
    bst, orc = build(mixed_layout(L, lut_heads, seed), bs, heads, cb)
    assert staged_expected(bs, xdt, ydt, bst.nn_max) == path.startswith("staged")
    rng = np.random.default_rng((seed, bs, L))
    xr = rng.normal(0, x_sd, (2, heads, orc.blocks, bs, bs))
    return bst, orc, xr, rng, xdt, ydt, kernel_names(path.startswith("staged"))


def mask_kind(kind, bs):
    rnd = rand_mask(0.6, 7)
    if kind == "none":
        return None
    if kind == "causal":
        return causal_callback
    if kind == "random":
        return rnd
    if kind == "zero_block":            # every third block: all words zero
        return lambda shape, h, q, k, b: np.zeros(shape, bool) if b % 3 == 0 else rnd(shape, h, q, k, b)

    def masked_rows(shape, h, q, k, b):  # row 5 of query block 0 and every row of query block 2: masked in all blocks
        m = rnd(shape, h, q, k, b)
        if q == 0:
            m[5 % bs] = False
        if q == 2:
            m[:] = False
        return m
    return masked_rows


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["none", "causal", "random", "zero_block", "masked_rows"])
@pytest.mark.parametrize("path,bs", PATH_BS)
def test_softmax_masks(path, bs, kind):
    bst, orc, xr, rng, xdt, ydt, (kf, kg) = path_case(path, bs, mask_kind(kind, bs), lut_heads=2)
    x, xh = to_dev(xr, xdt)
    y = run_softmax(bst, x, 0.5, kind != "none", None, ydt, kf, kind)
    vis = visibility(orc)
    ref, mag, hard0 = ref_softmax(orc, xh, 0.5, vis)
    check_probs(orc, y, ref, mag, hard0, ydt, "%s %s bs%d" % (kind, kf, bs))
    if kind == "masked_rows":          # query block 2 is masked everywhere: its rows are uniform (and finite)
        g = as_f64(y)
        row = orc.nn_list[0][2]
        assert row and orc.lut_heads == 2
        n = len(row) * bs
        assert np.all(np.abs(g[:, 0][:, [b for b, _ in row]] - 1.0 / n) <= ulp(1.0 / n, ydt))
    yg, yh, dy, dyh = grad_inputs(orc, xh, vis, xdt, rng, 0.5)
    dx = run_grad(bst, dy, yg, 0.5, xdt, kg, kind + " grad")
    ref, err = ref_grad(orc, dyh, yh, 0.5)
    check_grad(dx, ref, err, xdt, "%s grad bs%d" % (kind, bs))


def ar_layout(C, lut_heads):
    """Query blocks 0, 1, C/2 and C-1 attend to all C key blocks (the partial-autoregressive rewrite matters when
    queries see keys after them); the other query rows are empty.  Head h shifts the query rows by h."""
    lay = np.zeros((lut_heads, C, C), np.int32)
    for h in range(lut_heads):
        lay[h, [(q + h) % C for q in (0, 1, C // 2, C - 1)]] = 1
    return lay


def ar_values(C, bs):
    return {"0": 0, "1": 1, "bs-1": bs - 1, "bs": bs, "bs+1": bs + 1, "mid": (C * bs) // 2 + 3,
            "end-1": C * bs - 1, "end": C * bs, "past": C * bs + 7}


@pytest.mark.gpu
@pytest.mark.parametrize("ak", list(ar_values(1, 1)))
@pytest.mark.parametrize("path,bs", [("staged_bf16", 32), ("staged_bf16", 64), ("reg_bf16", 8), ("reg_bf16", 16),
                                     ("reg_bf16", 32), ("reg_bf16", 64), ("reg_f32", 16), ("reg_f32", 64)])
def test_softmax_autoregress_at_key(path, bs, ak):
    xdt, ydt, _ = PATHS[path]
    C = 12 if path.startswith("staged") else 20
    heads = 2
    cb = rand_mask(0.85, 11)
    bst, orc = build(ar_layout(C, heads), bs, heads, cb)
    kf = kernel_names(path.startswith("staged"))[0]
    a = ar_values(C, bs)[ak]
    rng = np.random.default_rng(bs)
    x, xh = to_dev(rng.normal(0, 3, (2, heads, orc.blocks, bs, bs)), xdt)
    y = run_softmax(bst, x, 0.5, True, a, ydt, kf, "ak=%d" % a)
    ref, mag, hard0 = ref_softmax(orc, xh, 0.5, visibility(orc, a))
    check_probs(orc, y, ref, mag, hard0, ydt, "%s ak=%d bs%d" % (kf, a, bs))


@pytest.mark.gpu
@pytest.mark.parametrize("lut_heads", [1, 3])
@pytest.mark.parametrize("bs", [8, 16, 32, 64])
def test_partial_autoregressive_mask_words(bs, lut_heads):
    """The standalone mask rewrite equals the oracle's words for every block, row and LUT head."""
    C = 6
    lay = np.tril(np.ones((C, C), np.int32)) | np.eye(C, k=2, dtype=np.int32)
    lay = np.stack([np.roll(np.roll(lay, h, 0), h, 1) for h in range(lut_heads)])
    cb = rand_mask(0.8, 5)
    bst, orc = build(lay, bs, 3, cb)
    weights = np.uint64(1) << np.arange(bs, dtype=np.uint64)
    for a in sorted(set(ar_values(C, bs).values())):
        got = bst.partial_autoregressive_mask(a).cpu().numpy().view(orc.softmax_mask_np.dtype)
        got = got.reshape(orc.softmax_mask_np.shape).astype(np.uint64)
        want = (visibility(orc, a).astype(np.uint64) * weights).sum(axis=3, dtype=np.uint64)
        np.testing.assert_array_equal(got, want, err_msg="autoregress_at_key=%d" % a)
    assert _lib.device_error() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [16, 64])
def test_public_masked_softmax_autoregress_autograd(bs):
    """masked_softmax(autoregress_at_key=...) with autograd at 16-bit on rows of 20 blocks: the register kernels run
    inside the public op, forward and backward."""
    C, heads, scale, a = 20, 2, 0.3, 7 * bs + 3
    bst, orc = build(ar_layout(C, 1), bs, heads, causal_callback)
    rng = np.random.default_rng(3)
    x, xh = to_dev(rng.normal(0, 3, (2, heads, orc.blocks, bs, bs)), BF16)
    dy, dyh = to_dev(rng.normal(0, 1, x.shape), BF16)
    x.requires_grad_()
    y = bst.masked_softmax(x, scale=scale, autoregress_at_key=a)
    assert _lib.last_kernel() == "bst_softmax" and y.dtype == BF16
    y.backward(dy)
    assert _lib.device_error() == 0
    # autograd runs backward on its own thread, and last_kernel() is per thread: repeat the call here to see the kernel
    assert torch.equal(bst._softmax_grad(dy, y.detach(), scale), x.grad)
    assert _lib.last_kernel() == "bst_softmax_grad"
    ref, mag, hard0 = ref_softmax(orc, xh, scale, visibility(orc, a))
    check_probs(orc, y, ref, mag, hard0, BF16, "public forward")
    assert not np.allclose(ref, ref_softmax(orc, xh, scale, visibility(orc))[0]), "autoregress_at_key had no effect"
    gref, err = ref_grad(orc, dyh, y.detach().double().cpu().numpy(), scale)
    check_grad(x.grad, gref, err, BF16, "public backward")


# ---------------------------------------------------------------------------------------------------- hard values
def hard_case(case, orc, rng, bs, heads):
    """(x before rounding, scale, use mask) of one 'hard values' case."""
    shape = (2, heads, orc.blocks, bs, bs)
    if case.startswith("scale"):
        return rng.normal(0, 2, shape), {"scale_eighth": 0.125, "scale_one": 1.0, "scale_eight": 8.0, "scale_zero": 0.0,
                                         "scale_neg": -0.5}[case], True
    if case == "large":                 # e^200 overflows fp32: only the max shift keeps this finite
        return rng.uniform(-250, 250, shape), 1.0, True
    if case == "large_neg":
        return rng.uniform(-250, 250, shape), -0.5, True
    if case == "constant":
        return np.full(shape, 1.5), 1.0, True
    if case == "ties":                  # many equal scores, the row max among them
        return np.clip(np.round(rng.normal(0, 1, shape) * 2) / 2, -1, 1), 1.0, True
    x = rng.normal(0, 1, shape)
    for hl, hs, bids in rows(orc):
        if case == "late_max":          # the max only in the row's 5th-last block (entry 35 of 40: after KEEP, after 32)
            late = bids[len(bids) - 5] if len(bids) >= 5 else bids[-1]
            r = np.arange(bs)
            x[:, hs, late, r, (3 * r + 1) % bs] += 25.0       # a different lane group for different rows
        elif case == "early_max":       # block 0 holds the max; the rest lie 110 below: e^-110 < 2^-149, exactly 0
            x[:, hs, bids[1:]] -= 110.0
    return x, 1.0 if case == "early_max" else 0.5, False


HARD = ["scale_eighth", "scale_one", "scale_eight", "scale_zero", "scale_neg", "large", "large_neg", "constant", "ties",
        "late_max", "early_max"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", HARD)
@pytest.mark.parametrize("path,bs", PATH_BS)
def test_softmax_hard_values(path, bs, case):
    bst, orc, _, rng, xdt, ydt, (kf, kg) = path_case(path, bs, rand_mask(0.8, 2))
    xr, scale, use_mask = hard_case(case, orc, rng, bs, 2)
    x, xh = to_dev(xr, xdt)
    y = run_softmax(bst, x, scale, use_mask, None, ydt, kf, case)
    vis = visibility(orc) if use_mask else None
    ref, mag, hard0 = ref_softmax(orc, xh, scale, vis)
    check_probs(orc, y, ref, mag, hard0, ydt, "%s %s bs%d" % (case, kf, bs))
    if case == "early_max":
        under = ref < 2.0 ** -153     # well below half the smallest fp32 subnormal (2^-150)
        assert under.sum() > 0 and np.all(as_f64(y)[under] == 0), "underflowed probabilities are not exactly 0"
    yg, yh, dy, dyh = grad_inputs(orc, xh, vis, xdt, rng, scale)
    dx = run_grad(bst, dy, yg, scale, xdt, kg, case + " grad")
    gref, err = ref_grad(orc, dyh, yh, scale)
    check_grad(dx, gref, err, xdt, "%s grad bs%d" % (case, bs))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["constant_dy", "one_hot_y"])
@pytest.mark.parametrize("path,bs", PATH_BS)
def test_softmax_grad_special_rows(path, bs, kind):
    bst, orc, xr, rng, dt, _, (_, kg) = path_case(path, bs, None)
    scale = -0.7
    yr = ref_softmax(orc, xr, 0.5)[0] if kind == "constant_dy" else np.zeros(xr.shape)
    dyr = rng.normal(0, 1, xr.shape)
    for hl, hs, bids in rows(orc):
        if kind == "constant_dy":       # dy = c along each row: dx = c (1 - sum y) y scale, ~0
            dyr[:, hs, bids] = rng.normal(0, 2, dyr[:, hs, bids].shape[:2] + (1, bs, 1))
        else:                           # a single 1 per row, at a different block and lane group per row
            n = len(bids)
            r = np.arange(bs)
            yr[:, hs, np.array(bids)[r % n], r, (5 * r + 2) % bs] = 1.0
    y, yh = to_dev(yr, dt)
    dy, dyh = to_dev(dyr, dt)
    dx = run_grad(bst, dy, y, scale, dt, kg, kind)
    g = as_f64(dx)
    ref, err = ref_grad(orc, dyh, yh, scale)
    check_grad(dx, ref, err, dt, "%s bs%d" % (kind, bs))
    if kind == "one_hot_y":             # sum_row(dy*y) = dy at the 1, exactly: every dx is exactly 0
        assert np.all(g == 0)
    else:
        for hl, hs, bids in rows(orc):
            p, c = yh[:, hs][:, :, bids], dyh[:, hs][:, :, bids]
            off = np.abs(1 - p.sum(axis=(2, 4), keepdims=True))
            bound = abs(scale) * np.abs(p) * np.abs(c) * off + err[:, hs][:, :, bids] + TINY[dt] + GRAD_EPS[dt] * np.abs(ref[:, hs][:, :, bids])
            assert np.all(np.abs(g[:, hs][:, :, bids]) <= bound)


# ---------------------------------------------------------------------------------------------------- staged vs register
def _compare_cases():
    """The staged cases of the sweep (perhead variant): forward and gradient outputs and the kernels that ran."""
    out = {}
    for bs in (32, 64):
        for xdt, ydt in PAIRS16:
            for L in (4, 8, 12, 16):
                bst, orc, x, xh, rng = sweep_case(bs, xdt, L, "perhead", seed=4)
                y = bst._softmax(x, SWEEP_SCALE, True, None, ydt)
                kf = _lib.last_kernel()
                yg, yh, dy, dyh = grad_inputs(orc, xh, visibility(orc), xdt, rng)
                dx = grad_call(bst, dy, yg, SWEEP_SCALE, ydt)
                kg = _lib.last_kernel()
                key = "bs%d_%s_%s_L%d" % (bs, NAME[xdt], NAME[ydt], L)
                out[key + "_y"] = y.float().cpu().numpy()
                out[key + "_dx"] = dx.float().cpu().numpy()
                out[key + "_dx_order"] = 2 * ref_grad(orc, dyh, yh, SWEEP_SCALE)[1]
                out[key + "_kernels"] = np.array([kf, kg])
    assert _lib.device_error() == 0
    return out


def _dump_compare_cases(path):
    np.savez(path, **_compare_cases())


@pytest.mark.gpu
def test_staged_matches_register(tmp_path):
    """The same staged cases in a process with BSMM_SOFTMAX_STAGED=0 (read once per process) run the register kernels;
    both store 16-bit values of the same fp32 math, so they agree within one output ulp.  The gradient's row sum is
    added in a different order by the two kernels, and (dy - sum) can cancel: dx may also differ by the two sums'
    accumulation bounds (ref_grad)."""
    mine = _compare_cases()
    out = str(tmp_path / "register.npz")
    env = dict(os.environ, BSMM_SOFTMAX_STAGED="0")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
          ["-c", "import sys; sys.path.insert(0, %r); from tests.test_softmax_gpu import _dump_compare_cases; "
                 "_dump_compare_cases(sys.argv[1])" % ROOT, out]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    theirs = np.load(out)
    assert sorted(theirs.files) == sorted(mine)
    for key in mine:
        if key.endswith("_dx_order"):
            continue
        if key.endswith("_kernels"):
            assert list(mine[key]) == ["bst_softmax_staged", "bst_softmax_grad_staged"], key
            assert list(theirs[key]) == ["bst_softmax", "bst_softmax_grad"], key
            continue
        dtype = {"bf16": BF16, "f16": F16}[key.split("_")[2]]     # y and dx have the output dtype
        a, b = mine[key], theirs[key]
        tol = ulp(np.maximum(np.abs(a), np.abs(b)), dtype) + (mine[key + "_order"] if key.endswith("_dx") else 0)
        ok = np.abs(a.astype(np.float64) - b) <= tol
        assert ok.all(), "%s: %d values differ by more than one ulp" % (key, int((~ok).sum()))


# ---------------------------------------------------------------------------------------------------- > 2^31 elements
@pytest.mark.gpu
@pytest.mark.parametrize("band,batch,heads,kernels", [(16, 145, 4, kernel_names(True)), (20, 121, 4, kernel_names(False))])
def test_offsets_past_2_31(band, batch, heads, kernels):
    """batch*heads*blocks*bs^2 > 2^31 (bst_nt's limit is 2^32): element offsets of the last batch entry need 64 bits.
    bs 64, a causal band of `band` blocks on a 64 x 64 block grid; rows <= 16 blocks take the staged kernels."""
    nb, bs = 64, 64
    q, k = np.indices((nb, nb))
    lay = ((k <= q) & (q - k < band)).astype(np.int32)
    bst, orc = build(lay, bs, heads, causal_callback)
    shape = (batch, heads, orc.blocks, bs, bs)
    assert np.prod(shape, dtype=np.int64) > 2 ** 31
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    gen = torch.Generator(device="cuda").manual_seed(band)
    x = torch.randn(shape, generator=gen, device="cuda", dtype=BF16)
    y = bst._softmax(x, 0.5, True, None, BF16)
    assert _lib.last_kernel() == kernels[0] and _lib.device_error() == 0
    xl = as_f64(x[-1:])
    del x
    dy = torch.randn(shape, generator=gen, device="cuda", dtype=BF16)
    dx = bst._softmax_grad(dy, y, 0.5)
    assert _lib.last_kernel() == kernels[1] and _lib.device_error() == 0
    yl, dyl, dxl = (as_f64(t[-1:]) for t in (y, dy, dx))
    del y, dy, dx
    peak = torch.cuda.max_memory_allocated()
    torch.cuda.empty_cache()
    ref, mag, hard0 = ref_softmax(orc, xl, 0.5, visibility(orc))
    check_probs(orc, yl, ref, mag, hard0, BF16, "last batch entry")
    gref, err = ref_grad(orc, dyl, yl, 0.5)
    check_grad(dxl, gref, err, BF16, "last batch entry grad")
    print("offsets past 2^31, band %d: %d elements, peak %.2f GB" % (band, int(np.prod(shape)), peak / 1e9))
