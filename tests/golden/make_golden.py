"""Generate the golden fixtures in this directory from the REFERENCE implementation.

Needs a checkout of openai/blocksparse; the tests only read the committed .npz files:

    python tests/golden/make_golden.py <path to the openai/blocksparse checkout>

How the reference is imported without TensorFlow (SURVEY.md appendix C.4): a
MagicMock stands in for `tensorflow` (only graph-building code touches it, none of
which runs here), and the package __init__ is bypassed so that only
blocksparse/matmul.py, transformer.py and utils.py are loaded.  Everything the
fixtures record is computed by the reference's own Python/NumPy code:

  * BlocksparseMatMul.__init__/xprop_lut  -> LUT wire formats, lists, segments, locks
  * fprop_test / bprop_test / updat_test  -> numeric outputs on seeded inputs
  * BlocksparseTransformer.__init__/xn_lut/init_softmax_mask -> LUTs and bit masks
  * nt_test / nn_test / tn_test / masked_softmax_test / masked_softmax_grad_test

One caveat, recorded in every matmul fixture as `find_order`:
matmul.py:113-115 relies on scipy.sparse.find returning blocks sorted by column.
SciPy >= 1.8 returns them row-major, which fragments every output column into many
lock-less segments.  We record BOTH behaviours: `asis_*` keys hold what the
unmodified reference produces with this container's SciPy, and the unprefixed keys
hold what it produces when scipy.sparse.find is wrapped to return the
column-sorted order its comment assumes.  Numeric *_test outputs are identical
in both cases and are stored once.
"""
import importlib
import os
import sys
import types
from unittest import mock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference(ref):
    tf = mock.MagicMock()
    for name in ["tensorflow", "tensorflow.python", "tensorflow.python.framework",
                 "tensorflow.python.framework.ops", "tensorflow.python.ops",
                 "tensorflow.python.ops.init_ops"]:
        sys.modules[name] = tf if name == "tensorflow" else mock.MagicMock()
    sys.modules["tensorflow.python.framework.ops"].RegisterGradient = lambda *_a, **_k: (lambda f: f)
    sys.modules["tensorflow.python.ops.init_ops"].Initializer = object
    sys.modules["tensorflow.python.framework"].ops = sys.modules["tensorflow.python.framework.ops"]
    pkg = types.ModuleType("blocksparse")
    pkg.__path__ = [os.path.join(ref, "blocksparse")]
    sys.modules["blocksparse"] = pkg
    ew = types.ModuleType("blocksparse.ewops")
    sys.modules["blocksparse.ewops"] = ew
    mm = importlib.import_module("blocksparse.matmul")
    tr = importlib.import_module("blocksparse.transformer")
    return mm, tr


def layouts_matmul(rng):
    """Layouts modelled on the reference's tests (test/blocksparse_matmul_test.py:276-280)."""
    out = {}
    lay = (rng.random((8, 8)) < 0.25).astype(np.int32)
    np.fill_diagonal(lay, 1)
    out["cfg1_8x8_d25"] = lay
    lay = (rng.random((6, 10)) < 0.4).astype(np.int32)
    lay[:, 3] = 0            # empty output column  -> zero-filled segment
    lay[2, :] = 0            # empty input row
    lay[0, 0] = 1
    out["ragged_6x10_empty"] = lay
    # skewed: a dense corner plus sparse tail, triggers segmentation + locks
    lay = (rng.random((24, 24)) < 0.08).astype(np.int32)
    np.fill_diagonal(lay, 1)
    lay[:, :2] = 1
    lay[:2, :] = 1
    out["skewed_24x24"] = lay
    out["dense_4x4"] = np.ones((4, 4), dtype=np.int32)
    return out


def gen_matmul(mm):
    import scipy.sparse as sparse
    real_find = sparse.find

    def find_colmajor(csr):
        r, c, v = real_find(csr)
        order = np.lexsort((r, c))
        return r[order], c[order], v[order]

    rng = np.random.default_rng(20260922)
    for name, lay in layouts_matmul(rng).items():
        for bsize, axis in [(32, 0), (16, 0), (8, 0), (32, 1), (64, 1)]:
            if bsize >= 32 and lay.shape[0] > 8:
                continue        # keep fixtures small: big layouts only at bs 8/16
            rec = {"layout": lay, "bsize": bsize, "axis": axis}
            for tag, finder in [("", find_colmajor), ("asis_", real_find)]:
                mm.sparse.find = finder
                try:
                    ref = mm.BlocksparseMatMul(lay.copy(), block_size=bsize, feature_axis=axis)
                finally:
                    mm.sparse.find = real_find
                rec[tag + "fprop_lut"] = ref.fprop_lut
                rec[tag + "bprop_lut"] = ref.bprop_lut
                rec[tag + "updat_lut"] = ref.updat_lut
                rec[tag + "meta"] = np.array([ref.fprop_segments, ref.fprop_locks, ref.fprop_shared,
                                              ref.bprop_segments, ref.bprop_locks, ref.bprop_shared,
                                              ref.blocks, ref.C, ref.K], dtype=np.int64)
                if tag == "":
                    keep = ref
            ref = keep
            N = 8 if bsize >= 32 else 12
            W = rng.normal(0, 0.1, ref.w_shape).astype(np.float32)
            X = rng.normal(0, 1.0, ref.i_shape(N)).astype(np.float32)
            E = rng.normal(0, 1.0, ref.o_shape(N)).astype(np.float32)
            rec["W"], rec["X"], rec["E"] = W, X, E
            rec["Y"] = ref.fprop_test(X, W).astype(np.float64)
            rec["DX"] = ref.bprop_test(E, W).astype(np.float64)
            rec["DW"] = ref.updat_test(X, E).astype(np.float64)
            if axis == 0:
                gate = (rng.random(ref.blocks) < 0.7).astype(np.float32) * rng.uniform(0.5, 1.5, ref.blocks).astype(np.float32)
                rec["gate"] = gate
                rec["Y_gated"] = ref.fprop_test(X, W, gate=gate)
                rec["DX_gated"] = ref.bprop_test(E, W, gate=gate)
                rec["DW_gated"] = ref.updat_test(X, E, gate=gate, dw_gated=True)
            np.savez_compressed(os.path.join(HERE, "bsmm_%s_bs%d_ax%d.npz" % (name, bsize, axis)), **rec)
            print("wrote", name, bsize, axis, "blocks", ref.blocks,
                  "segments", ref.fprop_segments, ref.bprop_segments, "locks", ref.fprop_locks, ref.bprop_locks)


def causal_callback(blk_shape, head_idx, qry_idx, key_idx, blk_idx):
    """test/blocksparse_transformer_test.py:21-33 recipe: causal inside diagonal blocks."""
    mask = np.ones(blk_shape, dtype=bool)
    if qry_idx == key_idx:
        for q, k in np.ndindex(blk_shape):
            if k > q:
                mask[q, k] = False
    return mask


def checker_callback(blk_shape, head_idx, qry_idx, key_idx, blk_idx):
    q, k = np.indices(blk_shape)
    m = ((q + k + head_idx) % 3) != 0
    m[:, 0] = True      # keep every row non-empty
    return m


def gen_transformer(tr):
    rng = np.random.default_rng(20260923)
    cases = []
    # lower-triangular shared layout, causal mask (…Sparse test :106-182)
    cases.append(("tril_bs32", np.tril(np.ones((4, 4), np.int32)), 32, 2, causal_callback, 16))
    cases.append(("tril_bs64", np.tril(np.ones((3, 3), np.int32)), 64, 2, causal_callback, 16))
    # per-head random layouts with equal block counts, odd mask, rectangular ctx
    lay = np.zeros((2, 5, 6), np.int32)
    for h in range(2):
        idx = rng.permutation(30)[:13]
        lay[h].reshape(-1)[idx] = 1
        for q in range(5):
            if lay[h, q].sum() == 0:
                pass
    # make sure each head has the same count (13) and every query row is non-empty
    lay = np.zeros((2, 5, 6), np.int32)
    for h in range(2):
        for q in range(5):
            lay[h, q, (q + h) % 6] = 1
        extra = [i for i in rng.permutation(30) if lay[h].reshape(-1)[i] == 0][:8]
        lay[h].reshape(-1)[extra] = 1
    cases.append(("perhead_bs16", lay, 16, 2, checker_callback, 8))
    cases.append(("perhead_bs8", lay, 8, 2, checker_callback, 8))
    cases.append(("nomask_bs32", np.tril(np.ones((4, 4), np.int32)), 32, 2, None, 16))

    for name, lay, bs, heads, cb, hs in cases:
        ref = tr.BlocksparseTransformer(lay, block_size=bs, heads=heads, mask_callback=cb)
        batch = 2
        S = heads * hs
        Q = rng.uniform(-1, 1, (batch, ref.ctx_blks_q * bs, S)).astype(np.float32)
        K = rng.uniform(-1, 1, (batch, ref.ctx_blks_k * bs, S)).astype(np.float32)
        V = rng.uniform(-1, 1, (batch, ref.ctx_blks_k * bs, S)).astype(np.float32)
        scale = 1.0 / np.sqrt(hs)
        Wt = ref.nt_test(Q, K)
        P = ref.masked_softmax_test(Wt, scale=scale)
        Y = ref.nn_test(P, V)
        DY = rng.uniform(-1, 1, Y.shape).astype(np.float32)
        DV = ref.tn_test(P, DY)
        DP = ref.nt_test(DY, V)
        DS = ref.masked_softmax_grad_test(DP, P, scale=scale)
        rec = dict(layout=lay, bs=bs, heads=heads, hs=hs, scale=scale, has_mask=cb is not None,
                   nt_lut=ref.nt_lut, nn_lut=ref.nn_lut, tn_lut=ref.tn_lut,
                   meta=np.array([ref.blocks, ref.nn_max, ref.tn_max, ref.ctx_blks_q, ref.ctx_blks_k]),
                   Q=Q, K=K, V=V, DY=DY, S=Wt, P=P, Y=Y, DV=DV, DP=DP, DS=DS)
        if cb is not None:
            rec["mask_np"] = ref.softmax_mask_np
            rec["mask_dev"] = ref.softmax_mask
            ak = (ref.ctx_blks_k * bs) // 2 + 3
            rec["autoregress_at_key"] = ak
            rec["P_auto"] = ref.masked_softmax_test(Wt, scale=scale, autoregress_at_key=ak)
        if name == "tril_bs64":
            # batch entries are computed independently: storing the first one keeps this fixture under 1 MB
            for k in ("Q", "K", "V", "DY", "S", "P", "Y", "DV", "DP", "DS", "P_auto"):
                rec[k] = rec[k][:1]
        np.savez_compressed(os.path.join(HERE, "bst_%s.npz" % name), **rec)
        print("wrote", name, "blocks", ref.blocks, "nn_max", ref.nn_max, "tn_max", ref.tn_max)


def gen_wutil(mm):
    """l2_normalize_test / l2_normalize_grad_test (matmul.py:421-443) on seeded inputs -> wutil_*.npz."""
    import scipy.sparse as sparse
    real_find = sparse.find

    def find_colmajor(csr):
        r, c, v = real_find(csr)
        order = np.lexsort((r, c))
        return r[order], c[order], v[order]

    rng = np.random.default_rng(20260924)
    lays = {"rand_6x7": (rng.random((6, 7)) < 0.45).astype(np.int32), "dense_3x3": np.ones((3, 3), np.int32)}
    lays["rand_6x7"][0, 0] = 1
    lays["rand_6x7"][:, 5] = 0                      # an empty output column
    for name, lay in lays.items():
        for bsize in (8, 16, 32):
            mm.sparse.find = find_colmajor
            try:
                ref = mm.BlocksparseMatMul(lay.copy(), block_size=bsize, feature_axis=0)
            finally:
                mm.sparse.find = real_find
            W = rng.normal(0, 1.0, ref.w_shape).astype(np.float32)
            U = rng.normal(0, 1.0, ref.w_shape).astype(np.float32)
            rec = dict(layout=lay, bsize=bsize, W=W, U=U,
                       Y=ref.l2_normalize_test(W.copy()), DX=ref.l2_normalize_grad_test(W.copy(), U.copy()))
            np.savez_compressed(os.path.join(HERE, "wutil_%s_bs%d.npz" % (name, bsize)), **rec)
            print("wrote wutil", name, bsize)


if __name__ == "__main__":
    mm, tr = import_reference(sys.argv[1])
    gen_matmul(mm)
    gen_transformer(tr)
    gen_wutil(mm)
