"""BlocksparseTransformer for B200 -- host side.

Keeps the Python op surface of the reference's blocksparse/transformer.py (class
BlocksparseTransformer :51-383, gradient wiring :391-480) on torch tensors, calling the
sm_100a kernels through the C ABI in include/bsmm_b200.h.

Tensor conventions (reference transformer.py:186-203):
  dense  q/k/v : (batch, ctx, heads*head_state), heads-major state
  sparse w     : (batch, heads, blocks, block_size, block_size)
"""
import numpy as np
import torch

from . import _lib
from .checkers import TransformerCheckers
from .lut import TransformerLuts


class BlocksparseTransformer(TransformerCheckers):
    """Drop-in for blocksparse.transformer.BlocksparseTransformer (reference transformer.py:51)."""

    def __getstate__(self):
        # the reference leaves pickling as a TODO (transformer.py:53-59); we support it
        return (self.layout, self.blk_size, self.heads, self.mask_callback, self.name)

    def __setstate__(self, state):
        self.__init__(*state)

    def __init__(self, layout, block_size=64, heads=None, mask_callback=None, name=None):
        layout = np.asarray(layout)
        if layout.ndim == 2:
            assert heads is not None, "heads must be explicitly specified when using shared layouts per head"
            layout = layout[None]
        if heads is None:
            heads = layout.shape[0]
        assert block_size in (8, 16, 32, 64), "Block sizes of 8, 16, 32 and 64 currently supported"
        assert layout.ndim == 3, "bad layout shape: " + str(layout.shape)
        assert layout.shape[0] in (1, heads), "layout must have 1 or `heads` leading entries"
        self.layout = layout != 0
        self.mask_callback = mask_callback
        self.blk_size = block_size
        self.name = name
        self.heads = heads
        self.blk_shape = (block_size, block_size)
        self.softmax_dtype = None
        luts = TransformerLuts(layout, block_size, mask_callback)
        self._luts = luts
        for k in ("lut_heads", "ctx_blks_q", "ctx_blks_k", "blocks", "nn_max", "tn_max",
                  "nt_lut", "nn_lut", "tn_lut", "nt_list", "nn_list", "tn_list",
                  "softmax_mask", "softmax_mask_np"):
            setattr(self, k, getattr(luts, k))
        self._dev = {}

    def block_coord(self, block, head=0):
        return self.nt_list[head][block]

    def _device_luts(self, device):
        key = (device.type, device.index)
        d = self._dev.get(key)
        if d is None:
            d = {"nt": torch.as_tensor(self.nt_lut, device=device),
                 "nn": torch.as_tensor(self.nn_lut, device=device),
                 "tn": torch.as_tensor(self.tn_lut, device=device),
                 "nt_items": torch.as_tensor(self._luts.nt_items, device=device),
                 "nn_order": torch.as_tensor(self._luts.nn_order, device=device),
                 "tn_order": torch.as_tensor(self._luts.tn_order, device=device),
                 "mask": None}
            if self.softmax_mask_np is not None:
                m = self.softmax_mask_np
                # torch has no uint16/32/64 arithmetic but can carry the bytes
                d["mask"] = torch.as_tensor(m.view(np.uint8).reshape(-1).copy(), device=device)
            self._dev[key] = d
        return d

    # ------------------------------------------------------------------ raw ops
    @_lib.guarded
    def _nt(self, a, b, c_dtype, flags=0):
        lib = _lib.load()
        if not a.is_cuda:
            raise _lib.BsmmError("BlocksparseTransformer needs CUDA tensors (no CPU path)")
        a, b = a.contiguous(), b.contiguous()
        batch, ctx_a, S = a.shape
        if ctx_a != self.ctx_blks_q * self.blk_size or b.shape[1] != self.ctx_blks_k * self.blk_size:
            raise ValueError("context sizes do not match the layout")
        if S % self.heads or b.shape[2] != S or a.dtype != b.dtype:
            raise ValueError("state size / dtype mismatch")
        hs = S // self.heads
        c = torch.empty((batch, self.heads, self.blocks, self.blk_size, self.blk_size), dtype=c_dtype, device=a.device)
        d = self._device_luts(a.device)
        rc = lib.bst_nt(_lib.dtype_code(a.dtype), _lib.dtype_code(c_dtype), self.blk_size,
                        d["nt"].data_ptr(), self.lut_heads, self.blocks,
                        d["nt_items"].data_ptr(), int(self._luts.nt_items.shape[1]),
                        a.data_ptr(), b.data_ptr(), c.data_ptr(),
                        batch, self.heads, hs, self.ctx_blks_q, self.ctx_blks_k, flags, _lib.stream_ptr())
        _lib.check(rc, "bst_nt")
        return c

    @_lib.guarded
    def _xn(self, a, b, transpose_a, flags=0):
        lib = _lib.load()
        if not a.is_cuda:
            raise _lib.BsmmError("BlocksparseTransformer needs CUDA tensors (no CPU path)")
        a, b = a.contiguous(), b.contiguous()
        batch, ctx_b, S = b.shape
        ctx_blks_b = self.ctx_blks_q if transpose_a else self.ctx_blks_k
        ctx_blks_c = self.ctx_blks_k if transpose_a else self.ctx_blks_q
        if ctx_b != ctx_blks_b * self.blk_size:
            raise ValueError("context size does not match the layout")
        if tuple(a.shape) != (batch, self.heads, self.blocks, self.blk_size, self.blk_size):
            raise ValueError("sparse operand has the wrong shape %s" % (tuple(a.shape),))
        hs = S // self.heads
        c = torch.empty((batch, ctx_blks_c * self.blk_size, S), dtype=b.dtype, device=b.device)
        d = self._device_luts(b.device)
        lut = d["tn"] if transpose_a else d["nn"]
        order = d["tn_order"] if transpose_a else d["nn_order"]
        rc = lib.bst_xn(_lib.dtype_code(a.dtype), _lib.dtype_code(b.dtype), self.blk_size, int(transpose_a),
                        lut.data_ptr(), order.data_ptr(), self.lut_heads, self.blocks, self.tn_max if transpose_a else self.nn_max,
                        a.data_ptr(), b.data_ptr(), c.data_ptr(),
                        batch, self.heads, hs, ctx_blks_b, ctx_blks_c, flags, _lib.stream_ptr())
        _lib.check(rc, "bst_xn")
        return c

    def _check_sparse(self, t, what):
        """The kernels index a (batch, heads, blocks, bs, bs) tensor through the LUTs: any other shape reads past it."""
        if t.dim() != 5 or tuple(t.shape[1:]) != (self.heads, self.blocks, self.blk_size, self.blk_size):
            raise ValueError("%s has shape %s; expected (batch, %d, %d, %d, %d)"
                             % (what, tuple(t.shape), self.heads, self.blocks, self.blk_size, self.blk_size))

    @staticmethod
    def _aligned(t):
        """Contiguous and 16-byte aligned, as the softmax kernels' vector and bulk accesses need: a view that starts part
        way into its storage (x[1:], a slice of a flat buffer) is copied."""
        t = t.contiguous()
        return t if t.data_ptr() % 16 == 0 else t.clone()

    @_lib.guarded
    def _softmax(self, x, scale, use_mask, autoregress_at_key, dtype):
        self._check_sparse(x, "softmax input")
        if not x.is_cuda:
            raise _lib.BsmmError("BlocksparseTransformer needs CUDA tensors (no CPU path)")
        lib = _lib.load()
        x = self._aligned(x)
        batch = x.shape[0]
        y = torch.empty(x.shape, dtype=dtype, device=x.device)
        d = self._device_luts(x.device)
        mask = d["mask"] if use_mask else None
        ak = -1 if autoregress_at_key is None else int(autoregress_at_key)
        rc = lib.bst_softmax(_lib.dtype_code(x.dtype), _lib.dtype_code(dtype), self.blk_size,
                             d["nn"].data_ptr(), d["nt"].data_ptr(), self.lut_heads, self.blocks, self.nn_max,
                             _lib.ptr(mask), self.lut_heads, ak,
                             x.data_ptr(), y.data_ptr(), float(scale),
                             batch, self.heads, self.ctx_blks_q, _lib.stream_ptr())
        _lib.check(rc, "bst_softmax")
        return y

    @_lib.guarded
    def _softmax_grad(self, dy, y, scale):
        self._check_sparse(y, "softmax output")
        if dy.shape != y.shape:
            raise ValueError("softmax gradient has shape %s, softmax output %s" % (tuple(dy.shape), tuple(y.shape)))
        if not (y.is_cuda and dy.is_cuda):
            raise _lib.BsmmError("BlocksparseTransformer needs CUDA tensors (no CPU path)")
        lib = _lib.load()
        dy = self._aligned(dy.to(y.dtype))
        y = self._aligned(y)
        dx = torch.empty_like(dy)
        d = self._device_luts(y.device)
        rc = lib.bst_softmax_grad(_lib.dtype_code(y.dtype), _lib.dtype_code(dx.dtype), self.blk_size,
                                  d["nn"].data_ptr(), self.lut_heads, self.blocks, self.nn_max,
                                  dy.data_ptr(), y.data_ptr(), dx.data_ptr(), float(scale),
                                  y.shape[0], self.heads, self.ctx_blks_q, _lib.stream_ptr())
        _lib.check(rc, "bst_softmax_grad")
        return dx

    def partial_autoregressive_mask(self, autoregress_at_key, device="cuda"):
        """Device mask rewritten so causality starts at key `autoregress_at_key` (bst_op.cc:519-575).

        Returns a uint8 byte tensor holding uint{blk_size}[lut_heads][blocks][blk_size].
        """
        if self.softmax_mask_np is None:
            raise ValueError("autoregress_at_key only applies to ops with mask_callback defined.")
        lib = _lib.load()
        device = torch.device(device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        d = self._device_luts(device)
        out = torch.empty_like(d["mask"])
        with torch.cuda.device(device):        # launch on the device (and its current stream) that holds the mask
            rc = lib.bst_autoregressive_mask(self.blk_size, d["nt"].data_ptr(), self.lut_heads, self.blocks,
                                             d["mask"].data_ptr(), out.data_ptr(), int(autoregress_at_key),
                                             _lib.stream_ptr())
        _lib.check(rc, "bst_autoregressive_mask")
        return out

    # ------------------------------------------------------------------ public ops (autograd)
    def _bench(self, what, fn, a, hs, repeat, name):
        """The reference's `bench` op attribute (transformer.py:166-181, src/bst_op.cc:160-176,221-222): time `repeat`
        launches between two CUDA events and print one line."""
        import ctypes
        lib = _lib.load()
        timer = ctypes.c_void_p()
        _lib.check(lib.bsmm_timer_create(ctypes.byref(timer)), "timer_create")
        fn()
        _lib.check(lib.bsmm_timer_begin(timer, _lib.stream_ptr()), "timer_begin")
        for _ in range(repeat):
            fn()
        ms = ctypes.c_float()
        _lib.check(lib.bsmm_timer_end(timer, _lib.stream_ptr(), ctypes.byref(ms)), "timer_end")
        lib.bsmm_timer_destroy(timer)
        ms_per = ms.value / repeat
        flops = 2.0 * self.blocks * self.blk_size * self.blk_size * hs * a.shape[0] * self.heads
        print("%s %s ms: %.4f gflops: %.0f" % (name or self.name or "bst", what, ms_per, flops / (ms_per * 1e6)))
        return ms_per

    def nt_op(self, a, b, name=None, bench=0):
        if bench:
            self._bench("nt", lambda: self._nt(a, b, torch.bfloat16), a, a.shape[2] // self.heads, bench, name)
        return _NtFunction.apply(a, b, self, torch.bfloat16)

    def nn_op(self, a, b, name=None, bench=0):
        if bench:
            self._bench("nn", lambda: self._xn(a, b, False), b, b.shape[2] // self.heads, bench, name)
        return _XnFunction.apply(a, b, self, False)

    def tn_op(self, a, b, name=None, bench=0):
        if bench:
            self._bench("tn", lambda: self._xn(a, b, True), b, b.shape[2] // self.heads, bench, name)
        return _XnFunction.apply(a, b, self, True)

    def query_key_op(self, q, k, name=None, bench=0):
        # reference transformer.py:337-347: scores are always bf16; softmax output dtype follows q
        self.softmax_dtype = torch.bfloat16 if q.dtype == torch.float32 else q.dtype
        return self.nt_op(q, k, name=name, bench=bench)

    def weight_value_op(self, w, v, name=None, bench=0):
        return self.nn_op(w, v, name=name, bench=bench)

    def masked_softmax(self, x, scale=1.0, autoregress_at_key=None, dtype=None):
        if self.softmax_mask_np is None:
            if autoregress_at_key is not None:
                raise ValueError("autoregress_at_key only applies to ops with mask_callback defined.")
            return self.softmax(x, scale, dtype)
        dtype = dtype or self.softmax_dtype or x.dtype
        return _SoftmaxFunction.apply(x, self, float(scale), True, autoregress_at_key, dtype)

    def softmax(self, x, scale=1.0, dtype=None):
        dtype = dtype or self.softmax_dtype or x.dtype
        return _SoftmaxFunction.apply(x, self, float(scale), False, None, dtype)


class _NtFunction(torch.autograd.Function):
    """reference transformer.py:391-416: d(a.b^T) -> db = dw^T.a (TN), da = dw.b (NN)."""

    @staticmethod
    def forward(ctx, a, b, bst, c_dtype):
        ctx.bst = bst
        ctx.save_for_backward(a, b)
        return bst._nt(a, b, c_dtype)

    @staticmethod
    def backward(ctx, dw):
        a, b = ctx.saved_tensors
        bst = ctx.bst
        dw = dw.contiguous()
        db = bst._xn(dw, a, True) if ctx.needs_input_grad[1] else None
        da = bst._xn(dw, b, False) if ctx.needs_input_grad[0] else None
        return da, db, None, None


class _XnFunction(torch.autograd.Function):
    """reference transformer.py:423-449: y = w.v -> dv = w^T.dy (TN), dw = dy.v^T (NT)."""

    @staticmethod
    def forward(ctx, w, v, bst, transpose):
        ctx.bst, ctx.transpose = bst, transpose
        ctx.save_for_backward(w, v)
        return bst._xn(w, v, transpose)

    @staticmethod
    def backward(ctx, dy):
        w, v = ctx.saved_tensors
        bst = ctx.bst
        dy = dy.contiguous()
        dv = dw = None
        if ctx.needs_input_grad[1]:
            dv = bst._xn(w, dy, not ctx.transpose)
        if ctx.needs_input_grad[0]:
            # NN: dw[blk] = dy[q-blk] . v[k-blk]^T ; TN: dw[blk] = v[q-blk] . dy[k-blk]^T
            dw = bst._nt(v, dy, w.dtype) if ctx.transpose else bst._nt(dy, v, w.dtype)
        return dw, dv, None, None


class _SoftmaxFunction(torch.autograd.Function):
    """reference transformer.py:452-480."""

    @staticmethod
    def forward(ctx, x, bst, scale, use_mask, autoregress_at_key, dtype):
        y = bst._softmax(x, scale, use_mask, autoregress_at_key, dtype)
        ctx.bst, ctx.scale, ctx.x_dtype = bst, scale, x.dtype
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dx = ctx.bst._softmax_grad(dy, y, ctx.scale)
        return dx.to(ctx.x_dtype), None, None, None, None, None
