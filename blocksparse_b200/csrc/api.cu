// C ABI of libbsmm_b200.so -- argument validation and kernel-family dispatch.
// See include/bsmm_b200.h for the contract and the reference launchers each entry replaces.
#include "common.cuh"
#include "generic.cuh"
#include "softmax.cuh"
#include "tc.cuh"
#include "wutil.cuh"

using namespace bsmm;

extern "C" {

int bsmm_version(void) { return 1000 * 0 + 1; }
const char* bsmm_last_error(void) { return err_buf(); }
const char* bsmm_last_kernel(void) { return kernel_name_slot(); }

int bsmm_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  const DeviceInfo& d = device_info();
  if (!d.ok) return fail(BSMM_E_NODEV, "no CUDA device");
  if (sm_count) *sm_count = d.sm_count;
  if (cc_major) *cc_major = d.cc_major;
  if (cc_minor) *cc_minor = d.cc_minor;
  return 0;
}

int bsmm_device_error(void) {
  int v = 0, zero = 0;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { cudaGetLastError(); fail((int)e, "device fault: %s", cudaGetErrorString(e)); return -1; }
  if (cudaMemcpyFromSymbol(&v, g_tc_error, sizeof(int)) != cudaSuccess) return -1;
  if (v != 0) cudaMemcpyToSymbol(g_tc_error, &zero, sizeof(int));
  int wv = 0;
  if (cudaMemcpyFromSymbol(&wv, ptx::g_wait_error, sizeof(int)) != cudaSuccess) return -1;
  if (wv != 0) cudaMemcpyToSymbol(ptx::g_wait_error, &zero, sizeof(int));
  return v ? v : wv;
}

int bsmm_debug_trace(unsigned long long* out, int n) {
  unsigned long long* b = xprop2_trace_buffer();
  if (!b || !out || n <= 0 || n > 256 * 8) return fail(BSMM_E_ARG, "bsmm_debug_trace: tracing is off (BSMM_TRACE) or bad arguments");
  cudaError_t e = cudaMemcpy(out, b, (size_t)n * 8, cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? 0 : fail((int)e, "bsmm_debug_trace: %s", cudaGetErrorString(e));
}

int bsmm_set_wait_timeout_ms(int ms, int trap) {
  if (ms <= 0) return fail(BSMM_E_ARG, "bsmm_set_wait_timeout_ms: ms must be positive");
  const unsigned long long ns = (unsigned long long)ms * 1000000ull;
  const int t = trap ? 1 : 0;
  cudaError_t e = cudaMemcpyToSymbol(ptx::g_wait_timeout_ns, &ns, sizeof(ns));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(ptx::g_wait_trap, &t, sizeof(t));
  if (e != cudaSuccess) { cudaGetLastError(); return fail((int)e, "bsmm_set_wait_timeout_ms: %s", cudaGetErrorString(e)); }
  return 0;
}

// ---------------------------------------------------------------------------------------
// A 16-bit call that cannot take the tcgen05 kernel runs ~25x slower on the CUDA-core path: say so once per process (the
// reason is whatever tc_* recorded), unless BSMM_QUIET is set.  fp32 calls are expected there and stay silent.
static void note_fallback(const char* op, int dtype) {
  static std::atomic<bool> warned{false};
  if (dtype == BSMM_F32 || warned.exchange(true)) return;
  if (getenv("BSMM_QUIET")) return;
  fprintf(stderr, "[bsmm_b200] %s: no tensor-core kernel for this call (%s); using the CUDA-core FMA kernel (about 25x slower). "
                  "This message is printed once.\n", op, err_buf());
}

static int check_bsize_axis(int bsize, int axis) {
  if (axis != 0 && axis != 1) return fail(BSMM_E_BSIZE, "feature axis must be 0 or 1, got %d", axis);
  if (bsize != 8 && bsize != 16 && bsize != 32 && bsize != 64)
    return fail(BSMM_E_BSIZE, "block size must be 8, 16, 32 or 64, got %d", bsize);
  return 0;
}

int bsmm_xprop(int dtype, int axis, int bsize, int bprop,
               const int32_t* lut, int n_out, int n_in, int blocks,
               const void* x, const void* w, void* y, int N,
               const float* gate,
               const int32_t* sched, int sched_tiles, int sched_tile_blocks, int sched_groups_off,
               int sched_list_off, int sched_ctas, int sched_ntiles,
               int flags, void* stream) {
  if (int e = check_bsize_axis(bsize, axis)) return e;
  if (!lut || !x || !w || !y) return fail(BSMM_E_ARG, "bsmm_xprop: null pointer");
  if (n_out <= 0 || n_in <= 0 || blocks < 0 || N < 0) return fail(BSMM_E_ARG, "bsmm_xprop: bad sizes");
  // reference limit: C, K < bsize*65536 (src/blocksparse_matmul_op.cc:96-97)
  if (n_out >= 65536 || n_in >= 65536) return fail(BSMM_E_LIMIT, "bsmm_xprop: more than 65535 blocks per dimension");
  if (N == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;

  if (!(flags & BSMM_FLAG_FORCE_GENERIC)) {
    int rc;
    if ((sched_tile_blocks >> 16) & 1)       // pair schedule (lut.py:build_pair_schedule) -> csrc/tc_xprop2.cuh
      rc = tc_xprop2(dtype, axis, bprop, n_out, n_in, blocks, x, w, y, N, sched, sched_tiles, (sched_tile_blocks >> 8) & 0xff,
                     sched_groups_off, sched_list_off, sched_ctas, sched_ntiles, s);
    else                                      // sched_list_off = optional tile order table (heaviest first) for sched_ntiles minibatch tiles
      rc = tc_xprop(dtype, axis, bsize, bprop, lut, n_out, n_in, blocks, x, w, y, N, gate, sched, sched_tiles, sched_tile_blocks & 0xffff,
                    sched_groups_off, sched_list_off, sched_ntiles, s);
    if (rc != TC_NOT_APPLICABLE) return rc;
    if (flags & BSMM_FLAG_FORCE_TC)
      return fail(BSMM_E_ARG, "bsmm_xprop: no tcgen05 kernel for dtype=%d axis=%d bsize=%d (%s)", dtype, axis, bsize, err_buf());
    note_fallback("bsmm_xprop", dtype);
  } else if (flags & BSMM_FLAG_FORCE_TC) {
    return fail(BSMM_E_ARG, "bsmm_xprop: contradictory flags");
  }

  XnParams p = {};
  p.lut = lut; p.lut_head_stride = 0; p.n_out = n_out;
  p.w = w; p.w_z_stride = 0;
  p.x = x; p.y = y;
  p.heads = 1; p.N = N; p.gate = gate;
  if (axis == 0) { p.x_sf = N; p.x_sn = 1; p.y_sf = N; p.y_sn = 1; }
  else { p.x_sf = 1; p.x_sn = (long long)n_in * bsize; p.y_sf = 1; p.y_sn = (long long)n_out * bsize; }
  // Wm[fi][fo]: fprop uses W[fi][fo] directly, bprop needs the transpose.
  const bool trans_w = bprop != 0;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    BSMM_DISPATCH_BSIZE(bsize, BS, { return launch_sdd_xn<T, T, BS>(p, axis == 1, trans_w, 1, s); });
  });
  return 0;
}

int bsmm_updat(int dtype, int dw_dtype, int axis, int bsize,
               const int32_t* updat_lut, int blocks, int n_c_blocks, int n_k_blocks,
               const void* const* xs, const void* const* dys, int pcount,
               void* dw, int N, float alpha, float beta,
               const float* gate, int gated_dw,
               const int32_t* sched, int sched_tiles, int sched_tile_blocks, int sched_groups_off,
               int flags, void* stream) {
  if (int e = check_bsize_axis(bsize, axis)) return e;
  if (!updat_lut || !xs || !dys || !dw) return fail(BSMM_E_ARG, "bsmm_updat: null pointer");
  if (pcount < 1 || pcount > BSMM_MAX_PAIRS)
    return fail(BSMM_E_ARG, "bsmm_updat: pcount must be in [1,%d], got %d", BSMM_MAX_PAIRS, pcount);
  if (beta != 0.f && beta != 1.f) return fail(BSMM_E_ARG, "bsmm_updat: beta must be 0 or 1");
  if (dw_dtype != dtype && dw_dtype != BSMM_F32) return fail(BSMM_E_DTYPE, "bsmm_updat: dw dtype must be fp32 or the input dtype");
  if (blocks <= 0 || N < 0) return fail(BSMM_E_ARG, "bsmm_updat: bad sizes");
  for (int i = 0; i < pcount; ++i)
    if (!xs[i] || !dys[i]) return fail(BSMM_E_ARG, "bsmm_updat: null pointer in pair %d", i);
  cudaStream_t s = (cudaStream_t)stream;

  if (!(flags & BSMM_FLAG_FORCE_GENERIC)) {
    int rc = tc_updat(dtype, dw_dtype, axis, bsize, updat_lut, blocks, n_c_blocks, n_k_blocks, xs, dys, pcount,
                      dw, N, alpha, beta, gate, gated_dw, sched, sched_tiles, sched_tile_blocks, sched_groups_off, s);
    if (rc != TC_NOT_APPLICABLE) return rc;
    if (flags & BSMM_FLAG_FORCE_TC)
      return fail(BSMM_E_ARG, "bsmm_updat: no tcgen05 kernel for dtype=%d axis=%d bsize=%d (%s)", dtype, axis, bsize, err_buf());
    note_fallback("bsmm_updat", dtype);
  }

  NtParams p = {};
  p.lut = updat_lut; p.lut_head_stride = 0; p.blocks = blocks;
  for (int i = 0; i < pcount; ++i) { p.a[i] = xs[i]; p.b[i] = dys[i]; }
  p.pcount = pcount; p.out = dw; p.out_z_stride = 0;
  p.R = N; p.heads = 1; p.alpha = alpha; p.beta = beta; p.gate = gate; p.gated = gated_dw && gate;
  if (axis == 0) { p.a_sf = N; p.a_sr = 1; p.b_sf = N; p.b_sr = 1; }
  else { p.a_sf = 1; p.a_sr = (long long)n_c_blocks * bsize; p.b_sf = 1; p.b_sr = (long long)n_k_blocks * bsize; }
  BSMM_DISPATCH_DTYPE(dtype, T, {
    BSMM_DISPATCH_BSIZE(bsize, BS, {
      if (dw_dtype == BSMM_F32) return launch_dds_nt<T, float, BS>(p, axis == 1, 1, s);
      else                      return launch_dds_nt<T, T, BS>(p, axis == 1, 1, s);
    });
  });
  return 0;
}

int bsmm_gate_grad(int dtype, int bsize, int blocks, const void* dw, const void* w, float* dg, void* stream) {
  if (!dw || !w || !dg || blocks <= 0) return fail(BSMM_E_ARG, "bsmm_gate_grad: bad arguments");
  if (int e = check_bsize_axis(bsize, 0)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  const int warps = 4;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    gate_grad_kernel<T><<<(blocks + warps - 1) / warps, warps * 32, 0, s>>>(
        (const T*)dw, (const T*)w, dg, blocks, bsize * bsize);
  });
  return check_launch("gate_grad");
}

int bsmm_gate_weights(int dtype, int bsize, int blocks, const void* w, const float* gate, void* w_out, void* stream) {
  if (!w || !gate || !w_out || blocks <= 0) return fail(BSMM_E_ARG, "bsmm_gate_weights: bad arguments");
  if (int e = check_bsize_axis(bsize, 0)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  const long long total = (long long)blocks * bsize * bsize;
  const int threads = 256;
  const long long grid = (total / 2 + threads - 1) / threads;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    gate_weights_kernel<T><<<(unsigned)grid, threads, 0, s>>>((const T*)w, gate, (T*)w_out, total, bsize * bsize);
  });
  return check_launch("gate_weights");
}

// ---------------------------------------------------------------------------------------
static int check_bst(int bsize, int lut_heads, int heads, int head_state, int batch, int blocks) {
  if (bsize != 8 && bsize != 16 && bsize != 32 && bsize != 64)
    return fail(BSMM_E_BSIZE, "block size must be 8, 16, 32 or 64, got %d", bsize);
  if (lut_heads != 1 && lut_heads != heads) return fail(BSMM_E_ARG, "lut_heads must be 1 or heads");
  if (batch <= 0 || heads <= 0 || blocks <= 0) return fail(BSMM_E_ARG, "bad batch/heads/blocks");
  if (head_state <= 0 || (head_state & 7)) return fail(BSMM_E_ARG, "head_state must be a positive multiple of 8 (bst_op.cc:208)");
  return 0;
}

int bst_nt(int dtype, int c_dtype, int bsize,
           const int32_t* nt_lut, int lut_heads, int blocks,
           const int32_t* nt_items, int n_items,
           const void* a, const void* b, void* c,
           int batch, int heads, int head_state, int ctx_blks_a, int ctx_blks_b,
           int flags, void* stream) {
  if (int e = check_bst(bsize, lut_heads, heads, head_state, batch, blocks)) return e;
  if (!nt_lut || !a || !b || !c) return fail(BSMM_E_ARG, "bst_nt: null pointer");
  // attention tensor must have < 2^32 elements (bst_op.cc:214)
  if ((unsigned long long)batch * heads * blocks * bsize * bsize >= (1ull << 32))
    return fail(BSMM_E_LIMIT, "bst_nt: output has >= 2^32 elements");
  cudaStream_t s = (cudaStream_t)stream;

  if (!(flags & BSMM_FLAG_FORCE_GENERIC)) {
    int rc = tc_bst_nt(dtype, c_dtype, bsize, nt_items, n_items, lut_heads, blocks, a, b, c, batch, heads, head_state,
                       ctx_blks_a, ctx_blks_b, s);
    if (rc != TC_NOT_APPLICABLE) return rc;
    if (flags & BSMM_FLAG_FORCE_TC) return fail(BSMM_E_ARG, "bst_nt: no tcgen05 kernel for this configuration (%s)", err_buf());
  }

  const long long S = (long long)heads * head_state;
  NtParams p = {};
  p.lut = nt_lut; p.lut_head_stride = lut_heads > 1 ? 2LL * blocks : 0; p.blocks = blocks;
  p.a[0] = a; p.b[0] = b; p.pcount = 1; p.out = c;
  p.a_zb = (long long)ctx_blks_a * bsize * S; p.a_zh = head_state;
  p.b_zb = (long long)ctx_blks_b * bsize * S; p.b_zh = head_state;
  p.a_sf = S; p.a_sr = 1; p.b_sf = S; p.b_sr = 1;
  p.out_z_stride = (long long)blocks * bsize * bsize;
  p.R = head_state; p.heads = heads; p.alpha = 1.f; p.beta = 0.f; p.gate = nullptr; p.gated = 0;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    BSMM_DISPATCH_DTYPE(c_dtype, TC, {
      BSMM_DISPATCH_BSIZE(bsize, BS, { return launch_dds_nt<T, TC, BS>(p, false, batch * heads, s); });
    });
  });
  return 0;
}

int bst_xn(int a_dtype, int dtype, int bsize, int transpose_a,
           const int32_t* lut, const int32_t* out_order, int lut_heads, int blocks, int max_lut,
           const void* a, const void* b, void* c,
           int batch, int heads, int head_state, int ctx_blks_b, int ctx_blks_c,
           int flags, void* stream) {
  if (int e = check_bst(bsize, lut_heads, heads, head_state, batch, blocks)) return e;
  if (!lut || !a || !b || !c) return fail(BSMM_E_ARG, "bst_xn: null pointer");
  cudaStream_t s = (cudaStream_t)stream;

  if (!(flags & BSMM_FLAG_FORCE_GENERIC)) {
    int rc = tc_bst_xn(a_dtype, dtype, bsize, transpose_a, lut, out_order, lut_heads, blocks, max_lut, a, b, c, batch, heads,
                       head_state, ctx_blks_b, ctx_blks_c, s);
    if (rc != TC_NOT_APPLICABLE) return rc;
    if (flags & BSMM_FLAG_FORCE_TC) return fail(BSMM_E_ARG, "bst_xn: no tcgen05 kernel for this configuration (%s)", err_buf());
  }

  const long long S = (long long)heads * head_state;
  XnParams p = {};
  p.lut = lut; p.lut_head_stride = lut_heads > 1 ? 2LL * (ctx_blks_c + blocks) : 0; p.n_out = ctx_blks_c;
  p.w = a; p.w_z_stride = (long long)blocks * bsize * bsize;
  p.x = b; p.y = c;
  p.x_zb = (long long)ctx_blks_b * bsize * S; p.x_zh = head_state;
  p.y_zb = (long long)ctx_blks_c * bsize * S; p.y_zh = head_state;
  p.x_sf = S; p.x_sn = 1; p.y_sf = S; p.y_sn = 1;
  p.N = head_state; p.heads = heads; p.gate = nullptr;
  // NN: out row i of A (fo = i, fi = j) -> transposed staging; TN: fo = j, fi = i -> direct.
  const bool trans_w = transpose_a == 0;
  BSMM_DISPATCH_DTYPE(a_dtype, TA, {
    BSMM_DISPATCH_DTYPE(dtype, T, {
      BSMM_DISPATCH_BSIZE(bsize, BS, { return launch_sdd_xn<TA, T, BS>(p, false, trans_w, batch * heads, s); });
    });
  });
  return 0;
}

int bst_softmax(int x_dtype, int y_dtype, int bsize,
                const int32_t* nn_lut, const int32_t* nt_lut, int lut_heads, int blocks, int max_lut,
                const void* mask, int mask_heads, int autoregress_at_key,
                const void* x, void* y, float scale,
                int batch, int heads, int ctx_blks_q, void* stream) {
  if (int e = check_bst(bsize, lut_heads, heads, 8, batch, blocks)) return e;
  if (!nn_lut || !x || !y) return fail(BSMM_E_ARG, "bst_softmax: null pointer");
  if ((long long)max_lut * bsize > 32768) return fail(BSMM_E_LIMIT, "bst_softmax: max_lut*bsize > 32768 (bst_op.cc:383)");
  if (autoregress_at_key >= 0 && (!mask || !nt_lut))
    return fail(BSMM_E_ARG, "bst_softmax: autoregress_at_key needs a mask and nt_lut");
  if (mask && mask_heads != 1 && mask_heads != heads) return fail(BSMM_E_ARG, "bst_softmax: mask_heads must be 1 or heads");
  cudaStream_t s = (cudaStream_t)stream;
  SoftmaxParams p = {};
  p.nn_lut = nn_lut; p.nt_lut = nt_lut;
  p.nn_head_stride = lut_heads > 1 ? 2LL * (ctx_blks_q + blocks) : 0;
  p.nt_head_stride = lut_heads > 1 ? 2LL * blocks : 0;
  p.mask = mask; p.mask_head_stride = (mask && mask_heads > 1) ? (long long)blocks * bsize : 0;
  p.autoregress_at_key = autoregress_at_key;
  p.x = x; p.y = y; p.scale = scale;
  p.batch = batch; p.heads = heads; p.blocks = blocks; p.ctx_blks_q = ctx_blks_q;
  // TMA-staged kernel: 16-bit tensors, 32 x 32 / 64 x 64 blocks, every row's blocks fit shared memory (<= 16 of them), and
  // 16-byte-aligned x and y (bulk copies).  Everything else takes the register kernel, which needs x and y aligned to its
  // vector accesses (softmax_vec_bytes); a misaligned pointer is refused there rather than faulting in the kernel.
  static const bool no_staged = [] { const char* e = getenv("BSMM_SOFTMAX_STAGED"); return e && atoi(e) == 0; }();
  if (!no_staged && x_dtype != BSMM_F32 && y_dtype != BSMM_F32 && (bsize == 32 || bsize == 64) && max_lut >= 1 && max_lut <= 16 &&
      (((uintptr_t)x | (uintptr_t)y) & 15) == 0 && device_info().ok && device_info().cc_major >= 9) {
#define BSMM_SM_STAGED(TXT, TYT)                                                                              \
    return bsize == 64 ? launch_softmax_staged<TXT, TYT, 64>(p, max_lut, s) : launch_softmax_staged<TXT, TYT, 32>(p, max_lut, s);
    if (x_dtype == BSMM_BF16 && y_dtype == BSMM_BF16) { BSMM_SM_STAGED(__nv_bfloat16, __nv_bfloat16) }
    if (x_dtype == BSMM_BF16 && y_dtype == BSMM_F16)  { BSMM_SM_STAGED(__nv_bfloat16, __half) }
    if (x_dtype == BSMM_F16 && y_dtype == BSMM_F16)   { BSMM_SM_STAGED(__half, __half) }
    if (x_dtype == BSMM_F16 && y_dtype == BSMM_BF16)  { BSMM_SM_STAGED(__half, __nv_bfloat16) }
#undef BSMM_SM_STAGED
  }
  BSMM_DISPATCH_DTYPE(x_dtype, TX, {
    BSMM_DISPATCH_DTYPE(y_dtype, TY, {
      BSMM_DISPATCH_BSIZE(bsize, BS, {
        if (!softmax_aligned<TX, BS>(x) || !softmax_aligned<TY, BS>(y))
          return fail(BSMM_E_ARG, "bst_softmax: x and y must be aligned to %d / %d bytes", softmax_vec_bytes<TX, BS>(),
                      softmax_vec_bytes<TY, BS>());
        const long long groups = (long long)ctx_blks_q * SoftmaxMap<BS>::GROUPS;
        dim3 grid((unsigned)((groups + SOFTMAX_WARPS - 1) / SOFTMAX_WARPS), heads, batch);
        bst_softmax_kernel<TX, TY, BS><<<grid, SOFTMAX_WARPS * 32, 0, s>>>(p);
      });
    });
  });
  return check_launch("bst_softmax");
}

int bst_softmax_grad(int dtype, int dx_dtype, int bsize,
                     const int32_t* nn_lut, int lut_heads, int blocks, int max_lut,
                     const void* dy, const void* y, void* dx, float scale,
                     int batch, int heads, int ctx_blks_q, void* stream) {
  if (int e = check_bst(bsize, lut_heads, heads, 8, batch, blocks)) return e;
  if (!nn_lut || !dy || !y || !dx) return fail(BSMM_E_ARG, "bst_softmax_grad: null pointer");
  if ((long long)max_lut * bsize > 32768) return fail(BSMM_E_LIMIT, "bst_softmax_grad: max_lut*bsize > 32768");
  cudaStream_t s = (cudaStream_t)stream;
  SoftmaxParams p = {};
  p.nn_lut = nn_lut;
  p.nn_head_stride = lut_heads > 1 ? 2LL * (ctx_blks_q + blocks) : 0;
  p.x = dy; p.y_in = y; p.y = dx; p.scale = scale;
  p.batch = batch; p.heads = heads; p.blocks = blocks; p.ctx_blks_q = ctx_blks_q;
  static const bool no_staged = [] { const char* e = getenv("BSMM_SOFTMAX_STAGED"); return e && atoi(e) == 0; }();
  if (!no_staged && dtype != BSMM_F32 && dx_dtype != BSMM_F32 && (bsize == 32 || bsize == 64) && max_lut >= 1 && max_lut <= 16 &&
      (((uintptr_t)dy | (uintptr_t)y | (uintptr_t)dx) & 15) == 0 && device_info().ok && device_info().cc_major >= 9) {
#define BSMM_SG_STAGED(TT, TDT)                                                                               \
    return bsize == 64 ? launch_softmax_grad_staged<TT, TDT, 64>(p, max_lut, s) : launch_softmax_grad_staged<TT, TDT, 32>(p, max_lut, s);
    if (dtype == BSMM_BF16 && dx_dtype == BSMM_BF16) { BSMM_SG_STAGED(__nv_bfloat16, __nv_bfloat16) }
    if (dtype == BSMM_F16 && dx_dtype == BSMM_F16)   { BSMM_SG_STAGED(__half, __half) }
    if (dtype == BSMM_F16 && dx_dtype == BSMM_BF16)  { BSMM_SG_STAGED(__half, __nv_bfloat16) }
    if (dtype == BSMM_BF16 && dx_dtype == BSMM_F16)  { BSMM_SG_STAGED(__nv_bfloat16, __half) }
#undef BSMM_SG_STAGED
  }
  BSMM_DISPATCH_DTYPE(dtype, T, {
    BSMM_DISPATCH_DTYPE(dx_dtype, TD, {
      BSMM_DISPATCH_BSIZE(bsize, BS, {
        if (!softmax_aligned<T, BS>(dy) || !softmax_aligned<T, BS>(y) || !softmax_aligned<TD, BS>(dx))
          return fail(BSMM_E_ARG, "bst_softmax_grad: dy, y and dx must be aligned to %d / %d bytes", softmax_vec_bytes<T, BS>(),
                      softmax_vec_bytes<TD, BS>());
        const long long groups = (long long)ctx_blks_q * SoftmaxMap<BS>::GROUPS;
        dim3 grid((unsigned)((groups + SOFTMAX_WARPS - 1) / SOFTMAX_WARPS), heads, batch);
        bst_softmax_grad_kernel<T, TD, BS><<<grid, SOFTMAX_WARPS * 32, 0, s>>>(p);
      });
    });
  });
  return check_launch("bst_softmax_grad");
}

int bst_autoregressive_mask(int bsize, const int32_t* nt_lut, int lut_heads, int blocks,
                            const void* mask_in, void* mask_out, int autoregress_at_key, void* stream) {
  if (!nt_lut || !mask_in || !mask_out || lut_heads <= 0 || blocks <= 0)
    return fail(BSMM_E_ARG, "bst_autoregressive_mask: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  dim3 grid((blocks * bsize + 127) / 128, lut_heads);
  BSMM_DISPATCH_BSIZE(bsize, BS, {
    bst_autoregressive_mask_kernel<BS><<<grid, 128, 0, s>>>(nt_lut, lut_heads > 1 ? 2LL * blocks : 0,
                                                            mask_in, mask_out, blocks, autoregress_at_key);
  });
  return check_launch("bst_autoregressive_mask");
}

// ---------------------------------------------------------------------------------------
struct Timer { cudaEvent_t start, stop; };

int bsmm_timer_create(void** timer) {
  if (!timer) return fail(BSMM_E_ARG, "null timer");
  Timer* t = new Timer;
  if (cudaEventCreate(&t->start) != cudaSuccess || cudaEventCreate(&t->stop) != cudaSuccess) {
    delete t;
    return fail(BSMM_E_NODEV, "cudaEventCreate failed");
  }
  *timer = t;
  return 0;
}
int bsmm_timer_begin(void* timer, void* stream) {
  if (!timer) return fail(BSMM_E_ARG, "null timer");
  return (int)cudaEventRecord(((Timer*)timer)->start, (cudaStream_t)stream);
}
int bsmm_timer_end(void* timer, void* stream, float* ms_out) {
  if (!timer || !ms_out) return fail(BSMM_E_ARG, "null timer");
  Timer* t = (Timer*)timer;
  cudaError_t e = cudaEventRecord(t->stop, (cudaStream_t)stream);
  if (e == cudaSuccess) e = cudaEventSynchronize(t->stop);
  if (e == cudaSuccess) e = cudaEventElapsedTime(ms_out, t->start, t->stop);
  if (e != cudaSuccess) return fail((int)e, "timer: %s", cudaGetErrorString(e));
  return 0;
}
int bsmm_timer_destroy(void* timer) {
  if (!timer) return 0;
  Timer* t = (Timer*)timer;
  cudaEventDestroy(t->start); cudaEventDestroy(t->stop);
  delete t;
  return 0;
}


// ---- weight utilities (csrc/wutil.cuh) ---------------------------------------------------------------------------
static int check_blocks(const char* what, int bsize, int blocks, const void* p) {
  if (!p || blocks <= 0) return fail(BSMM_E_ARG, "%s: bad arguments", what);
  return check_bsize_axis(bsize, 0);
}

int bsmm_block_norm(int dtype, int bsize, int blocks, const void* w, float* norm, int norm_type, void* stream) {
  if (int e = check_blocks("bsmm_block_norm", bsize, blocks, w)) return e;
  if (!norm) return fail(BSMM_E_ARG, "bsmm_block_norm: null output");
  const int wpb = 4;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    block_norm_kernel<T><<<(blocks + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>((const T*)w, norm, blocks, bsize * bsize, norm_type != 0);
  });
  return check_launch("block_norm");
}

int bsmm_l2_decay(int dtype, int bsize, int blocks, void* w, const float* gate, float rate, float epsilon, void* stream) {
  if (int e = check_blocks("bsmm_l2_decay", bsize, blocks, w)) return e;
  const int wpb = 4;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    l2_decay_kernel<T><<<(blocks + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>((T*)w, gate, blocks, bsize * bsize, rate, epsilon);
  });
  return check_launch("l2_decay");
}

int bsmm_threshold_prune(int dtype, int bsize, int blocks, const void* w, float* gate, float threshold, int norm_type, void* stream) {
  if (int e = check_blocks("bsmm_threshold_prune", bsize, blocks, w)) return e;
  if (!gate) return fail(BSMM_E_ARG, "bsmm_threshold_prune: null gate");
  const int wpb = 4;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    threshold_prune_kernel<T><<<(blocks + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>((const T*)w, gate, blocks, bsize * bsize, threshold, norm_type != 0);
  });
  return check_launch("threshold_prune");
}

int bsmm_prune_topk(float* gate, const int32_t* idx, int blocks, int keep, void* stream) {
  if (!gate || !idx || blocks <= 0 || keep < 0) return fail(BSMM_E_ARG, "bsmm_prune_topk: bad arguments");
  prune_topk_kernel<<<(blocks + 255) / 256, 256, 0, (cudaStream_t)stream>>>(gate, idx, blocks, keep);
  return check_launch("prune_topk");
}

int bsmm_identity_init(int dtype, int bsize, int blocks, const int32_t* updat_lut, int n_c_blocks, int n_k_blocks, void* w, float scale, void* stream) {
  if (int e = check_blocks("bsmm_identity_init", bsize, blocks, w)) return e;
  if (!updat_lut || n_c_blocks <= 0 || n_k_blocks <= 0) return fail(BSMM_E_ARG, "bsmm_identity_init: bad arguments");
  BSMM_DISPATCH_DTYPE(dtype, T, {
    identity_init_kernel<T><<<blocks, 128, 0, (cudaStream_t)stream>>>((T*)w, updat_lut, blocks, bsize, n_c_blocks, n_k_blocks, scale);
  });
  return check_launch("identity_init");
}

int bsmm_l2_normalize(int dtype, int y_dtype, int bsize, const int32_t* lut, int n_out, const void* w, const float* gain, void* y,
                      float* sum_sqr, float epsilon, void* stream) {
  if (int e = check_bsize_axis(bsize, 0)) return e;
  if (!lut || !w || !y || !sum_sqr || n_out <= 0) return fail(BSMM_E_ARG, "bsmm_l2_normalize: bad arguments");
  if (y_dtype != dtype && y_dtype != BSMM_F32) return fail(BSMM_E_DTYPE, "bsmm_l2_normalize: output dtype must be fp32 or the input dtype");
  cudaStream_t s = (cudaStream_t)stream;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    if (y_dtype == BSMM_F32) l2_normalize_kernel<T, float><<<n_out, L2N_THREADS, 0, s>>>((const T*)w, gain, (float*)y, sum_sqr, lut, bsize, epsilon);
    else                     l2_normalize_kernel<T, T><<<n_out, L2N_THREADS, 0, s>>>((const T*)w, gain, (T*)y, sum_sqr, lut, bsize, epsilon);
  });
  return check_launch("l2_normalize");
}

int bsmm_l2_normalize_grad(int dtype, int y_dtype, int bsize, const int32_t* lut, int n_out, const void* dy, const void* w, const float* gain,
                           const float* sum_sqr, void* dx, float* dg, float epsilon, void* stream) {
  if (int e = check_bsize_axis(bsize, 0)) return e;
  if (!lut || !dy || !w || !sum_sqr || !dx || n_out <= 0) return fail(BSMM_E_ARG, "bsmm_l2_normalize_grad: bad arguments");
  if (y_dtype != dtype && y_dtype != BSMM_F32) return fail(BSMM_E_DTYPE, "bsmm_l2_normalize_grad: dy dtype must be fp32 or the weight dtype");
  cudaStream_t s = (cudaStream_t)stream;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    if (y_dtype == BSMM_F32) l2_normalize_grad_kernel<T, float><<<n_out, L2N_THREADS, 0, s>>>((const float*)dy, (const T*)w, gain, sum_sqr, (T*)dx, dg, lut, bsize, epsilon);
    else                     l2_normalize_grad_kernel<T, T><<<n_out, L2N_THREADS, 0, s>>>((const T*)dy, (const T*)w, gain, sum_sqr, (T*)dx, dg, lut, bsize, epsilon);
  });
  return check_launch("l2_normalize_grad");
}

size_t bsmm_reduced_dw_workspace_bytes(int n_c_blocks, int n_k_blocks) { return (size_t)8 * n_c_blocks * n_k_blocks * sizeof(float); }

int bsmm_reduced_dw(int dtype, int axis, int bsize, const void* const* xs, const void* const* dys, int pcount,
                    int n_c_blocks, int n_k_blocks, int N, float scale, int norm_type, float* dw, int accumulate,
                    void* x_red, void* y_red, void* workspace, void* stream) {
  if (int e = check_bsize_axis(bsize, axis)) return e;
  if (!xs || !dys || !dw || !x_red || !y_red || !workspace) return fail(BSMM_E_ARG, "bsmm_reduced_dw: null pointer");
  if (pcount < 1 || pcount > BSMM_MAX_PAIRS || n_c_blocks <= 0 || n_k_blocks <= 0 || N <= 0) return fail(BSMM_E_ARG, "bsmm_reduced_dw: bad sizes");
  if (dtype == BSMM_F32) return fail(BSMM_E_DTYPE, "bsmm_reduced_dw: 16-bit activations only (reference: half)");
  cudaStream_t s = (cudaStream_t)stream;
  const int l2 = norm_type != 0;
  const int splits = 8;
  BSMM_DISPATCH_DTYPE(dtype, T, {
    if (scale != 0.0f) {        // a zero scale skips the reductions (reference op.cc:754-766)
      for (int p = 0; p < pcount; ++p) {
        if (!xs[p] || !dys[p]) return fail(BSMM_E_ARG, "bsmm_reduced_dw: null pointer in pair %d", p);
        const long long tx = (long long)n_c_blocks * N, ty = (long long)n_k_blocks * N;
        feature_reduce_kernel<T><<<(unsigned)((tx + 255) / 256), 256, 0, s>>>((const T*)xs[p], (T*)x_red, axis, bsize, n_c_blocks, N, p, pcount, l2);
        feature_reduce_kernel<T><<<(unsigned)((ty + 255) / 256), 256, 0, s>>>((const T*)dys[p], (T*)y_red, axis, bsize, n_k_blocks, N, p, pcount, l2);
      }
    }
    const long long R = (long long)pcount * N;
    dim3 grid((n_c_blocks + 15) / 16, (n_k_blocks + 15) / 16, splits);
    if (axis == 1)     // (pair, n, block): row r = pair*N + n, block contiguous
      reduced_gemm_partial_kernel<T><<<grid, 256, 0, s>>>((const T*)x_red, (const T*)y_red, (float*)workspace, n_c_blocks, n_k_blocks, R,
                                                          n_c_blocks, 1, n_k_blocks, 1, splits);
    else               // (block, pair, n): row r = pair*N + n contiguous, block stride R
      reduced_gemm_partial_kernel<T><<<grid, 256, 0, s>>>((const T*)x_red, (const T*)y_red, (float*)workspace, n_c_blocks, n_k_blocks, R,
                                                          1, R, 1, R, splits);
  });
  const int total = n_c_blocks * n_k_blocks;
  reduced_gemm_finish_kernel<<<(total + 255) / 256, 256, 0, s>>>((const float*)workspace, dw, total, splits, scale, accumulate);
  return check_launch("reduced_dw");
}

int bsmm_gather_rows(int dtype, const void* x, const void* y, const int32_t* idx, void* out, int rows, long long N, int op, void* stream) {
  if (!x || !idx || !out || rows <= 0 || N <= 0 || op < 0 || op > 2 || (op != 0 && !y)) return fail(BSMM_E_ARG, "bsmm_gather_rows: bad arguments");
  const unsigned gx = (unsigned)((N + 255) / 256 > 64 ? 64 : (N + 255) / 256);
  BSMM_DISPATCH_DTYPE(dtype, T, {
    gather_rows_kernel<T><<<dim3(gx, rows), 256, 0, (cudaStream_t)stream>>>((const T*)x, (const T*)y, idx, (T*)out, rows, N, op);
  });
  return check_launch("gather_rows");
}

int bsmm_pad_blocks(int dtype, int bsize, int blocks_big, const int32_t* sub_map, const void* w_small, const float* gate, void* w_big, void* stream) {
  if (!sub_map || !w_small || !w_big || blocks_big <= 0 || (bsize != 8 && bsize != 16 && bsize != 32)) return fail(BSMM_E_ARG, "bsmm_pad_blocks: bad arguments");
  BSMM_DISPATCH_DTYPE(dtype, T, {
    pad_blocks_kernel<T><<<blocks_big, 128, 0, (cudaStream_t)stream>>>((const T*)w_small, sub_map, gate, (T*)w_big, blocks_big, bsize);
  });
  return check_launch("pad_blocks");
}

int bsmm_unpad_blocks(int in_dtype, int out_dtype, int bsize, int blocks_small, const int32_t* inv_map, const void* dw_big, const float* gate,
                      void* dw_small, int accumulate, void* stream) {
  if (!inv_map || !dw_big || !dw_small || blocks_small <= 0 || (bsize != 8 && bsize != 16 && bsize != 32)) return fail(BSMM_E_ARG, "bsmm_unpad_blocks: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  BSMM_DISPATCH_DTYPE(in_dtype, TI, {
    BSMM_DISPATCH_DTYPE(out_dtype, TO, {
      unpad_blocks_kernel<TI, TO><<<blocks_small, 64, 0, s>>>((const TI*)dw_big, inv_map, gate, (TO*)dw_small, blocks_small, bsize, accumulate);
    });
  });
  return check_launch("unpad_blocks");
}
}  // extern "C"
