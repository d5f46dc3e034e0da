/*
 * bsmm_b200.h -- C ABI of libbsmm_b200.so: block-sparse matmul (fprop / bprop / updat)
 * and block-sparse transformer ops (NT / NN / TN, masked softmax, softmax grad,
 * partial autoregressive mask) for NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the hot path of openai/blocksparse.  Each entry
 * point replaces one host launcher that the reference's TensorFlow OpKernels call
 * (file:line relative to the reference tree):
 *
 *   bsmm_xprop            <- hgemm_blocksparse_xn_{64,128}_sdd / hgemm_blocksparse_nx_dsd /
 *                            BsmmXprop_CN   (src/blocksparse_matmul_op.cc:49-68,185-215)
 *   bsmm_updat            <- hgemm_blocksparse_nt_{64,128}_dds / hgemm_blocksparse_tn_dds /
 *                            BsmmUpdat_CN   (src/blocksparse_matmul_op.cc:223-311)
 *   bsmm_gate_grad        <- BlocksparseGateGrad (src/blocksparse_matmul_op.cc:490-540)
 *   bsmm_gate_weights     <- the gate scaling inside the reference's gated xprop kernels (cn_64.cu:96-98)
 *   bst_nt                <- bst_hgemm_nt / bst_sgemm_nt   (src/bst_op.cc:139-144,183-250)
 *   bst_xn                <- bst_hgemm_xn / bst_sgemm_xn   (src/bst_op.cc:251-320)
 *   bst_softmax           <- BlocksparseMaskedSoftmax<T,V> (src/bst_op.cc:331-340,374-428)
 *   bst_softmax_grad      <- BlocksparseSoftmaxGrad<T,V>   (src/bst_op.cc:443-512)
 *   bst_autoregressive_mask <- BstPartialAutoregressiveMask (src/bst_op.cc:519-575)
 *   bsmm_block_norm / bsmm_l2_decay / bsmm_threshold_prune / bsmm_prune_topk
 *                         <- BlocksparseNorm / BlocksparseL2Decay / BlocksparseThresholdPrune / BlocksparsePrune
 *                            (src/optimize_op_gpu.cu:794-1098)
 *   bsmm_identity_init    <- IdentityInitCK (src/blocksparse_matmul_op_gpu.cu:2988-3028)
 *   bsmm_l2_normalize(_grad) <- L2NormalizeCK / L2NormalizeGainCK and their gradients
 *                            (src/blocksparse_l2_norm_op_gpu.cu:150-234,593-708)
 *   bsmm_reduced_dw       <- BlocksparseReducedDWOp: BlocksparseFeatureReduce{CN,NC} + hGemm{NT,TN}
 *                            (src/blocksparse_matmul_op.cc:639-773)
 *   bsmm_gather_rows      <- GatherScatter / ScatterAddMul ops behind SparseProj (blocksparse/matmul.py:835-921)
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer except `err` strings is DEVICE memory
 *     owned by the caller (the library never allocates device memory and keeps no state
 *     other than a lazily filled device-property cache);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant,
 *     and performs no host synchronisation;
 *   - return value 0 = success; >0 = cudaError_t from the launch; <0 = argument error
 *     (BSMM_E_*).  bsmm_last_error() gives a thread-local message for the last failure;
 *   - dtype codes: BSMM_F32 / BSMM_F16 / BSMM_BF16.  fp32 paths use true fp32 FMA (no TF32).
 *
 * LUT wire format consumed by xprop / xn / softmax ("row LUT", int32 [n_out + nnz][2]):
 *   rows [0, n_out)        = (first_entry_row, n_entries)   one header per output block
 *   rows [n_out, n_out+nnz) = (w_block, in_block)            grouped by output block
 *   -- this IS the reference's bst nn_lut/tn_lut format (blocksparse/transformer.py:161-181);
 *   the bsmm host layer emits the same format from fprop_list / bprop_list
 *   (blocksparse/matmul.py:137-138) instead of the segmented/locked Volta format.
 * updat / NT consume the reference's own updat_lut / nt_lut: int32 [blocks][2] = (c,k) / (q,k)
 *   (blocksparse/matmul.py:134-135, transformer.py:107-111).
 */
#ifndef BSMM_B200_H_
#define BSMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { BSMM_F32 = 0, BSMM_F16 = 1, BSMM_BF16 = 2 };

enum {
  BSMM_E_DTYPE   = -1,   /* unsupported dtype (combination)            */
  BSMM_E_BSIZE   = -2,   /* unsupported block size / axis combination  */
  BSMM_E_ARG     = -3,   /* null pointer, negative size, pcount > 8 …  */
  BSMM_E_LIMIT   = -4,   /* size limit exceeded (mirrors reference OP_REQUIRES) */
  BSMM_E_NODEV   = -5,   /* no sm_100 device / driver entry point missing */
  BSMM_E_ALIGN   = -6    /* pointer or leading dimension not aligned as the tensor-core path needs */
};

/* flags for bsmm_xprop / bsmm_updat / bst_* */
enum {
  BSMM_FLAG_FORCE_GENERIC = 1,   /* use the CUDA-core kernels even where a tcgen05 kernel exists */
  BSMM_FLAG_FORCE_TC      = 2    /* fail (BSMM_E_ARG) instead of falling back to CUDA-core kernels */
};

#define BSMM_MAX_PAIRS 8         /* reference: <= 8 (x,dy) pairs per updat launch (op.cc:233-234) */

/* ---- library / device ------------------------------------------------------------ */
int         bsmm_version(void);                 /* 1000*major + minor */
const char* bsmm_last_error(void);              /* thread-local, never NULL */
int         bsmm_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* name of the kernel family the last successful call on this thread dispatched to
 * ("tcgen05_xprop_bs32", "fma_xprop", ...) -- used by tests to prove which path ran */
const char* bsmm_last_kernel(void);
/* Debug aid: synchronises the current device, then returns and clears the sticky device-side error
 * word (non-zero if a tensor-core kernel's bounded barrier wait timed out since the last call). */
int         bsmm_device_error(void);
/* Every mbarrier wait inside the tcgen05 kernels is wall-clock bounded.  A wait that exceeds `ms` milliseconds
 * (default 2000) records an error code and, when `trap` is non-zero (default), executes `trap`: the launch fails and
 * the next CUDA call of the host reports the fault, so a starved or mis-sequenced kernel can never return partially
 * written outputs with rc 0.  trap = 0 keeps the context alive (the kernel exits early; poll bsmm_device_error()). */
int         bsmm_set_wait_timeout_ms(int ms, int trap);
/* Tuning aid: with BSMM_TRACE set in the environment, CTA 0 of the pair-schedule xprop kernel records clock64() at five
 * pipeline events (producer: stage free, loads issued; issuer: stage full, turn taken, MMAs committed) of its first 256
 * groups; this copies n <= 2048 words (8 per group) of the last launch to `out`. */
int         bsmm_debug_trace(unsigned long long* out, int n);

/* ---- block-sparse matmul -------------------------------------------------------- */

/*
 * fprop (bprop=0):  axis 0: Y[k-blk,:,n] = sum_{(c,w) in lut[k]} W[w]^T X[c-blk,:,n] (*gate[w])
 *                   axis 1: Y[n,k-blk]   = sum X[n,c-blk] W[w]
 * bprop (bprop=1):  axis 0: DX[c-blk]    = sum_{(k,w) in lut[c]} W[w] DY[k-blk]
 *                   axis 1: DX[n,c-blk]  = sum DY[n,k-blk] W[w]^T
 * x: (n_in*bsize, N) for axis 0, (N, n_in*bsize) for axis 1; y likewise with n_out.
 * w: (blocks, bsize, bsize), element [w][i][j], i = input-feature, j = output-feature of FPROP
 *    (blocksparse/matmul.py:360,369).
 * lut: row LUT grouped by output block (n_out headers).  Output blocks with no entries are
 *    zero-filled (reference behaviour, cn_64.cu:243-253).
 * sched: optional tile schedule for the tcgen05 kernels built by the host layer
 *    (blocksparse_b200/lut.py:build_tile_schedule, device memory) with its shape passed by value:
 *    sched_tiles output tiles of (sched_tile_blocks & 0xff) consecutive output blocks each (bits 8.. = W blocks
 *    per schedule group when it differs from the default: 2 or 4 select the deeper-pipeline variants used for
 *    layouts below ~12 % / ~37 % density), group records starting at int32 index sched_groups_off; NULL selects
 *    the CUDA-core kernels.
 *    The persistent CTAs pull tiles from a global counter; sched_list_off > 0 gives the int32 index (inside sched) of an
 *    optional tile ORDER table (tile ids, heaviest first, built for sched_ntiles = ceil(N/128) minibatch tiles).
 *    Pair schedule (32 x 32 blocks, lut.py:build_pair_schedule, opt-in): bit 16 of sched_tile_blocks set; then
 *    sched_list_off indexes the per-CTA tile lists (built for sched_ctas CTAs and sched_ntiles minibatch tiles) and
 *    bits 8..15 select the kernel variant (1 sparse, 2 mid, 3 wide tiles).
 * gate: optional float[blocks]; a zero gate skips the block (cn_64.cu:96-98).  With a gate the call runs on the
 *    CUDA-core kernels; for 16-bit weights call bsmm_gate_weights first and pass gate = NULL to stay on tcgen05.
 */
int bsmm_xprop(int dtype, int axis, int bsize, int bprop,
               const int32_t* lut, int n_out, int n_in, int blocks,
               const void* x, const void* w, void* y, int N,
               const float* gate,
               const int32_t* sched, int sched_tiles, int sched_tile_blocks, int sched_groups_off,
               int sched_list_off, int sched_ctas, int sched_ntiles,
               int flags, void* stream);

/*
 * updat:  DW[w] = alpha * sum_{p<pcount} X_p[c-blk] . DY_p[k-blk]^T  (+ beta * DW[w]),  (c,k) = updat_lut[w]
 *   axis 0: X_p (C,N), DY_p (K,N);  axis 1: X_p (N,C), DY_p (N,K).
 * xs/dys: HOST arrays of pcount device pointers (the reference passes them by value in
 *   Plist<T,8>, gpu_types.h:167-170).  beta must be 0 or 1 (DWA accumulate-in-place, op.cc:262-272).
 * dw_dtype: BSMM_F32 or `dtype` (the reference always produces the activation dtype; fp32
 *   accumulation across launches is our extension).
 * gate != NULL with gated_dw: blocks whose gate is 0 produce 0, others are scaled by the gate
 *   (blocksparse/matmul.py:414-417).
 */
int bsmm_updat(int dtype, int dw_dtype, int axis, int bsize,
               const int32_t* updat_lut, int blocks, int n_c_blocks, int n_k_blocks,
               const void* const* xs, const void* const* dys, int pcount,
               void* dw, int N, float alpha, float beta,
               const float* gate, int gated_dw,
               const int32_t* sched, int sched_tiles, int sched_tile_blocks, int sched_groups_off,
               int flags, void* stream);

/* dg[w] = sum_ij dw[w][i][j] * w[w][i][j]   (BlocksparseMatmulDG, op.cc:490-540) */
int bsmm_gate_grad(int dtype, int bsize, int blocks, const void* dw, const void* w,
                   float* dg, void* stream);

/* w_out[w] = gate[w] * w[w] (zero gate => exact zero block).  Host layers call it before a gated bsmm_xprop of 16-bit
 * weights so that the gated product runs on the tcgen05 kernel: the reference's gated kernels apply the gate to the
 * loaded weights the same way (cn_64.cu:96-98, blocksparse_hgemm_nc_op_gpu.cu gate handling). */
int bsmm_gate_weights(int dtype, int bsize, int blocks, const void* w, const float* gate,
                      void* w_out, void* stream);

/* ---- block-sparse transformer ------------------------------------------------------ */

/*
 * NT: C[b,h,blk,:,:] = A[b, q-blk, h, :] . B[b, k-blk, h, :]^T     (q,k) = nt_lut[hl][blk]
 *   a: (batch, ctx_blks_a*bsize, heads*head_state), b: (batch, ctx_blks_b*bsize, heads*head_state)
 *   c: (batch, heads, blocks, bsize, bsize) of c_dtype.
 *   nt_lut: int32 [lut_heads][blocks][2]; lut_heads in {1, heads}.
 *   nt_items / n_items: optional schedule for the tcgen05 kernel (blocksparse_b200/lut.py:build_nt_items, device
 *     int32 [lut_heads][n_items][8] = (k_blk, n_valid, blk0, q0, blk1, q1, 0, 0): blocks sharing a key block, two
 *     at a time); NULL selects the CUDA-core kernel.
 */
int bst_nt(int dtype, int c_dtype, int bsize,
           const int32_t* nt_lut, int lut_heads, int blocks,
           const int32_t* nt_items, int n_items,
           const void* a, const void* b, void* c,
           int batch, int heads, int head_state, int ctx_blks_a, int ctx_blks_b,
           int flags, void* stream);

/*
 * XN: transpose_a=0 (NN): C[b, q-blk, h, :] = sum_{(blk,k) in lut[q]} A[b,h,blk]   . B[b, k-blk, h, :]
 *     transpose_a=1 (TN): C[b, k-blk, h, :] = sum_{(blk,q) in lut[k]} A[b,h,blk]^T . B[b, q-blk, h, :]
 *   lut: int32 [lut_heads][ctx_blks_c + blocks][2] -- the reference's nn_lut / tn_lut verbatim.
 *   out_order: optional int32 [lut_heads][ctx_blks_c], output blocks sorted by decreasing LUT row length; the
 *     persistent tcgen05 kernel walks it so that long rows (e.g. strided attention columns) start first.
 */
int bst_xn(int a_dtype, int dtype, int bsize, int transpose_a,
           const int32_t* lut, const int32_t* out_order, int lut_heads, int blocks, int max_lut,
           const void* a, const void* b, void* c,
           int batch, int heads, int head_state, int ctx_blks_b, int ctx_blks_c,
           int flags, void* stream);

/*
 * y = softmax(scale * x) along each query row across all key blocks of the row, with an
 * optional bit mask (bit j of word r of block blk set <=> key j visible to query r).
 *   x, y: (batch, heads, blocks, bsize, bsize);  lut = nn_lut (rows = query blocks).
 *   mask: NULL or uint{bsize}[mask_heads][blocks][bsize]  (the host layer's softmax_mask_np
 *         layout, blocksparse/transformer.py:155) ; mask_heads in {1, heads}.
 *   autoregress_at_key >= 0 applies the partial-autoregressive rewrite on the fly
 *         (blocksparse/transformer.py:264-274); nt_lut is then required.
 * Limit: max_lut * bsize <= 32768 (bst_op.cc:383).
 * x and y (bst_softmax_grad: dy, y and dx) must start at an address aligned to the kernels' vector accesses (4 to 16
 * bytes; 16 always suffices), else BSMM_E_ARG.
 */
int bst_softmax(int x_dtype, int y_dtype, int bsize,
                const int32_t* nn_lut, const int32_t* nt_lut, int lut_heads, int blocks, int max_lut,
                const void* mask, int mask_heads, int autoregress_at_key,
                const void* x, void* y, float scale,
                int batch, int heads, int ctx_blks_q, void* stream);

/* dx = (dy - sum_row(dy*y)) * y * scale   (blocksparse/transformer.py:301) */
int bst_softmax_grad(int dtype, int dx_dtype, int bsize,
                     const int32_t* nn_lut, int lut_heads, int blocks, int max_lut,
                     const void* dy, const void* y, void* dx, float scale,
                     int batch, int heads, int ctx_blks_q, void* stream);

/* mask_out[hl][blk][r] = mask_in[hl][blk][r] & (ones >> shift(r)), same layout as bst_softmax's mask */
int bst_autoregressive_mask(int bsize, const int32_t* nt_lut, int lut_heads, int blocks,
                            const void* mask_in, void* mask_out, int autoregress_at_key,
                            void* stream);

/* ---- utilities on the (blocks, bsize, bsize) weight format (SURVEY.md 8f) -------------------------------------- */

/* norm[b] = max|w| (norm_type 0) or sqrt(sum w^2) (norm_type 1) of block b; norm is float[blocks]. */
int bsmm_block_norm(int dtype, int bsize, int blocks, const void* w, float* norm, int norm_type, void* stream);
/* In place: w[b] -= w[b] * min(rate / sqrt(sum(w[b]^2) + epsilon), 1); blocks whose gate is 0 are skipped (gate may be NULL). */
int bsmm_l2_decay(int dtype, int bsize, int blocks, void* w, const float* gate, float rate, float epsilon, void* stream);
/* gate[b] = norm(w[b]) < threshold ? 0 : 1 */
int bsmm_threshold_prune(int dtype, int bsize, int blocks, const void* w, float* gate, float threshold, int norm_type, void* stream);
/* idx = block ids sorted by decreasing norm: gate[idx[i]] = i < keep ? 1 : 0 */
int bsmm_prune_topk(float* gate, const int32_t* idx, int blocks, int keep, void* stream);
/* W[b] = scale * I for blocks with (c % KB) == (k % CB), 0 elsewhere; updat_lut = int32 [blocks][2] = (c, k). */
int bsmm_identity_init(int dtype, int bsize, int blocks, const int32_t* updat_lut, int n_c_blocks, int n_k_blocks, void* w, float scale, void* stream);
/* y[w][i][j] = gain[k*bs + j] * w[w][i][j] / sqrt(max(sum_sqr[k*bs + j], epsilon)), the sum running over every row of every
 * block of OUTPUT block column k (lut = the fprop row LUT, n_out = KB); sum_sqr (float[KB*bsize]) is kept for the gradient.
 * gain may be NULL.  y_dtype: the weight dtype or fp32. */
int bsmm_l2_normalize(int dtype, int y_dtype, int bsize, const int32_t* lut, int n_out, const void* w, const float* gain, void* y,
                      float* sum_sqr, float epsilon, void* stream);
/* dx (weight dtype), dg (float[KB*bsize], NULL without gain):
 * dx = (dy*g + w * (sum_sqr >= eps) * sum(-dy*g*w / max(sum_sqr, eps))) / sqrt(max(sum_sqr, eps));  dg = sum(dy * w / norm) */
int bsmm_l2_normalize_grad(int dtype, int y_dtype, int bsize, const int32_t* lut, int n_out, const void* dy, const void* w, const float* gain,
                           const float* sum_sqr, void* dx, float* dg, float epsilon, void* stream);
/* Block-reduced FULL weight gradient for network growth: x_red / y_red = per-block max|.| (norm_type 0) or l2 norm over the
 * bsize features of each block of every x_p / dy_p (layout (pair, n, block) for axis 1, (block, pair, n) for axis 0, activation
 * dtype), then dw[bC][bK] (float) = scale * sum_{p,n} x_red * y_red (+ dw when accumulate).  scale == 0 skips the reductions.
 * workspace: bsmm_reduced_dw_workspace_bytes(bC, bK) bytes of device memory. */
size_t bsmm_reduced_dw_workspace_bytes(int n_c_blocks, int n_k_blocks);
int bsmm_reduced_dw(int dtype, int axis, int bsize, const void* const* xs, const void* const* dys, int pcount,
                    int n_c_blocks, int n_k_blocks, int N, float scale, int norm_type, float* dw, int accumulate,
                    void* x_red, void* y_red, void* workspace, void* stream);
/* Row gather / scatter on (rows, N) activations (SparseProj): op 0: out[r] = idx[r] >= 0 ? x[idx[r]] : 0;
 * op 1: out[r] = x[r] + (idx[r] >= 0 ? y[idx[r]] : 0);  op 2: out[r] = x[r] * (idx[r] >= 0 ? y[idx[r]] : 1). */
int bsmm_gather_rows(int dtype, const void* x, const void* y, const int32_t* idx, void* out, int rows, long long N, int op, void* stream);

/* 8 x 8 blocks on tcgen05 (N >= 16 per MMA): scatter a (blocks_small, bs, bs) weight tensor into (blocks_big, 2bs, 2bs)
 * super-blocks -- sub_map[4*b + 2*(row half) + (col half)] = small block id or -1 (zero fill), optional per-small-block gate
 * folded in -- and gather the weight gradient back: inv_map[w] = 4 * super-block + sub-position, optional per-block gate
 * (gated dW), accumulate adds to dw_small. */
int bsmm_pad_blocks(int dtype, int bsize, int blocks_big, const int32_t* sub_map, const void* w_small, const float* gate, void* w_big, void* stream);
int bsmm_unpad_blocks(int in_dtype, int out_dtype, int bsize, int blocks_small, const int32_t* inv_map, const void* dw_big, const float* gate,
                      void* dw_small, int accumulate, void* stream);

/* ---- measurement helper (the reference's `bench` op attribute, op.cc:99-106) ---------
 * Records two events around whatever the caller enqueues between begin and end.      */
int bsmm_timer_create(void** timer);
int bsmm_timer_begin(void* timer, void* stream);
int bsmm_timer_end(void* timer, void* stream, float* ms_out);   /* synchronises on the stop event */
int bsmm_timer_destroy(void* timer);

#ifdef __cplusplus
}
#endif
#endif /* BSMM_B200_H_ */
