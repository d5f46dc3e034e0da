// Block-sparse (masked) softmax, its gradient and the partial-autoregressive mask.
//
// Replaces bst_masked_softmax / bst_masked_softmax_grad / bst_partial_autoregressive_mask
// (src/bst_softmax_op_gpu.cu:12-198, 200-310, 461-520).
//
// HBM-bound: algorithmic traffic is (s_in + s_out) bytes per element of the
// (batch, heads, blocks, bs, bs) tensor.  Work decomposition (differs from the
// reference's one-CTA-per-query-row): one WARP owns 4 (bs 64) or 8 consecutive query
// rows of one query block and each lane 16 bytes of a row, so every warp-wide access is
// one contiguous 256..512-byte chunk of a block; the row's LUT entries are loaded once
// (one per lane) and broadcast by shuffle; row statistics are reduced with xor-shuffles
// inside the 4/8-lane group that shares a row.  Values stay in registers between the
// statistics pass and the write pass for rows of <= KEEP key blocks; longer rows re-read.
#pragma once
#include <float.h>
#include "common.cuh"

namespace bsmm {

struct SoftmaxParams {
  const int32_t* nn_lut;      // [lut_heads][ctx_blks_q + blocks][2]
  const int32_t* nt_lut;      // [lut_heads][blocks][2], only for autoregress
  long long nn_head_stride, nt_head_stride;
  const void* mask;           // uintBS [mask_heads][blocks][BS] or null
  long long mask_head_stride; // words
  int autoregress_at_key;     // <0: off
  const void* x; void* y;     // x = input (or dy for grad); y = output (or dx)
  const void* y_in;           // grad only: softmax output
  float scale;
  int batch, heads, blocks, ctx_blks_q;
};

template <int BS> struct MaskWord;
template <> struct MaskWord<8>  { using type = uint8_t;  };
template <> struct MaskWord<16> { using type = uint16_t; };
template <> struct MaskWord<32> { using type = uint32_t; };
template <> struct MaskWord<64> { using type = uint64_t; };

template <typename T> struct Pair;
template <> struct Pair<float>         { using type = float2; };
template <> struct Pair<__half>        { using type = __half2; };
template <> struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };

template <typename T> __device__ __forceinline__ float2 load2(const T* p) {
  typename Pair<T>::type v = *reinterpret_cast<const typename Pair<T>::type*>(p);
  return make_float2(to_f32<T>(v.x), to_f32<T>(v.y));
}
template <typename T> __device__ __forceinline__ void store2(T* p, float a, float b) {
  typename Pair<T>::type v;
  v.x = from_f32<T>(a); v.y = from_f32<T>(b);
  *reinterpret_cast<typename Pair<T>::type*>(p) = v;
}

template <int BS>
__device__ __forceinline__ uint64_t autoregress_word(uint64_t word, int ak, int k_blk, int q_row) {
  // blocksparse/transformer.py:264-274
  const int k0 = k_blk * BS;
  const int sa = BS - min(max(ak - k0, 0), BS);
  const int sb = min(max(BS - 1 + k0 - q_row, 0), BS);
  const int sh = min(sa, sb);
  const uint64_t ones = (BS == 64) ? ~0ull : ((1ull << BS) - 1ull);
  return sh >= BS ? 0ull : (word & (ones >> sh));
}

constexpr int SOFTMAX_WARPS = 4;

// Lane mapping: a warp covers RP consecutive query rows of one block per pass; LPR lanes share a row and each
// lane owns EPL consecutive keys (16 bytes of 16-bit data when bs >= 32), so one warp-wide load is a single
// contiguous RP*bs*sizeof(T) chunk of the block (512 B for bs 64).
template <int BS> struct SoftmaxMap {
  static constexpr int LPR = (BS == 64) ? 8 : 4;        // lanes per row
  static constexpr int EPL = BS / LPR;                  // elements per lane: 8, 8, 4, 2
  static constexpr int RP = 32 / LPR;                   // rows per pass: 4, 8, 8, 8
  static constexpr int GROUPS = BS / RP;                // passes per query block
  static constexpr int KEEP = (EPL >= 8) ? 4 : 8;       // key blocks of a row kept in registers (more costs occupancy: measured)
};

template <typename T, int EPL> __device__ __forceinline__ void load_vec(const T* p, float (&f)[EPL]) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < EPL; i += 2) { const float2 v = *reinterpret_cast<const float2*>(p + i); f[i] = v.x; f[i + 1] = v.y; }
  } else if constexpr (EPL == 8) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { const typename Pair<T>::type h = *reinterpret_cast<const typename Pair<T>::type*>(&w[i]); f[2 * i] = to_f32<T>(h.x); f[2 * i + 1] = to_f32<T>(h.y); }
  } else if constexpr (EPL == 4) {
    const uint2 v = *reinterpret_cast<const uint2*>(p);
    const uint32_t w[2] = {v.x, v.y};
#pragma unroll
    for (int i = 0; i < 2; ++i) { const typename Pair<T>::type h = *reinterpret_cast<const typename Pair<T>::type*>(&w[i]); f[2 * i] = to_f32<T>(h.x); f[2 * i + 1] = to_f32<T>(h.y); }
  } else {
    const float2 v = load2<T>(p); f[0] = v.x; f[1] = v.y;
  }
}
template <typename T, int EPL> __device__ __forceinline__ void store_vec(T* p, const float (&f)[EPL]) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < EPL; i += 2) *reinterpret_cast<float2*>(p + i) = make_float2(f[i], f[i + 1]);
  } else if constexpr (EPL == 8) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { typename Pair<T>::type h; h.x = from_f32<T>(f[2 * i]); h.y = from_f32<T>(f[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&h); }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  } else if constexpr (EPL == 4) {
    uint32_t w[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) { typename Pair<T>::type h; h.x = from_f32<T>(f[2 * i]); h.y = from_f32<T>(f[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&h); }
    *reinterpret_cast<uint2*>(p) = make_uint2(w[0], w[1]);
  } else {
    store2<T>(p, f[0], f[1]);
  }
}

// Widest access load_vec / store_vec make to a T tensor: float2 for fp32, EPL packed 16-bit values otherwise.  Every access
// sits a multiple of this many bytes past the tensor's start, so the start must be aligned to it.
template <typename T, int BS> constexpr int softmax_vec_bytes() { return sizeof(T) == 4 ? 8 : SoftmaxMap<BS>::EPL * 2; }
template <typename T, int BS> inline bool softmax_aligned(const void* p) { return ((uintptr_t)p % softmax_vec_bytes<T, BS>()) == 0; }

template <typename TX, typename TY, int BS>
__global__ void __launch_bounds__(SOFTMAX_WARPS * 32)
bst_softmax_kernel(const SoftmaxParams p) {
  using MT = typename MaskWord<BS>::type;
  using M = SoftmaxMap<BS>;
  constexpr int LPR = M::LPR, EPL = M::EPL, RP = M::RP, GROUPS = M::GROUPS, KEEP = M::KEEP;
  const int lane = threadIdx.x % 32;
  const long long gid = (long long)blockIdx.x * SOFTMAX_WARPS + threadIdx.x / 32;
  if (gid >= (long long)p.ctx_blks_q * GROUPS) return;
  const int q = (int)(gid / GROUPS);
  const int row = (int)(gid % GROUPS) * RP + lane / LPR;
  const int col = (lane % LPR) * EPL;
  const int h = blockIdx.y, b = blockIdx.z;

  const int hl = p.nn_head_stride ? h : 0;
  const int32_t* lut = p.nn_lut + (long long)hl * p.nn_head_stride;
  const int first = lut[2 * q], count = lut[2 * q + 1];
  if (count == 0) return;
  const long long zoff = ((long long)b * p.heads + h) * p.blocks;
  const TX* x = reinterpret_cast<const TX*>(p.x) + (long long)row * BS + col;
  TY* y = reinterpret_cast<TY*>(p.y) + (long long)row * BS + col;
  const MT* mask = reinterpret_cast<const MT*>(p.mask);
  if (mask) mask += (p.mask_head_stride ? (long long)h * p.mask_head_stride : 0) + row;
  // the row's LUT entries, one per lane (rows longer than 32 key blocks reload per chunk of 32)
  const int2* ent = reinterpret_cast<const int2*>(lut) + first;
  int2 my = (lane < count) ? ent[lane] : make_int2(0, 0);

  auto entry = [&](int e, int& blk, int& kb) {
    if (e < 32) { blk = __shfl_sync(0xffffffffu, my.x, e); kb = __shfl_sync(0xffffffffu, my.y, e); }
    else { const int2 v = ent[e]; blk = v.x; kb = v.y; }
  };
  auto load_entry = [&](int e, float (&v)[EPL]) {
    int blk, kb;
    entry(e, blk, kb);
    load_vec<TX, EPL>(x + (zoff + blk) * (BS * BS), v);
#pragma unroll
    for (int i = 0; i < EPL; ++i) v[i] *= p.scale;
    if (mask) {
      uint64_t w = (uint64_t)mask[(long long)blk * BS];
      if (p.autoregress_at_key >= 0) w = autoregress_word<BS>(w, p.autoregress_at_key, kb, q * BS + row);
      // most blocks are fully visible (only e.g. the diagonal ones carry a causal pattern): skip the bit tests there
      const uint64_t mine = (w >> col) & ((1ull << EPL) - 1ull);
      if (mine != ((1ull << EPL) - 1ull)) {
#pragma unroll
        for (int i = 0; i < EPL; ++i) if (!((mine >> i) & 1ull)) v[i] = -FLT_MAX;
      }
    }
  };

  // Pass A (one read of the row): online max / sum -- (m, s) with s = sum exp(v - m), rescaled whenever m grows.
  constexpr float LOG2E = 1.4426950408889634f;
  // exp2 is the other bound of this kernel (MUFU: 16/clk/SM, i.e. ~0.1 ms for cfg 3 if every element needed two):
  // kept entries are exponentiated ONCE, against the running max at that time (mref[e]), and rescaled by one
  // scalar exp2 per entry at the end.
  float keep[KEEP][EPL];
  float mref[KEEP];
  float m = -FLT_MAX, s = 0.f;
  auto absorb = [&](float (&v)[EPL]) -> float {
    float mv = v[0];
#pragma unroll
    for (int i = 1; i < EPL; ++i) mv = fmaxf(mv, v[i]);
    const float mn = fmaxf(m, mv);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < EPL; ++i) { v[i] = exp2f((v[i] - mn) * LOG2E); acc += v[i]; }
    s = s * exp2f((m - mn) * LOG2E) + acc;
    m = mn;
    return mn;
  };
#pragma unroll
  for (int e = 0; e < KEEP; ++e) {
    mref[e] = 0.f;
    if (e < count) { load_entry(e, keep[e]); mref[e] = absorb(keep[e]); }
  }
#pragma unroll 4
  for (int e = KEEP; e < count; ++e) {
    float v[EPL]; load_entry(e, v);
    absorb(v);
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) {
    const float mo = __shfl_xor_sync(0xffffffffu, m, o);
    const float so = __shfl_xor_sync(0xffffffffu, s, o);
    const float mn = fmaxf(m, mo);
    s = s * exp2f((m - mn) * LOG2E) + so * exp2f((mo - mn) * LOG2E);
    m = mn;
  }
  const float inv = 1.f / s;

  // Pass B: normalise and write (kept values from registers, the rest re-read -- L2 hits)
#pragma unroll
  for (int e = 0; e < KEEP; ++e) {
    if (e < count) {
      int blk, kb; entry(e, blk, kb);
      const float sc = exp2f((mref[e] - m) * LOG2E) * inv;
#pragma unroll
      for (int i = 0; i < EPL; ++i) keep[e][i] *= sc;
      store_vec<TY, EPL>(y + (zoff + blk) * (BS * BS), keep[e]);
    }
  }
#pragma unroll 4
  for (int e = KEEP; e < count; ++e) {
    float v[EPL]; load_entry(e, v);
    int blk, kb; entry(e, blk, kb);
#pragma unroll
    for (int i = 0; i < EPL; ++i) v[i] = exp2f((v[i] - m) * LOG2E) * inv;
    store_vec<TY, EPL>(y + (zoff + blk) * (BS * BS), v);
  }
}

// ---- TMA-staged variant (16-bit in and out, 32 x 32 / 64 x 64 blocks, rows of <= MAXE key blocks) -------------------
// One small CTA per (query block, 16-row chunk, head, batch).  Rows of a softmax are independent, and 16 consecutive rows of a
// block are one contiguous 16*bs*2-byte piece of the sparse tensor: one thread pulls the chunk's piece of every block of the
// row into shared memory with bulk async copies (one mbarrier), the 4 warps then own 4 query rows each -- a warp-wide
// shared-memory access is one whole row of one block, conflict free -- keep the row's values in registers across max / exp /
// sum / normalise, write the 16-bit results back IN PLACE, and one thread sends every piece to HBM with a bulk store.  HBM
// sees each element exactly once in and once out, in 1-2 KB bursts, and with ~22 KB of shared memory per CTA ten CTAs share
// an SM, so loads, arithmetic and stores of different chunks overlap.  (First version: one CTA per whole query block, 88 KB,
// two per SM, phases serialised: 0.347 ms at cfg 3 against 0.165 ms for the register kernel, profiles/r2_softmax.txt.)
constexpr int SOFTMAX_STAGED_THREADS = 128;
constexpr int SOFTMAX_STAGED_ROWS = 16;

template <typename TX, typename TY, int BS, int MAXE>
__global__ void __launch_bounds__(SOFTMAX_STAGED_THREADS, 8)      // <= 64 registers: eight CTAs (~180 KB of chunks) in flight per SM
bst_softmax_staged_kernel(const SoftmaxParams p) {
  static_assert(sizeof(TX) == 2 && sizeof(TY) == 2 && (BS == 32 || BS == 64), "staged softmax: 16-bit, bs 32/64");
  using MT = typename MaskWord<BS>::type;
  constexpr int EPL = BS / 32;                    // elements per lane: a warp reads one row of one block per access
  constexpr int RC = SOFTMAX_STAGED_ROWS, NCH = BS / RC;
  constexpr uint32_t BLK_BYTES = RC * BS * 2;     // the chunk's piece of one block
  extern __shared__ __align__(128) uint8_t sm_blocks[];
  __shared__ uint64_t bar;
  __shared__ int2 s_ent[MAXE];
  __shared__ uint64_t s_mask[MAXE][RC];           // mask word of every (block, row) of the chunk, fetched while the tiles fly
  const int q = blockIdx.x / NCH, row0 = (blockIdx.x % NCH) * RC, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid / 32, lane = tid % 32;
  const int hl = p.nn_head_stride ? h : 0;
  const int32_t* lut = p.nn_lut + (long long)hl * p.nn_head_stride;
  const int first = lut[2 * q], count = lut[2 * q + 1];
  if (count == 0) return;
  const long long zoff = ((long long)b * p.heads + h) * p.blocks;
  const int2* ent = reinterpret_cast<const int2*>(lut) + first;
  if (tid < count) s_ent[tid] = ent[tid];
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
  if (tid == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"((uint32_t)count * BLK_BYTES) : "memory");
    for (int e = 0; e < count; ++e) {
      const TX* src = reinterpret_cast<const TX*>(p.x) + (zoff + s_ent[e].x) * (long long)(BS * BS) + row0 * BS;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(sm_blocks + (size_t)e * BLK_BYTES)), "l"(src), "r"(BLK_BYTES), "r"(bar_a) : "memory");
    }
  }
  const MT* mask = reinterpret_cast<const MT*>(p.mask);
  if (mask) {
    mask += (p.mask_head_stride ? (long long)h * p.mask_head_stride : 0);
    for (int i = tid; i < count * RC; i += SOFTMAX_STAGED_THREADS) {
      const int e = i / RC, r = i % RC;
      uint64_t w = (uint64_t)mask[(long long)s_ent[e].x * BS + row0 + r];
      if (p.autoregress_at_key >= 0) w = autoregress_word<BS>(w, p.autoregress_at_key, s_ent[e].y, q * BS + row0 + r);
      s_mask[e][r] = w;
    }
    __syncthreads();
  }
  {   // every thread waits for the data (parity 0: single use of the barrier)
    uint32_t ok = 0;
    while (!ok)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(bar_a) : "memory");
  }
  constexpr float LOG2E = 1.4426950408889634f;
  constexpr uint64_t ALL = (BS == 64) ? ~0ull : ((1ull << BS) - 1ull);
  const float sc2 = p.scale * LOG2E;              // work in the exp2 domain: v = x * scale * log2(e)
  for (int lr = warp; lr < RC; lr += SOFTMAX_STAGED_THREADS / 32) {
    const int row = row0 + lr;
    float v[MAXE][EPL];
    float m = -FLT_MAX;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
      if (e < count) {
        const TX* src = reinterpret_cast<const TX*>(sm_blocks + (size_t)e * BLK_BYTES) + lr * BS + lane * EPL;
        if constexpr (EPL == 2) { const float2 t = load2<TX>(src); v[e][0] = t.x * sc2; v[e][1] = t.y * sc2; }
        else v[e][0] = to_f32<TX>(*src) * sc2;
        if (mask) {
          const uint64_t w = s_mask[e][lr];                 // warp-uniform; most blocks are fully visible: skip the bit tests
          if (w != ALL) {
#pragma unroll
            for (int i = 0; i < EPL; ++i) if (!((w >> (lane * EPL + i)) & 1ull)) v[e][i] = -FLT_MAX;
          }
        }
#pragma unroll
        for (int i = 0; i < EPL; ++i) m = fmaxf(m, v[e][i]);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float ssum = 0.f;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
      if (e < count) {
#pragma unroll
        for (int i = 0; i < EPL; ++i) { v[e][i] = exp2f(v[e][i] - m); ssum += v[e][i]; }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
    const float inv = 1.f / ssum;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
      if (e < count) {
        TY* dst = reinterpret_cast<TY*>(sm_blocks + (size_t)e * BLK_BYTES) + lr * BS + lane * EPL;
        if constexpr (EPL == 2) store2<TY>(dst, v[e][0] * inv, v[e][1] * inv);
        else *dst = from_f32<TY>(v[e][0] * inv);
      }
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes -> visible to the bulk store
  __syncthreads();
  if (tid == 0) {
    for (int e = 0; e < count; ++e) {
      TY* dst = reinterpret_cast<TY*>(p.y) + (zoff + s_ent[e].x) * (long long)(BS * BS) + row0 * BS;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                   ::"l"(dst), "r"((uint32_t)__cvta_generic_to_shared(sm_blocks + (size_t)e * BLK_BYTES)), "r"(BLK_BYTES) : "memory");
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory must outlive the reads
  }
}

// Gradient, same decomposition: dy and y pieces are staged (2 x ~22 KB per CTA), dx = (dy - sum_row(dy*y)) * y * scale is
// written over the dy piece and bulk-stored.
template <typename T, typename TD, int BS, int MAXE>
__global__ void __launch_bounds__(SOFTMAX_STAGED_THREADS)
bst_softmax_grad_staged_kernel(const SoftmaxParams p) {
  static_assert(sizeof(T) == 2 && sizeof(TD) == 2 && (BS == 32 || BS == 64), "staged softmax grad: 16-bit, bs 32/64");
  constexpr int EPL = BS / 32;
  constexpr int RC = SOFTMAX_STAGED_ROWS, NCH = BS / RC;
  constexpr uint32_t BLK_BYTES = RC * BS * 2;
  extern __shared__ __align__(128) uint8_t sm_blocks[];      // [count] dy pieces, then [count] y pieces
  __shared__ uint64_t bar;
  __shared__ int s_blk[MAXE];
  const int q = blockIdx.x / NCH, row0 = (blockIdx.x % NCH) * RC, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid / 32, lane = tid % 32;
  const int hl = p.nn_head_stride ? h : 0;
  const int32_t* lut = p.nn_lut + (long long)hl * p.nn_head_stride;
  const int first = lut[2 * q], count = lut[2 * q + 1];
  if (count == 0) return;
  const long long zoff = ((long long)b * p.heads + h) * p.blocks;
  if (tid < count) s_blk[tid] = lut[2 * (first + tid)];
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
  uint8_t* sm_y = sm_blocks + (size_t)count * BLK_BYTES;
  if (tid == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(2u * (uint32_t)count * BLK_BYTES) : "memory");
    for (int e = 0; e < count; ++e) {
      const long long off = (zoff + s_blk[e]) * (long long)(BS * BS) + row0 * BS;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(sm_blocks + (size_t)e * BLK_BYTES)), "l"(reinterpret_cast<const T*>(p.x) + off), "r"(BLK_BYTES), "r"(bar_a) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(sm_y + (size_t)e * BLK_BYTES)), "l"(reinterpret_cast<const T*>(p.y_in) + off), "r"(BLK_BYTES), "r"(bar_a) : "memory");
    }
  }
  {
    uint32_t ok = 0;
    while (!ok)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(bar_a) : "memory");
  }
  for (int lr = warp; lr < RC; lr += SOFTMAX_STAGED_THREADS / 32) {
    float d[MAXE][EPL], y[MAXE][EPL];
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
      if (e < count) {
        const T* pd = reinterpret_cast<const T*>(sm_blocks + (size_t)e * BLK_BYTES) + lr * BS + lane * EPL;
        const T* py = reinterpret_cast<const T*>(sm_y + (size_t)e * BLK_BYTES) + lr * BS + lane * EPL;
        if constexpr (EPL == 2) { const float2 a = load2<T>(pd), c = load2<T>(py); d[e][0] = a.x; d[e][1] = a.y; y[e][0] = c.x; y[e][1] = c.y; }
        else { d[e][0] = to_f32<T>(*pd); y[e][0] = to_f32<T>(*py); }
#pragma unroll
        for (int i = 0; i < EPL; ++i) acc += d[e][i] * y[e][i];
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
      if (e < count) {
        TD* dst = reinterpret_cast<TD*>(sm_blocks + (size_t)e * BLK_BYTES) + lr * BS + lane * EPL;
        if constexpr (EPL == 2) store2<TD>(dst, (d[e][0] - acc) * y[e][0] * p.scale, (d[e][1] - acc) * y[e][1] * p.scale);
        else *dst = from_f32<TD>((d[e][0] - acc) * y[e][0] * p.scale);
      }
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  if (tid == 0) {
    for (int e = 0; e < count; ++e) {
      TD* dst = reinterpret_cast<TD*>(p.y) + (zoff + s_blk[e]) * (long long)(BS * BS) + row0 * BS;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                   ::"l"(dst), "r"((uint32_t)__cvta_generic_to_shared(sm_blocks + (size_t)e * BLK_BYTES)), "r"(BLK_BYTES) : "memory");
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  }
}

template <typename T, typename TD, int BS>
int launch_softmax_grad_staged(const SoftmaxParams& p, int max_lut, cudaStream_t s) {
  dim3 grid(p.ctx_blks_q * (BS / SOFTMAX_STAGED_ROWS), p.heads, p.batch);
  const size_t smem = (size_t)2 * max_lut * SOFTMAX_STAGED_ROWS * BS * 2;
#define BSMM_STAGED(MAXE)                                                                                     \
  { auto kern = bst_softmax_grad_staged_kernel<T, TD, BS, MAXE>;                                              \
    static thread_local uint64_t cfg = 0;                                                                     \
    if (int e = ensure_dyn_smem(kern, (size_t)2 * MAXE * SOFTMAX_STAGED_ROWS * BS * 2, cfg)) return e;        \
    kern<<<grid, SOFTMAX_STAGED_THREADS, smem, s>>>(p); }
  if (max_lut <= 4) BSMM_STAGED(4)
  else if (max_lut <= 8) BSMM_STAGED(8)
  else if (max_lut <= 12) BSMM_STAGED(12)
  else BSMM_STAGED(16)
#undef BSMM_STAGED
  return check_launch("bst_softmax_grad_staged");
}

template <typename TX, typename TY, int BS>
int launch_softmax_staged(const SoftmaxParams& p, int max_lut, cudaStream_t s) {
  dim3 grid(p.ctx_blks_q * (BS / SOFTMAX_STAGED_ROWS), p.heads, p.batch);
  const size_t smem = (size_t)max_lut * SOFTMAX_STAGED_ROWS * BS * 2;
#define BSMM_STAGED(MAXE)                                                                                     \
  { auto kern = bst_softmax_staged_kernel<TX, TY, BS, MAXE>;                                                  \
    static thread_local uint64_t cfg = 0;                                                                     \
    if (int e = ensure_dyn_smem(kern, (size_t)MAXE * SOFTMAX_STAGED_ROWS * BS * 2, cfg)) return e;            \
    kern<<<grid, SOFTMAX_STAGED_THREADS, smem, s>>>(p); }
  if (max_lut <= 4) BSMM_STAGED(4)
  else if (max_lut <= 8) BSMM_STAGED(8)
  else if (max_lut <= 12) BSMM_STAGED(12)
  else BSMM_STAGED(16)
#undef BSMM_STAGED
  return check_launch("bst_softmax_staged");
}

template <typename T, typename TD, int BS>
__global__ void __launch_bounds__(SOFTMAX_WARPS * 32)
bst_softmax_grad_kernel(const SoftmaxParams p) {
  using M = SoftmaxMap<BS>;
  constexpr int LPR = M::LPR, EPL = M::EPL, RP = M::RP, GROUPS = M::GROUPS, KEEP = M::KEEP / 2 < 4 ? 4 : M::KEEP / 2;
  const int lane = threadIdx.x % 32;
  const long long gid = (long long)blockIdx.x * SOFTMAX_WARPS + threadIdx.x / 32;
  if (gid >= (long long)p.ctx_blks_q * GROUPS) return;
  const int q = (int)(gid / GROUPS);
  const int row = (int)(gid % GROUPS) * RP + lane / LPR;
  const int col = (lane % LPR) * EPL;
  const int h = blockIdx.y, b = blockIdx.z;
  const int hl = p.nn_head_stride ? h : 0;
  const int32_t* lut = p.nn_lut + (long long)hl * p.nn_head_stride;
  const int first = lut[2 * q], count = lut[2 * q + 1];
  if (count == 0) return;
  const long long zoff = ((long long)b * p.heads + h) * p.blocks;
  const long long roff = (long long)row * BS + col;
  const T* dy = reinterpret_cast<const T*>(p.x) + roff;
  const T* yv = reinterpret_cast<const T*>(p.y_in) + roff;
  TD* dx = reinterpret_cast<TD*>(p.y) + roff;
  const int2* ent = reinterpret_cast<const int2*>(lut) + first;
  const int my = (lane < count) ? ent[lane].x : 0;
  auto block_of = [&](int e) { return e < 32 ? __shfl_sync(0xffffffffu, my, e) : ent[e].x; };

  float kd[KEEP][EPL], ky[KEEP][EPL];
  float s = 0.f;
#pragma unroll
  for (int e = 0; e < KEEP; ++e) {
    if (e < count) {
      const long long off = (zoff + block_of(e)) * (BS * BS);
      load_vec<T, EPL>(dy + off, kd[e]);
      load_vec<T, EPL>(yv + off, ky[e]);
#pragma unroll
      for (int i = 0; i < EPL; ++i) s += kd[e][i] * ky[e][i];
    }
  }
  for (int e = KEEP; e < count; ++e) {
    const long long off = (zoff + block_of(e)) * (BS * BS);
    float d[EPL], v[EPL];
    load_vec<T, EPL>(dy + off, d); load_vec<T, EPL>(yv + off, v);
#pragma unroll
    for (int i = 0; i < EPL; ++i) s += d[i] * v[i];
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
  for (int e = 0; e < KEEP; ++e) {
    if (e < count) {
      const long long off = (zoff + block_of(e)) * (BS * BS);
      float o[EPL];
#pragma unroll
      for (int i = 0; i < EPL; ++i) o[i] = (kd[e][i] - s) * ky[e][i] * p.scale;
      store_vec<TD, EPL>(dx + off, o);
    }
  }
  for (int e = KEEP; e < count; ++e) {
    const long long off = (zoff + block_of(e)) * (BS * BS);
    float d[EPL], v[EPL];
    load_vec<T, EPL>(dy + off, d); load_vec<T, EPL>(yv + off, v);
#pragma unroll
    for (int i = 0; i < EPL; ++i) d[i] = (d[i] - s) * v[i] * p.scale;
    store_vec<TD, EPL>(dx + off, d);
  }
}

template <int BS>
__global__ void bst_autoregressive_mask_kernel(const int32_t* __restrict__ nt_lut, long long nt_head_stride,
                                               const void* __restrict__ mask_in, void* __restrict__ mask_out,
                                               int blocks, int ak) {
  using MT = typename MaskWord<BS>::type;
  const int hl = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // (blk, row)
  if (idx >= blocks * BS) return;
  const int blk = idx / BS, row = idx % BS;
  const int32_t* nt = nt_lut + (long long)hl * nt_head_stride;
  const int qb = nt[2 * blk], kb = nt[2 * blk + 1];
  const MT* in = reinterpret_cast<const MT*>(mask_in) + (long long)hl * blocks * BS;
  MT* out = reinterpret_cast<MT*>(mask_out) + (long long)hl * blocks * BS;
  out[idx] = (MT)autoregress_word<BS>((uint64_t)in[idx], ak, kb, qb * BS + row);
}

}  // namespace bsmm
