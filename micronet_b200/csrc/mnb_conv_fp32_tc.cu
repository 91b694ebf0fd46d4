// fp32 convolution with few input channels (the un-quantized FIRST layer of every QAT model: 3 -> 192/256,
// 5x5 or 3x3; nin_gc.py:82, nin.py, resnet.py) on tcgen05 tensor cores: forward and weight gradient.
//
// C*R*S (75 for 3x5x5) is far too small a reduction for a per-tap implicit GEMM (one MMA K-step would carry 3
// real channels out of 16), so this layer uses a real im2col operand, built in
// shared memory from a zero-padded input patch:
//
//   forward : y[b, n, pos]  = bias[n] + sum_kk  Xcol[pos, kk] * w[n, kk]      M = 128 positions, N = Cout, K = kk
//   wgrad   : dw[n, kk]     = sum_{b, pos}      dy[b, n, pos] * Xcol[pos, kk] M = 128 channels,  N = kk,   K = positions
//
// fp32 accuracy on bf16 tensor cores: every fp32 value is split exactly into three bf16 pieces (hi + mid + lo) and
// the six products down to 2^-16 relative weight (hh, hm, mh, hl, lh, mm) are accumulated in fp32; the dropped
// pieces are <= 2^-24 relative: the error is that of an fp32 convolution with a different summation order.
//
// Both kernels are persistent (one CTA per SM), HBM-bound by the one large tensor they stream (y written once,
// dy read once): forward 128 positions x Cout x 4 B per tile, weight gradient 32 positions x Cout x 4 B per step.
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>

#include "mnb_common.cuh"
#include "mnb_tc.cuh"

namespace tcfp32 {

constexpr int NTHREADS = 512;
constexpr int kMaxDynSmem = 227 * 1024 - 2560;
constexpr int SUB = 32;  // positions per weight-gradient step

struct Params {
  int B, C, K, H, W, R, pad;
  int KR, KP;         // C*R*R and its multiple-of-16 padding
  int NP;             // forward: Cout padded to 16 (MMA N); wgrad: Cout padded to 128 (MMA M halves)
  int TH, PH, PW;     // tile = TH full rows (TH * W = 128); patch = C x PH x PW floats (zero padded)
  int tiles_per_img, n_tiles;
  int nbuf_a, acc_cols, tmem_cols;
  int off_b, off_a, off_patch, off_tab, off_sum, sum_bytes, a_term_bytes, a_buf_bytes, b_term_bytes, patch_bytes;
  const float* x; const float* w; const float* bias; float* y;
  const float* dy; float* partial;
  int* err;
  int dbg;   // MNB_FCONV_DEBUG bit mask (timing experiments only): 1 skip im2col/dy conversion, 2 skip MMAs, 4 skip stores/drain adds, 8 skip x conversion
};

struct alignas(16) Shared {
  uint64_t a_full[2], a_empty[2], acc_full[2], acc_empty[2], done;
  uint32_t tmem_slot;
  uint32_t abort;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void split3_pair(float a, float b, uint32_t& hp, uint32_t& mp, uint32_t& lp) {
  hp = pack_bf16x2(a, b);
  const float ra = a - __uint_as_float(hp << 16), rb = b - __uint_as_float(hp & 0xffff0000u);
  mp = pack_bf16x2(ra, rb);
  const float la = ra - __uint_as_float(mp << 16), lb = rb - __uint_as_float(mp & 0xffff0000u);
  lp = pack_bf16x2(la, lb);
}
// eight fp32 values -> one 16-byte row of each of the three operand planes
__device__ __forceinline__ void store_split8(const float (&v)[8], uint8_t* dst, int term_bytes) {
  uint32_t hp[4], mp[4], lp[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) split3_pair(v[2 * j], v[2 * j + 1], hp[j], mp[j], lp[j]);
  *reinterpret_cast<uint4*>(dst) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
  *reinterpret_cast<uint4*>(dst + term_bytes) = make_uint4(mp[0], mp[1], mp[2], mp[3]);
  *reinterpret_cast<uint4*>(dst + 2 * term_bytes) = make_uint4(lp[0], lp[1], lp[2], lp[3]);
}
__device__ __forceinline__ void conv_bar_sync(int nthreads) {  // named barrier 1: converter warps only
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// The six (A piece, B piece) products kept, SMALLEST FIRST.  The tensor core truncates the running fp32 accumulator
// after every MMA (about half an ulp of |D|, always toward zero), so the 2^-16 and 2^-8 products are added while
// |D| is still tiny and only the hi x hi MMAs run at full magnitude.
__device__ __constant__ int kProdA[6] = {1, 2, 0, 1, 0, 0};
__device__ __constant__ int kProdB[6] = {1, 0, 2, 0, 1, 0};

// zero-padded input patch of one tile: patch[c][pr][pc] = x[b, c, h0 - pad + pr, pc - pad].  It is fetched one tile
// ahead: the first PF elements of every converter thread wait in registers while the current tile is converted
// (patch_fetch), and are written to the other patch buffer afterwards (patch_commit, which also moves the rare
// remainder of a patch larger than PF * nconv directly).
constexpr int PF = 4;
__device__ __forceinline__ float patch_element(const Params& p, int i, int b, int h0) {
  const int pc = i % p.PW, t = i / p.PW;
  const int pr = t % p.PH, c = t / p.PH;
  const int h = h0 - p.pad + pr, w = pc - p.pad;
  return (h >= 0 && h < p.H && w >= 0 && w < p.W) ? __ldg(p.x + (((int64_t)b * p.C + c) * p.H + h) * p.W + w) : 0.f;
}
__device__ __forceinline__ void patch_fetch(const Params& p, int tile, int ct, int nconv, float (&v)[PF]) {
  const int b = tile / p.tiles_per_img, h0 = (tile - b * p.tiles_per_img) * p.TH;
  const int n = p.C * p.PH * p.PW;
#pragma unroll
  for (int k = 0; k < PF; ++k) {
    const int i = ct + k * nconv;
    v[k] = i < n ? patch_element(p, i, b, h0) : 0.f;
  }
}
__device__ __forceinline__ void patch_commit(const Params& p, float* patch, int tile, int ct, int nconv, const float (&v)[PF]) {
  const int b = tile / p.tiles_per_img, h0 = (tile - b * p.tiles_per_img) * p.TH;
  const int n = p.C * p.PH * p.PW;
#pragma unroll
  for (int k = 0; k < PF; ++k) {
    const int i = ct + k * nconv;
    if (i < n) patch[i] = v[k];
  }
  for (int i = ct + PF * nconv; i < n; i += nconv) patch[i] = patch_element(p, i, b, h0);
}

// ------------------------------------------------------------------------------------------------ forward
// warps: 0 = MMA issue, 4..7 = epilogue (TMEM lane quarters), the other 11 = im2col converters
constexpr int FWD_NCONV = NTHREADS - 32 - 128;

__global__ void __launch_bounds__(NTHREADS, 1) fwd_kernel(const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ Shared sh;
  __shared__ __align__(16) float epi_bias[256];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* bop = smem + p.off_b;
  uint8_t* aop = smem + p.off_a;
  int* tab = reinterpret_cast<int*>(smem + p.off_tab);
  const int kchunks = p.KP / 8;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&sh.a_full[i], FWD_NCONV / 32); tc::mbar_init(&sh.a_empty[i], 1);
      tc::mbar_init(&sh.acc_full[i], 1); tc::mbar_init(&sh.acc_empty[i], 4);
    }
    sh.abort = 0;
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&sh.tmem_slot)),
                 "r"((uint32_t)p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int n = tid; n < 256; n += NTHREADS) epi_bias[n] = (p.bias && n < p.K) ? __ldg(p.bias + n) : 0.f;
  // resident B operand: w[n][kk] as K-major core matrices [piece][kk / 8][n][8], zero beyond Cout / KR
  for (int i = tid; i < kchunks * p.NP; i += NTHREADS) {
    const int j = i / p.NP, n = i - j * p.NP;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int kk = j * 8 + e;
      v[e] = (n < p.K && kk < p.KR) ? __ldg(p.w + (int64_t)n * p.KR + kk) : 0.f;
    }
    store_split8(v, bop + (size_t)i * 16, p.b_term_bytes);
  }
  for (int kk = tid; kk < p.KP; kk += NTHREADS) {
    int off = -1;
    if (kk < p.KR) {
      const int s = kk % p.R, t = kk / p.R;
      const int r = t % p.R, c = t / p.R;
      off = (c * p.PH + r) * p.PW + s;
    }
    tab[kk] = off;
  }
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sh.tmem_slot;

  if (warp == 0) {
    // ================================================================= MMA issuer (warp-converged, lane 0 issues)
    const uint32_t lead = lane == 0;
    const uint32_t idesc = tc::make_idesc(1, 1, 1, 128, (uint32_t)p.NP);
    const uint64_t a_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(aop), 128u * 16u, 128u);
    const uint64_t b_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(bop), (uint32_t)p.NP * 16u, 128u);
    const uint32_t a_term16 = (uint32_t)p.a_term_bytes >> 4, b_term16 = (uint32_t)p.b_term_bytes >> 4;
    const uint32_t a_buf16 = (uint32_t)p.a_buf_bytes >> 4;
    const uint32_t a_step16 = 2u * 128u, b_step16 = 2u * (uint32_t)p.NP;   // one K16 step = two 8-wide chunks
    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
      const uint32_t ab = p.nbuf_a == 2 ? (t & 1u) : 0u, aph = p.nbuf_a == 2 ? ((t >> 1) & 1u) : (t & 1u);
      const uint32_t acc = t & 1u, cph = (t >> 1) & 1u;
      tc::mbar_wait_soft(&sh.acc_empty[acc], cph ^ 1u, p.err, 501, &sh.abort);
      tc::mbar_wait_soft(&sh.a_full[ab], aph, p.err, 502, &sh.abort);
      tc::tc_fence_after();
      const uint32_t d_tmem = tmem + acc * (uint32_t)p.acc_cols;
      for (int q = (p.dbg & 2) ? 6 : 0; q < 6; ++q) {
        const uint64_t aq = a_desc0 + (uint64_t)(ab * a_buf16 + (uint32_t)kProdA[q] * a_term16);
        const uint64_t bq = b_desc0 + (uint64_t)((uint32_t)kProdB[q] * b_term16);
        for (int ks = 0; ks < p.KP / 16; ++ks)
          tc::mma_f16_guarded(d_tmem, aq + (uint64_t)((uint32_t)ks * a_step16), bq + (uint64_t)((uint32_t)ks * b_step16), idesc,
                              (uint32_t)(ks | q) != 0u, lead);
      }
      if (lead) { tc::mma_commit(&sh.a_empty[ab]); tc::mma_commit(&sh.acc_full[acc]); }
      __syncwarp();
    }
  } else if (warp >= 4 && warp < 8) {
    // ================================================================= epilogue: TMEM -> + bias -> y (NCHW)
    const int q = warp - 4, m = q * 32 + lane;
    const int64_t plane = (int64_t)p.H * p.W;
    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
      const int b = tile / p.tiles_per_img, h0 = (tile - b * p.tiles_per_img) * p.TH;
      const uint32_t acc = t & 1u, cph = (t >> 1) & 1u;
      if (!tc::mbar_wait(&sh.acc_full[acc], cph, p.err, 503)) break;
      tc::tc_fence_after();
      float* dst = p.y + (int64_t)b * p.K * plane + (int64_t)h0 * p.W + m;
      const uint32_t t_row = tmem + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)p.acc_cols;
      for (int n0 = 0; n0 < p.NP; n0 += 64) {
        // two 32-column chunks per TMEM round trip; bias as vector loads from shared memory up front so that the
        // store loop is a pure FADD + STG stream (a per-element bias load serialises against the stores)
        uint32_t r0[32], r1[32];
        const bool two = n0 + 32 < p.NP;
        tc::tmem_ld_32x32(t_row + (uint32_t)n0, r0);
        if (two) tc::tmem_ld_32x32(t_row + (uint32_t)n0 + 32u, r1);
        tc::tmem_ld_wait();
        if (p.dbg & 4) continue;
#pragma unroll
        for (int hc = 0; hc < 2; ++hc) {
          if (hc == 1 && !two) break;
          const int nb = n0 + 32 * hc;
          float bs[32];
#pragma unroll
          for (int v = 0; v < 8; ++v) {
            const float4 c4 = *reinterpret_cast<const float4*>(&epi_bias[nb + 4 * v]);
            bs[4 * v] = c4.x; bs[4 * v + 1] = c4.y; bs[4 * v + 2] = c4.z; bs[4 * v + 3] = c4.w;
          }
          float* op = dst + (int64_t)nb * plane;
#pragma unroll
          for (int j = 0; j < 32; ++j, op += plane)
            if (nb + j < p.K) *op = __uint_as_float(hc ? r1[j] : r0[j]) + bs[j];
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&sh.acc_empty[acc]);
    }
  } else {
    // ================================================================= converters: patch -> im2col A operand
    const int ct = warp < 4 ? tid - 32 : tid - 32 - 128;   // 0 .. FWD_NCONV-1
    float* patch0 = reinterpret_cast<float*>(smem + p.off_patch);
    const int items = 128 * kchunks;
    const int patch_floats = p.patch_bytes / 4;
    float pre[PF];
    if ((int)blockIdx.x < p.n_tiles) {
      patch_fetch(p, blockIdx.x, ct, FWD_NCONV, pre);
      patch_commit(p, patch0, blockIdx.x, ct, FWD_NCONV, pre);
    }
    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
      const float* patch = patch0 + (size_t)(t & 1u) * patch_floats;
      conv_bar_sync(FWD_NCONV);   // every converter committed its part of this tile's patch
      const int next = tile + (int)gridDim.x;
      if (next < p.n_tiles) patch_fetch(p, next, ct, FWD_NCONV, pre);
      const uint32_t ab = p.nbuf_a == 2 ? (t & 1u) : 0u, aph = p.nbuf_a == 2 ? ((t >> 1) & 1u) : (t & 1u);
      if (!tc::mbar_wait(&sh.a_empty[ab], aph ^ 1u, p.err, 504)) break;
      uint8_t* abuf = aop + (size_t)ab * p.a_buf_bytes;
      for (int i = (p.dbg & 1) ? items : ct; i < items; i += FWD_NCONV) {
        const int j = i >> 7, m = i & 127;
        const int base = (m / p.W) * p.PW + (m % p.W);
        int off[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) off[e] = tab[j * 8 + e];
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = off[e] >= 0 ? patch[off[e] + base] : 0.f;
        store_split8(v, abuf + (size_t)i * 16, p.a_term_bytes);
      }
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&sh.a_full[ab]);
      if (next < p.n_tiles) patch_commit(p, patch0 + (size_t)((t + 1) & 1u) * patch_floats, next, ct, FWD_NCONV, pre);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc::tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols));
  }
}

// ------------------------------------------------------------------------------------------------ weight gradient
// warps: 0 = MMA issue, 4..7 = accumulator drain, the other 11 = converters (dy split + im2col of x).
// A TMEM accumulator only ever holds FLUSH tiles (48 MMAs per column set and tile): the drain warps add it into an
// fp32 running sum in shared memory with round-to-nearest adds.  The accumulator truncation (see kProdA) is a bias
// proportional to chain length x |D|, so short chains matter: measured 8e-6 relative error for one chain over the
// whole batch, 3e-6 with FLUSH = 4, ~1e-6 with FLUSH = 1.
constexpr int WG_NCONV = NTHREADS - 32 - 128;
constexpr int FLUSH = 1;

__global__ void __launch_bounds__(NTHREADS, 1) wgrad_kernel(const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ Shared sh;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* bop = smem + p.off_b;   // Xcol^T : [buf][piece][pos / 8][kk][8 pos]
  uint8_t* aop = smem + p.off_a;   // dy     : [buf][piece][pos / 8][channel][8 pos]
  int* tab = reinterpret_cast<int*>(smem + p.off_tab);
  const int halves = p.NP / 128;
  const int nsub = 128 / SUB;
  const int my_tiles = (p.n_tiles > (int)blockIdx.x) ? (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&sh.a_full[i], WG_NCONV / 32); tc::mbar_init(&sh.a_empty[i], 1);
      tc::mbar_init(&sh.acc_full[i], 1); tc::mbar_init(&sh.acc_empty[i], 4);
    }
    sh.abort = 0;
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&sh.tmem_slot)),
                 "r"((uint32_t)p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // operand buffers start as zeros (channel rows >= Cout and im2col rows >= KR are never written), and so does the
  // running sum that follows them
  for (int i = tid; i < (2 * (p.a_buf_bytes + 3 * p.b_term_bytes) + p.sum_bytes) / 16; i += NTHREADS)
    reinterpret_cast<uint4*>(smem + p.off_b)[i] = make_uint4(0, 0, 0, 0);
  for (int kk = tid; kk < p.KP; kk += NTHREADS) {
    int off = -1;
    if (kk < p.KR) {
      const int s = kk % p.R, t = kk / p.R;
      const int r = t % p.R, c = t / p.R;
      off = (c * p.PH + r) * p.PW + s;
    }
    tab[kk] = off;
  }
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sh.tmem_slot;
  const int b_buf_bytes = 3 * p.b_term_bytes;

  if (warp == 0) {
    // ================================================================= MMA issuer
    const uint32_t lead = lane == 0;
    const uint32_t idesc = tc::make_idesc(1, 1, 1, 128, (uint32_t)p.KP);
    const uint64_t a_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(aop), (uint32_t)p.NP * 16u, 128u);
    const uint64_t b_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(bop), (uint32_t)p.KP * 16u, 128u);
    const uint32_t a_term16 = (uint32_t)p.a_term_bytes >> 4, b_term16 = (uint32_t)p.b_term_bytes >> 4;
    const uint32_t a_buf16 = (uint32_t)p.a_buf_bytes >> 4, b_buf16 = (uint32_t)b_buf_bytes >> 4;
    const uint32_t a_step16 = 2u * (uint32_t)p.NP, b_step16 = 2u * (uint32_t)p.KP;
    uint32_t it = 0, t = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
      const uint32_t grp = t / FLUSH, in_grp = t % FLUSH;
      const uint32_t acc = grp & 1u, cph = (grp >> 1) & 1u;
      if (in_grp == 0) tc::mbar_wait_soft(&sh.acc_empty[acc], cph ^ 1u, p.err, 514, &sh.abort);
      const uint32_t d_base = tmem + acc * 256u;
      for (int sub = 0; sub < nsub; ++sub, ++it) {
        const uint32_t ob = it & 1u, oph = (it >> 1) & 1u;
        tc::mbar_wait_soft(&sh.a_full[ob], oph, p.err, 511, &sh.abort);
        tc::tc_fence_after();
        for (int hf = (p.dbg & 2) ? halves : 0; hf < halves; ++hf) {
          for (int q = 0; q < 6; ++q) {
            const uint64_t aq = a_desc0 + (uint64_t)(ob * a_buf16 + (uint32_t)kProdA[q] * a_term16 + (uint32_t)hf * 128u);
            const uint64_t bq = b_desc0 + (uint64_t)(ob * b_buf16 + (uint32_t)kProdB[q] * b_term16);
#pragma unroll
            for (int ks = 0; ks < SUB / 16; ++ks)
              tc::mma_f16_guarded(d_base + (uint32_t)hf * 128u, aq + (uint64_t)((uint32_t)ks * a_step16),
                                  bq + (uint64_t)((uint32_t)ks * b_step16), idesc,
                                  (in_grp | (uint32_t)sub | (uint32_t)ks | (uint32_t)q) != 0u, lead);
          }
        }
        if (lead) tc::mma_commit(&sh.a_empty[ob]);
        __syncwarp();
      }
      if (in_grp == FLUSH - 1 || tile + (int)gridDim.x >= p.n_tiles) {
        if (lead) tc::mma_commit(&sh.acc_full[acc]);
        __syncwarp();
      }
    }
  } else if (warp < 4 || warp >= 8) {
    // ================================================================= converters
    const int ct = warp < 4 ? tid - 32 : tid - 32 - 128;
    float* patch0 = reinterpret_cast<float*>(smem + p.off_patch);
    const int64_t plane = (int64_t)p.H * p.W;
    const int d_items = p.K * (SUB / 8), x_items = p.KR * (SUB / 8);
    const int patch_floats = p.patch_bytes / 4;
    // dy is fetched one step (32 positions) ahead into registers: up to DMAX x 32 bytes per thread in flight while the
    // previous step is split and stored
    constexpr int DMAX = 3;
    float4 dpre[DMAX][2];
    auto fetch_dy = [&](int tile, int sub) {
      const int b = tile / p.tiles_per_img, h0 = (tile - b * p.tiles_per_img) * p.TH;
      const float* dy_tile = p.dy + (int64_t)b * p.K * plane + (int64_t)h0 * p.W + sub * SUB;
#pragma unroll
      for (int k = 0; k < DMAX; ++k) {
        const int i = ct + k * WG_NCONV;
        if (i < d_items) {
          const int n = i / (SUB / 8), j = i - n * (SUB / 8);
          const float4* src = reinterpret_cast<const float4*>(dy_tile + (int64_t)n * plane + j * 8);
          dpre[k][0] = __ldg(src); dpre[k][1] = __ldg(src + 1);
        }
      }
    };
    float pre[PF];
    if ((int)blockIdx.x < p.n_tiles) {
      patch_fetch(p, blockIdx.x, ct, WG_NCONV, pre);
      patch_commit(p, patch0, blockIdx.x, ct, WG_NCONV, pre);
      fetch_dy(blockIdx.x, 0);
    }
    uint32_t it = 0, t = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
      const float* patch = patch0 + (size_t)(t & 1u) * patch_floats;
      conv_bar_sync(WG_NCONV);
      const int next = tile + (int)gridDim.x;
      if (next < p.n_tiles) patch_fetch(p, next, ct, WG_NCONV, pre);
      for (int sub = 0; sub < nsub; ++sub, ++it) {
        const uint32_t ob = it & 1u, oph = (it >> 1) & 1u;
        float4 dcur[DMAX][2];
#pragma unroll
        for (int k = 0; k < DMAX; ++k) { dcur[k][0] = dpre[k][0]; dcur[k][1] = dpre[k][1]; }
        if (sub + 1 < nsub) fetch_dy(tile, sub + 1);
        else if (next < p.n_tiles) fetch_dy(next, 0);
        if (!tc::mbar_wait(&sh.a_empty[ob], oph ^ 1u, p.err, 512)) goto done;
        uint8_t* abuf = aop + (size_t)ob * p.a_buf_bytes;
        uint8_t* bbuf = bop + (size_t)ob * b_buf_bytes;
        // dy: item = (channel n, 8-position chunk j): 32 contiguous bytes of global memory
        if (!(p.dbg & 1)) {
#pragma unroll
          for (int k = 0; k < DMAX; ++k) {
            const int i = ct + k * WG_NCONV;
            if (i < d_items) {
              const int n = i / (SUB / 8), j = i - n * (SUB / 8);
              const float v[8] = {dcur[k][0].x, dcur[k][0].y, dcur[k][0].z, dcur[k][0].w,
                                  dcur[k][1].x, dcur[k][1].y, dcur[k][1].z, dcur[k][1].w};
              store_split8(v, abuf + ((size_t)j * p.NP + n) * 16, p.a_term_bytes);
            }
          }
        }
        // Xcol^T: item = (kk, 8-position chunk j): 8 consecutive patch columns
        for (int i = (p.dbg & 8) ? x_items : ct; i < x_items; i += WG_NCONV) {
          const int kk = i / (SUB / 8), j = i - kk * (SUB / 8);
          const int m = sub * SUB + j * 8;
          const float* src = patch + tab[kk] + (m / p.W) * p.PW + (m % p.W);
          float v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = src[e];
          store_split8(v, bbuf + ((size_t)j * p.KP + kk) * 16, p.b_term_bytes);
        }
        tc::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&sh.a_full[ob]);
      }
      if (next < p.n_tiles) patch_commit(p, patch0 + (size_t)((t + 1) & 1u) * patch_floats, next, ct, WG_NCONV, pre);
    }
  } else {
    // ================================================================= drain: TMEM accumulators -> fp32 running sum -> partial dw
    const int q = warp - 4, m = q * 32 + lane;
    float* sum = reinterpret_cast<float*>(smem + p.off_sum);   // [half][kk][128 channels]
    const int groups = (my_tiles + FLUSH - 1) / FLUSH;
    for (int grp = 0; grp < groups; ++grp) {
      const uint32_t acc = grp & 1u, cph = (grp >> 1) & 1u;
      if (!tc::mbar_wait(&sh.acc_full[acc], cph, p.err, 513)) goto done;
      tc::tc_fence_after();
      for (int hf = 0; hf < halves; ++hf) {
        for (int k0 = 0; k0 < p.KP; k0 += 32) {
          uint32_t r[32];
          tc::tmem_ld_32x32(tmem + ((uint32_t)(q * 32) << 16) + acc * 256u + (uint32_t)(hf * 128 + k0), r);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (k0 + j < p.KP && !(p.dbg & 4)) sum[((hf * p.KP) + k0 + j) * 128 + m] += __uint_as_float(r[j]);
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&sh.acc_empty[acc]);
    }
    float* mine = p.partial + (int64_t)blockIdx.x * p.K * p.KR;
    for (int hf = 0; hf < halves; ++hf) {
      const int n = hf * 128 + m;
      if (n < p.K)
        for (int kk = 0; kk < p.KR; ++kk) mine[(int64_t)n * p.KR + kk] = sum[((hf * p.KP) + kk) * 128 + m];
    }
  }
done:
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc::tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols));
  }
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partial, int n, int ranks,
                                                              float* __restrict__ dw) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int j = 0; j < ranks; ++j) s += partial[(int64_t)j * n + i];
    dw[i] = s;
  }
}

static int plan(const mnb_conv_shape* s, bool wgrad, Params& p, int& smem_bytes) {
  MNB_REQUIRE(s != nullptr, "conv shape is NULL");
  auto unsupported = [](const char* why) { return mnb_fail(MNB_E_UNSUPPORTED, "fp32 tc conv: %s", why); };
  p.B = s->batch; p.C = s->in_c; p.K = s->out_c; p.H = s->in_h; p.W = s->in_w; p.R = s->ker_h;
  MNB_REQUIRE(p.B > 0 && p.C > 0 && p.K > 0 && p.H > 0 && p.W > 0 && s->groups > 0, "bad conv shape");
  if (s->groups != 1 || s->stride_h != 1 || s->stride_w != 1 || s->dil_h != 1 || s->dil_w != 1)
    return unsupported("groups / stride / dilation != 1");
  if (s->ker_h != s->ker_w || (p.R & 1) == 0 || s->pad_h != p.R / 2 || s->pad_w != p.R / 2)
    return unsupported("not a 'same' odd square filter");
  p.pad = p.R / 2;
  p.KR = p.C * p.R * p.R;
  p.KP = (p.KR + 15) / 16 * 16;
  if (p.KP > 128) return unsupported("C*R*S > 128 (use the per-tap implicit GEMM)");
  if (p.K > 256) return unsupported("more than 256 output channels");   // also: K * 4 dy items <= DMAX * WG_NCONV
  if (p.W < 8 || p.W > 128 || 128 % p.W || (p.H * p.W) % 128) return unsupported("image rows do not tile into 128 positions");
  if ((int64_t)p.B * p.K * p.H * p.W >= (1ll << 31)) return unsupported("tensor too large");
  p.TH = 128 / p.W;
  p.PH = p.TH + 2 * p.pad; p.PW = p.W + 2 * p.pad;
  p.tiles_per_img = p.H / p.TH;
  p.n_tiles = p.B * p.tiles_per_img;
  p.patch_bytes = (p.C * p.PH * p.PW * 4 + 8 * 4 + 15) / 16 * 16;   // + slack: the wgrad gather of a padded kk row may overrun
  const int kchunks = p.KP / 8;
  if (!wgrad) {
    p.NP = (p.K + 15) / 16 * 16;
    p.b_term_bytes = kchunks * p.NP * 16;
    p.a_term_bytes = kchunks * 128 * 16;
    p.a_buf_bytes = 3 * p.a_term_bytes;
    p.off_b = 0;
    p.off_a = 3 * p.b_term_bytes;
    p.acc_cols = p.NP <= 32 ? 32 : p.NP <= 64 ? 64 : p.NP <= 128 ? 128 : 256;
    p.tmem_cols = 2 * p.acc_cols;
    for (p.nbuf_a = 2; p.nbuf_a >= 1; --p.nbuf_a) {
      p.off_patch = p.off_a + p.nbuf_a * p.a_buf_bytes;
      p.off_tab = p.off_patch + 2 * p.patch_bytes;
      smem_bytes = p.off_tab + p.KP * 4;
      if (smem_bytes <= kMaxDynSmem) break;
    }
    if (p.nbuf_a < 1) return unsupported("shared memory budget");
  } else {
    p.NP = (p.K + 127) / 128 * 128;
    p.a_term_bytes = (SUB / 8) * p.NP * 16;
    p.a_buf_bytes = 3 * p.a_term_bytes;
    p.b_term_bytes = (SUB / 8) * p.KP * 16;
    // [B buf0][B buf1][A buf0][A buf1][running sum] contiguous (zeroed in one sweep by the kernel)
    p.off_b = 0;
    p.off_a = 2 * 3 * p.b_term_bytes;
    p.off_sum = p.off_a + 2 * p.a_buf_bytes;
    p.sum_bytes = (p.NP / 128) * p.KP * 128 * 4;
    p.off_patch = p.off_sum + p.sum_bytes;
    p.off_tab = p.off_patch + 2 * p.patch_bytes;
    smem_bytes = p.off_tab + p.KP * 4;
    p.nbuf_a = 2;
    p.acc_cols = 128;
    p.tmem_cols = 512;   // two accumulator sets of (2 halves x 128 columns)
    if (smem_bytes > kMaxDynSmem) return unsupported("shared memory budget");
  }
  return 0;
}

static int grid_size(const Params& p) { return std::max(1, std::min(p.n_tiles, MNB_NUM_SMS)); }
static int debug_mask() {
  static const int m = [] { const char* e = getenv("MNB_FCONV_DEBUG"); return e ? atoi(e) : 0; }();
  return m;
}

}  // namespace tcfp32

extern "C" int mnb_fconv2d_fwd_tc(const mnb_conv_shape* s, const float* x, const float* w, const float* bias, float* y,
                                  int32_t* err_flag, mnb_stream_t stream) {
  using namespace tcfp32;
  MNB_REQUIRE(s && x && w && y && err_flag, "NULL pointer");
  Params p{};
  int smem_bytes = 0;
  if (int e = plan(s, false, p, smem_bytes)) return e;
  p.x = x; p.w = w; p.bias = bias; p.y = y; p.err = err_flag; p.dbg = debug_mask();
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t ce = cudaFuncSetAttribute(fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem);
    if (ce != cudaSuccess) return mnb_fail((int)ce, "cudaFuncSetAttribute: %s", cudaGetErrorString(ce));
    attr_set = true;
  }
  fwd_kernel<<<grid_size(p), NTHREADS, smem_bytes, (cudaStream_t)stream>>>(p);
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int64_t mnb_fconv2d_wgrad_tc_scratch_bytes(const mnb_conv_shape* s) {
  tcfp32::Params p{};
  int smem = 0;
  if (tcfp32::plan(s, true, p, smem)) return -1;
  return (int64_t)tcfp32::grid_size(p) * p.K * p.KR * 4;
}

extern "C" int mnb_fconv2d_wgrad_tc(const mnb_conv_shape* s, const float* dy, const float* x, float* dw, void* scratch,
                                    int32_t* err_flag, mnb_stream_t stream) {
  using namespace tcfp32;
  MNB_REQUIRE(s && dy && x && dw && scratch && err_flag, "NULL pointer");
  MNB_REQUIRE((reinterpret_cast<uintptr_t>(dy) & 15) == 0, "dy must be 16-byte aligned");
  Params p{};
  int smem_bytes = 0;
  if (int e = plan(s, true, p, smem_bytes)) return e;
  p.x = x; p.dy = dy; p.partial = reinterpret_cast<float*>(scratch); p.err = err_flag; p.dbg = debug_mask();
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t ce = cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem);
    if (ce != cudaSuccess) return mnb_fail((int)ce, "cudaFuncSetAttribute: %s", cudaGetErrorString(ce));
    attr_set = true;
  }
  const int grid = grid_size(p);
  cudaStream_t st = (cudaStream_t)stream;
  wgrad_kernel<<<grid, NTHREADS, smem_bytes, st>>>(p);
  const int n = p.K * p.KR;
  reduce_partials_kernel<<<std::min(mnb_ceil_div(n, 256), MNB_NUM_SMS * 4), 256, 0, st>>>(p.partial, n, grid, dw);
  MNB_LAUNCHED(2);
  return 0;
}
