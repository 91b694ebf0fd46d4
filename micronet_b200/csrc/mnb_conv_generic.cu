// Generic implicit-GEMM convolution kernels (any stride / padding / dilation / groups).
//
// This is the shape-agnostic path of the engine: forward (exact s32 accumulation when both
// operands are integer levels, fp32 otherwise), dgrad fused with the activation STE mask, and
// split-K wgrad with a deterministic two-stage reduction.  Hot, regular shapes are taken by the
// tcgen05 tensor-core kernels in mnb_pk.cu and mnb_conv_fp32_tc.cu; everything else (C_in = 3 stems, 10-way heads,
// odd strides, asymmetric weights) lands here.
//
// GEMM views (per group g; Cg = in_c/groups, Ng = out_c/groups, RS = kh*kw):
//   fwd   : M = B*P*Q      N = Ng      K = Cg*RS     y[b,gNg+n,p,q]  = sum_k A(m,k) W[gNg+n, k]
//   dgrad : M = B*H*W      N = Cg      K = Ng*RS     dx[b,gCg+n,h,w] = sum_k dY(m,k) Wq[gNg+ko, n, rs]
//   wgrad : M = Ng         N = Cg*RS   K = B*P*Q     dWq[gNg+m, n]   = sum_k dY[b,gNg+m,pq] Xq(k,n)
#include <type_traits>

#include "mnb_common.cuh"

namespace {

constexpr int BM = 64, BK = 16, NT = 256;

struct ConvGeom {
  int B, C, H, W, K, R, S, sh, sw, ph, pw, dh, dw, G, P, Q, Cg, Ng, RS;
};

static int make_geom(const mnb_conv_shape* s, ConvGeom& g) {
  MNB_REQUIRE(s != nullptr, "conv shape is NULL");
  g.B = s->batch; g.C = s->in_c; g.H = s->in_h; g.W = s->in_w; g.K = s->out_c; g.R = s->ker_h; g.S = s->ker_w;
  g.sh = s->stride_h; g.sw = s->stride_w; g.ph = s->pad_h; g.pw = s->pad_w; g.dh = s->dil_h; g.dw = s->dil_w;
  g.G = s->groups;
  MNB_REQUIRE(g.B > 0 && g.C > 0 && g.H > 0 && g.W > 0 && g.K > 0 && g.R > 0 && g.S > 0, "non-positive conv dims");
  MNB_REQUIRE(g.sh > 0 && g.sw > 0 && g.dh > 0 && g.dw > 0 && g.ph >= 0 && g.pw >= 0, "bad stride/dilation/padding");
  MNB_REQUIRE(g.G > 0 && g.C % g.G == 0 && g.K % g.G == 0, "channels (%d,%d) not divisible by groups %d", g.C, g.K, g.G);
  g.P = (g.H + 2 * g.ph - g.dh * (g.R - 1) - 1) / g.sh + 1;
  g.Q = (g.W + 2 * g.pw - g.dw * (g.S - 1) - 1) / g.sw + 1;
  MNB_REQUIRE(g.P > 0 && g.Q > 0, "empty conv output");
  g.Cg = g.C / g.G; g.Ng = g.K / g.G; g.RS = g.R * g.S;
  return 0;
}

struct FwdArgs {
  ConvGeom g;
  const uint8_t* a_codes; const float* a_f32; int a_off; const float* a_off_zp; const float* a_scale;
  const int16_t* w_int; const float* w_scale; const float* w_f32; const float* bias;
  float* y;
};

// ---------------------------------------------------------------- forward
template <typename Acc, int BN>
__global__ void __launch_bounds__(NT) conv_fwd_kernel(FwdArgs a) {
  constexpr int TN = BN / 16;
  __shared__ Acc As[BK][BM];
  __shared__ Acc Bs[BK][BN + 1];
  const ConvGeom& g = a.g;
  const int grp = blockIdx.z;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int M = g.B * g.P * g.Q, Kd = g.Cg * g.RS, PQ = g.P * g.Q;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  // this thread's A pixel (fixed for the whole kernel)
  const int am = tid & (BM - 1), ak0 = tid >> 6;  // 4 k-rows per pass
  const int m = m0 + am;
  const bool m_ok = m < M;
  int ab = 0, ap = 0, aq = 0;
  if (m_ok) { ab = m / PQ; int r = m - ab * PQ; ap = r / g.Q; aq = r - ap * g.Q; }
  const int h0 = ap * g.sh - g.ph, w0 = aq * g.sw - g.pw;
  const int a_off = a.a_off + (a.a_off_zp ? (int)__ldg(a.a_off_zp) : 0);
  const float a_sc = a.a_scale ? __ldg(a.a_scale) : 1.f;
  const int64_t x_img = ((int64_t)ab * g.C + (int64_t)grp * g.Cg) * g.H * g.W;

  const int bk = tid & (BK - 1), bn0 = tid >> 4;  // B: k fastest

  Acc acc[4][TN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = (Acc)0;

  for (int k0 = 0; k0 < Kd; k0 += BK) {
#pragma unroll
    for (int l = 0; l < BK / 4; ++l) {
      const int kk = ak0 + 4 * l, k = k0 + kk;
      Acc v = (Acc)0;
      if (m_ok && k < Kd) {
        int c, r, s;
        if (g.RS == 1) { c = k; r = 0; s = 0; }
        else { c = k / g.RS; int rs = k - c * g.RS; r = rs / g.S; s = rs - r * g.S; }
        const int h = h0 + r * g.dh, w = w0 + s * g.dw;
        if ((unsigned)h < (unsigned)g.H && (unsigned)w < (unsigned)g.W) {
          const int64_t idx = x_img + ((int64_t)c * g.H + h) * g.W + w;
          if (a.a_codes) {
            int e = (int)__ldg(a.a_codes + idx) + a_off;
            if constexpr (std::is_integral<Acc>::value) v = (Acc)e;   // integer accumulate
            else v = (Acc)__fmul_rn((float)e, a_sc);                            // dequantized value
          } else {
            v = (Acc)__ldg(a.a_f32 + idx);
          }
        }
      }
      As[kk][am] = v;
    }
#pragma unroll
    for (int l = 0; l < BN / 16; ++l) {
      const int nn = bn0 + 16 * l, n = n0 + nn, k = k0 + bk;
      Acc v = (Acc)0;
      if (n < g.Ng && k < Kd) {
        const int64_t idx = ((int64_t)grp * g.Ng + n) * Kd + k;
        if constexpr (std::is_integral<Acc>::value) v = (Acc)__ldg(a.w_int + idx);
        else v = (Acc)__ldg(a.w_f32 + idx);
      }
      Bs[bk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      Acc av[4], bv[TN];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][tx + 16 * i];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][ty + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] += av[i] * bv[j];
    }
    __syncthreads();
  }

#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int n = n0 + ty + 16 * j;
    if (n >= g.Ng) continue;
    const int ch = grp * g.Ng + n;
    const float bsv = a.bias ? __ldg(a.bias + ch) : 0.f;
    float sc = 1.f;
    if constexpr (std::is_integral<Acc>::value) sc = __fmul_rn(a_sc, __ldg(a.w_scale + ch));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int mm = m0 + tx + 16 * i;
      if (mm >= M) continue;
      const int b = mm / PQ, pq = mm - b * PQ;
      float v;
      if constexpr (std::is_integral<Acc>::value) v = __fadd_rn(__fmul_rn((float)acc[i][j], sc), bsv);
      else v = (float)acc[i][j] + bsv;
      a.y[((int64_t)b * g.K + ch) * PQ + pq] = v;
    }
  }
}

// ---------------------------------------------------------------- dgrad (+ fused activation STE)
struct DgradArgs {
  ConvGeom g;
  const float* dy; const float* wq; const uint32_t* pass_bits; mnb_act_qparams qp; int has_qp;
  float* dx;
};

template <int BN>
__global__ void __launch_bounds__(NT) conv_dgrad_kernel(DgradArgs a) {
  constexpr int TN = BN / 16;
  __shared__ float As[BK][BM];
  __shared__ float Bs[BK][BN + 1];
  const ConvGeom& g = a.g;
  const int grp = blockIdx.z;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int HW = g.H * g.W, M = g.B * HW, Kd = g.Ng * g.RS, PQ = g.P * g.Q;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  const int am = tid & (BM - 1), ak0 = tid >> 6;
  const int m = m0 + am;
  const bool m_ok = m < M;
  int ab = 0, ah = 0, aw = 0;
  if (m_ok) { ab = m / HW; int r = m - ab * HW; ah = r / g.W; aw = r - ah * g.W; }
  const int64_t dy_img = ((int64_t)ab * g.K + (int64_t)grp * g.Ng) * PQ;
  const int bk = tid & (BK - 1), bn0 = tid >> 4;

  float acc[4][TN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < Kd; k0 += BK) {
#pragma unroll
    for (int l = 0; l < BK / 4; ++l) {
      const int kk = ak0 + 4 * l, k = k0 + kk;
      float v = 0.f;
      if (m_ok && k < Kd) {
        int ko, r, s;
        if (g.RS == 1) { ko = k; r = 0; s = 0; }
        else { ko = k / g.RS; int rs = k - ko * g.RS; r = rs / g.S; s = rs - r * g.S; }
        const int th = ah + g.ph - r * g.dh, tw = aw + g.pw - s * g.dw;
        if (th >= 0 && tw >= 0) {
          int p, q; bool ok;
          if (g.sh == 1 && g.sw == 1) { p = th; q = tw; ok = true; }
          else { p = th / g.sh; q = tw / g.sw; ok = (p * g.sh == th) && (q * g.sw == tw); }
          if (ok && p < g.P && q < g.Q) v = __ldg(a.dy + dy_img + (int64_t)ko * PQ + p * g.Q + q);
        }
      }
      As[kk][am] = v;
    }
#pragma unroll
    for (int l = 0; l < BN / 16; ++l) {
      const int nn = bn0 + 16 * l, n = n0 + nn, k = k0 + bk;
      float v = 0.f;
      if (n < g.Cg && k < Kd) {
        int ko, rs;
        if (g.RS == 1) { ko = k; rs = 0; } else { ko = k / g.RS; rs = k - ko * g.RS; }
        v = __ldg(a.wq + (((int64_t)grp * g.Ng + ko) * g.Cg + n) * g.RS + rs);
      }
      Bs[bk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[4], bv[TN];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][tx + 16 * i];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][ty + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

  MnbActQ q;
  if (a.has_qp) q = mnb_load_actq(a.qp);
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int n = n0 + ty + 16 * j;
    if (n >= g.Cg) continue;
    const int ch = grp * g.Cg + n;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int mm = m0 + tx + 16 * i;
      if (mm >= M) continue;
      const int b = mm / HW, hw = mm - b * HW;
      const int64_t idx = ((int64_t)b * g.C + ch) * HW + hw;
      float v = acc[i][j];
      if (a.has_qp) {
        bool pass = (__ldg(a.pass_bits + (idx >> 5)) >> (idx & 31)) & 1u;
        v = mnb_act_ste_one(q, v, pass);
      }
      a.dx[idx] = v;
    }
  }
}

// ---------------------------------------------------------------- wgrad (split-K, deterministic)
struct WgradArgs {
  ConvGeom g;
  const float* dy; const uint8_t* a_codes; const float* a_f32; int a_off; const float* a_off_zp;
  float* partial;  // [splits][out_c * Cg * RS]
  int splits, k_per_split;
};

template <int BN>
__global__ void __launch_bounds__(NT) conv_wgrad_kernel(WgradArgs a) {
  constexpr int TN = BN / 16;
  __shared__ float As[BK][BM + 1];
  __shared__ float Bs[BK][BN + 1];
  const ConvGeom& g = a.g;
  const int grp = blockIdx.z / a.splits, split = blockIdx.z - grp * a.splits;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int PQ = g.P * g.Q, Kd = g.B * PQ, Nd = g.Cg * g.RS, HW = g.H * g.W;
  const int kbeg = split * a.k_per_split, kend = min(Kd, kbeg + a.k_per_split);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int lk = tid & (BK - 1), l0 = tid >> 4;  // both operands: k (pixel) fastest
  const int a_off = a.a_off + (a.a_off_zp ? (int)__ldg(a.a_off_zp) : 0);

  // this thread's B columns (c, r, s), fixed for the whole kernel
  int bc[TN], br[TN], bs[TN];
  bool bok[TN];
#pragma unroll
  for (int l = 0; l < TN; ++l) {
    const int n = n0 + l0 + 16 * l;
    bok[l] = n < Nd;
    int c = 0, r = 0, s = 0;
    if (bok[l]) { c = n / g.RS; int rs = n - c * g.RS; r = rs / g.S; s = rs - r * g.S; }
    bc[l] = c; br[l] = r * g.dh - g.ph; bs[l] = s * g.dw - g.pw;
  }

  float acc[4][TN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    const int k = k0 + lk;
    const bool k_ok = k < kend;
    int b = 0, p = 0, q = 0, pq = 0;
    if (k_ok) { b = k / PQ; pq = k - b * PQ; p = pq / g.Q; q = pq - p * g.Q; }
#pragma unroll
    for (int l = 0; l < BM / 16; ++l) {
      const int mm = l0 + 16 * l, mo = m0 + mm;
      float v = 0.f;
      if (k_ok && mo < g.Ng) v = __ldg(a.dy + ((int64_t)b * g.K + (int64_t)grp * g.Ng + mo) * PQ + pq);
      As[lk][mm] = v;
    }
#pragma unroll
    for (int l = 0; l < TN; ++l) {
      float v = 0.f;
      if (k_ok && bok[l]) {
        const int h = p * g.sh + br[l], w = q * g.sw + bs[l];
        if ((unsigned)h < (unsigned)g.H && (unsigned)w < (unsigned)g.W) {
          const int64_t idx = ((int64_t)b * g.C + (int64_t)grp * g.Cg + bc[l]) * HW + h * g.W + w;
          v = a.a_codes ? (float)((int)__ldg(a.a_codes + idx) + a_off) : __ldg(a.a_f32 + idx);
        }
      }
      Bs[lk][l0 + 16 * l] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[4], bv[TN];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][tx + 16 * i];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][ty + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* out = a.partial + (int64_t)split * g.K * Nd;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int mo = m0 + tx + 16 * i;
    if (mo >= g.Ng) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int n = n0 + ty + 16 * j;
      if (n < Nd) out[((int64_t)grp * g.Ng + mo) * Nd + n] = acc[i][j];
    }
  }
}

__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial, int64_t n,
                                                           int splits, const float* a_scale,
                                                           float* __restrict__ dwq) {
  const float sc = a_scale ? __ldg(a_scale) : 1.f;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float s = 0.f;
    for (int j = 0; j < splits; ++j) s += partial[(int64_t)j * n + i];
    dwq[i] = a_scale ? __fmul_rn(s, sc) : s;
  }
}

static int pick_bn(int n) { return n <= 16 ? 16 : (n <= 32 ? 32 : 64); }

static void wgrad_plan(const ConvGeom& g, int& bn, int& splits, int& kps) {
  const int Nd = g.Cg * g.RS, Kd = g.B * g.P * g.Q;
  bn = pick_bn(Nd);
  const int64_t tiles = (int64_t)mnb_ceil_div(g.Ng, BM) * mnb_ceil_div(Nd, bn) * g.G;
  int want = (int)std::max<int64_t>(1, (MNB_NUM_SMS * 4) / tiles);
  int maxs = std::max(1, Kd / (BK * 8));
  splits = std::min(std::min(want, maxs), 256);
  kps = mnb_ceil_div(mnb_ceil_div(Kd, splits), BK) * BK;
  splits = mnb_ceil_div(Kd, kps);
}

}  // namespace

extern "C" int mnb_conv2d_fwd(const mnb_conv_shape* s, const mnb_conv_operands* op, float* y,
                              mnb_stream_t stream) {
  FwdArgs a;
  if (int e = make_geom(s, a.g)) return e;
  MNB_REQUIRE(op && y, "NULL operands/output");
  MNB_REQUIRE((op->a_codes != nullptr) != (op->a_f32 != nullptr), "exactly one of a_codes / a_f32 must be given");
  const bool int_path = op->a_codes && op->w_int && !op->w_f32;
  MNB_REQUIRE(int_path || op->w_f32, "fp32 path needs w_f32");
  MNB_REQUIRE(!int_path || op->w_scale, "integer path needs w_scale");
  a.a_codes = op->a_codes; a.a_f32 = op->a_f32; a.a_off = op->a_offset; a.a_off_zp = op->a_offset_zp;
  a.a_scale = op->a_scale; a.w_int = op->w_int; a.w_scale = op->w_scale; a.w_f32 = op->w_f32; a.bias = op->bias;
  a.y = y;
  const ConvGeom& g = a.g;
  const int M = g.B * g.P * g.Q;
  const int bn = pick_bn(g.Ng);
  dim3 grid(mnb_ceil_div(M, BM), mnb_ceil_div(g.Ng, bn), g.G);
  MNB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "grid too large");
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_FWD(ACC)                                                         \
  do {                                                                          \
    if (bn == 16) conv_fwd_kernel<ACC, 16><<<grid, NT, 0, st>>>(a);             \
    else if (bn == 32) conv_fwd_kernel<ACC, 32><<<grid, NT, 0, st>>>(a);        \
    else conv_fwd_kernel<ACC, 64><<<grid, NT, 0, st>>>(a);                      \
  } while (0)
  if (int_path) LAUNCH_FWD(int); else LAUNCH_FWD(float);
#undef LAUNCH_FWD
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_conv2d_dgrad(const mnb_conv_shape* s, const float* dy, const float* wq,
                                const uint32_t* pass_bits, const mnb_act_qparams* qp, float* dx,
                                mnb_stream_t stream) {
  DgradArgs a;
  if (int e = make_geom(s, a.g)) return e;
  MNB_REQUIRE(dy && wq && dx, "NULL dgrad pointers");
  MNB_REQUIRE((pass_bits == nullptr) == (qp == nullptr), "pass_bits and qp go together");
  a.dy = dy; a.wq = wq; a.pass_bits = pass_bits; a.has_qp = qp != nullptr; a.dx = dx;
  if (qp) a.qp = *qp; else a.qp = mnb_act_qparams{};
  const ConvGeom& g = a.g;
  const int M = g.B * g.H * g.W;
  const int bn = pick_bn(g.Cg);
  dim3 grid(mnb_ceil_div(M, BM), mnb_ceil_div(g.Cg, bn), g.G);
  MNB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  if (bn == 16) conv_dgrad_kernel<16><<<grid, NT, 0, st>>>(a);
  else if (bn == 32) conv_dgrad_kernel<32><<<grid, NT, 0, st>>>(a);
  else conv_dgrad_kernel<64><<<grid, NT, 0, st>>>(a);
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int64_t mnb_wgrad_scratch_bytes(const mnb_conv_shape* s) {
  ConvGeom g;
  if (make_geom(s, g)) return -1;
  int bn, splits, kps;
  wgrad_plan(g, bn, splits, kps);
  return (int64_t)splits * g.K * g.Cg * g.RS * 4;
}

extern "C" int mnb_conv2d_wgrad(const mnb_conv_shape* s, const float* dy, const mnb_conv_operands* op,
                                float* dwq, void* scratch, mnb_stream_t stream) {
  WgradArgs a;
  if (int e = make_geom(s, a.g)) return e;
  MNB_REQUIRE(dy && op && dwq && scratch, "NULL wgrad pointers");
  MNB_REQUIRE((op->a_codes != nullptr) != (op->a_f32 != nullptr), "exactly one of a_codes / a_f32 must be given");
  a.dy = dy; a.a_codes = op->a_codes; a.a_f32 = op->a_f32; a.a_off = op->a_offset; a.a_off_zp = op->a_offset_zp;
  a.partial = reinterpret_cast<float*>(scratch);
  const ConvGeom& g = a.g;
  int bn;
  wgrad_plan(g, bn, a.splits, a.k_per_split);
  const int Nd = g.Cg * g.RS;
  dim3 grid(mnb_ceil_div(g.Ng, BM), mnb_ceil_div(Nd, bn), g.G * a.splits);
  MNB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  if (bn == 16) conv_wgrad_kernel<16><<<grid, NT, 0, st>>>(a);
  else if (bn == 32) conv_wgrad_kernel<32><<<grid, NT, 0, st>>>(a);
  else conv_wgrad_kernel<64><<<grid, NT, 0, st>>>(a);
  const int64_t n = (int64_t)g.K * Nd;
  int blocks = (int)std::min<int64_t>(mnb_ceil_div(n, 256), MNB_NUM_SMS * 8);
  wgrad_reduce_kernel<<<blocks, 256, 0, st>>>(a.partial, n, a.splits, op->a_codes ? op->a_scale : nullptr, dwq);
  MNB_LAUNCHED(2);
  return 0;
}
