// Packed-operand ("pk") tensor-core convolution family: any conv geometry of the QAT models on tcgen05.
//
// ResNet-18 (up to 512 -> 512 3x3 = 9.4 MB of weights, stride 2, 4x4 images), NIN's 5x5 96 -> 192 and 224x224
// inputs need the B operand STREAMED and N / W tiling, so no weight slab stays resident in shared memory and no
// kernel converts fp32 activations itself.  Every operand reaches the kernel already in the layout the tensor core
// reads:
//
//   activations / gradients : bf16 "term planes"  pk[t][b][c/8][h][w][8]   (16 bytes = 8 channels of one pixel)
//                             t = 0 .. T-1 exact pieces of an fp32 value (x = p0 + p1 + p2, 8 significand bits each)
//                             or ONE plane of exact integer levels (fake-quantized activations);
//   weights                 : bf16 image [n-tile][group][stage][term][tap][c/8][n][8] (K-major, rows = n), written
//                             once per optimizer step by pk_pack_weight_kernel;
//
// so the convolution itself is the canonical Blackwell pipeline TMA -> tcgen05.mma -> TMEM -> epilogue with no
// converter warps.  A 5-D tensor map (8, W, H, B, C/8) with the channel-octet dimension declared LAST makes one
// box land in shared memory as op[c/8][position][8]: the UMMA K-major no-swizzle canonical layout with the
// positions of the zero-padded tile as GEMM rows (halo rows AND columns zero-filled by the TMA unit), so filter tap
// (r, s) is the same buffer with the descriptor start address moved by (r*BW + s)*16 bytes: implicit GEMM without
// im2col.  The same buffers read as MN-major operands give the weight gradient (positions = reduction dimension).
//
// Stride-2 convolutions use the space-to-depth form: the pack kernel writes the four (h%2, w%2) phase planes as extra
// channel octets, every filter tap then is a stride-1 tap of ONE phase plane with a shift in {-1, 0} (data gradient:
// four output phases, each a stride-1 conv of dy with a subset of the taps).
//
// Exactness: integer levels (|e| <= 256) are exact in bf16, products exact, fp32 accumulation in TMEM.  fp32 operands
// are split into T exact bf16 pieces; the products p_i * q_j with i + j < max(Ta, Tb) are accumulated, smallest first.
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "mnb_common.cuh"
#include "mnb_tc.cuh"

namespace pk {

constexpr int NTHREADS = 256;      // warp 0 TMA, warp 1 MMA issue, warp 2 TMEM alloc, warps 4..7 epilogue
constexpr int MAXST = 8;           // operand ring (power of two: ring index = counter & mask)
constexpr int MAXTAP = 64, MAXTMPL = 16, MAXY = 4, MAXPAIR = 6, MAXPROG = 512;
constexpr int kSmemBudget = 227 * 1024 - 3072;   // dynamic shared memory the kernels may ask for

// ---------------------------------------------------------------------------------------------------------
// plan: everything about a (shape, mode) pair that the weight packer and the convolution must agree on
// ---------------------------------------------------------------------------------------------------------
struct Tmpl { int kph, tap0, ntap, blk_off, blk_bytes; };   // one (k-phase, tap group): a pipeline stage template

struct Plan {
  int mode;                 // 0 forward, 1 data gradient
  int B, G, R, S, stride;
  int HA, WA, C8A, nkph;    // A planes as stored: spatial dims, octets per k-phase (all groups), k-phases
  int kg, ng, NOUT;         // GEMM-K / GEMM-N channels per group, total output channels
  int OHr, OWr, OH, OW, omul, ny;   // raster (per output phase) and real output dims
  int hlo, hhi, wlo, whi;
  int Wt, BW, TH, THH, TB, npos, col_tiles, row_tiles, img_tiles, n_mtiles;
  int Nt, n_ntiles, MT, n_mgroups, n_items;
  int CC, ksteps, chunks;   // K-chunk channels (multiple of 16), MMAs along K per chunk, chunks per k-phase
  int TA, TBk, npairs, pair_a[MAXPAIR], pair_b[MAXPAIR];
  int ntmpl[MAXY], ntap[MAXY];
  Tmpl tmpl[MAXY][MAXTMPL];
  int tap_aoff[MAXY][MAXTAP];            // A start-row offset of a tap inside the box (16-byte units)
  short tap_r[MAXY][MAXTAP], tap_s[MAXY][MAXTAP];
  int img_bytes[MAXY], y_off[MAXY];      // bytes of one (n-tile, group) weight image of output phase y; prefix offsets
  int64_t wimg_bytes;
  int a_box_bytes, a_bytes, b_off, stage_bytes, nstage, st_log2, smem_bytes, tmem_cols;
  int segmented, seg_len;   // stages per accumulation segment (segmented mode)
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

static void make_pairs(int TA, int TBk, Plan& p) {
  // pieces have magnitudes 2^-8i: accumulate the products p_i q_j with i + j <= max(TA, TBk) - 1, smallest first
  const int lim = std::max(TA, TBk) - 1;
  p.npairs = 0;
  for (int sum = lim; sum >= 0; --sum)
    for (int a = 0; a < TA; ++a) {
      const int b = sum - a;
      if (b < 0 || b >= TBk) continue;
      if (p.npairs < MAXPAIR) { p.pair_a[p.npairs] = a; p.pair_b[p.npairs] = b; ++p.npairs; }
    }
}

static int unsupported(const char* why) { return mnb_fail(MNB_E_UNSUPPORTED, "pk conv: %s", why); }

// mode 0: y = conv2d(x, w); mode 1: dx = conv_transpose(dy, w).  TA / TBk: term planes of the streamed / weight operand.
static int make_plan(const mnb_conv_shape* s, int mode, int TA, int TBk, Plan& p) {
  MNB_REQUIRE(s != nullptr, "conv shape is NULL");
  memset(&p, 0, sizeof(p));
  const int C = s->in_c, K = s->out_c, G = s->groups, H = s->in_h, W = s->in_w, R = s->ker_h, S = s->ker_w;
  MNB_REQUIRE(s->batch > 0 && C > 0 && K > 0 && H > 0 && W > 0 && G > 0 && C % G == 0 && K % G == 0 && R > 0 && S > 0,
              "bad conv shape");
  MNB_REQUIRE(TA >= 1 && TA <= 3 && TBk >= 1 && TBk <= 3, "term counts must be 1..3");
  if (s->dil_h != 1 || s->dil_w != 1) return unsupported("dilation != 1");
  if (s->stride_h != s->stride_w || (s->stride_h != 1 && s->stride_h != 2)) return unsupported("stride must be 1 or 2");
  const int st = s->stride_h, ph_ = s->pad_h, pw_ = s->pad_w;
  if (ph_ > R - 1 || pw_ > S - 1) return unsupported("padding larger than the filter");
  const int P = (H + 2 * ph_ - R) / st + 1, Q = (W + 2 * pw_ - S) / st + 1;
  if (P < 1 || Q < 1) return unsupported("empty output");
  if (st == 2 && ((H | W) & 1)) return unsupported("stride 2 needs even H and W");
  const int cin_g = C / G, cout_g = K / G;
  p.mode = mode; p.B = s->batch; p.G = G; p.R = R; p.S = S; p.stride = st;
  p.TA = TA; p.TBk = TBk;
  make_pairs(TA, TBk, p);
  if (mode == 0) {
    p.kg = cin_g; p.ng = cout_g; p.NOUT = K;
    p.nkph = st == 2 ? 4 : 1;
    p.HA = H / st; p.WA = W / st; p.C8A = ceil_div(C, 8);
    p.OHr = P; p.OWr = Q; p.OH = P; p.OW = Q; p.omul = 1; p.ny = 1;
  } else {
    p.kg = cout_g; p.ng = cin_g; p.NOUT = C;
    p.nkph = 1; p.HA = P; p.WA = Q; p.C8A = ceil_div(K, 8);
    p.OHr = H / st; p.OWr = W / st; p.OH = H; p.OW = W; p.omul = st; p.ny = st == 2 ? 4 : 1;
  }
  if (G > 1 && (p.kg % 8)) return unsupported("grouped conv needs GEMM-K channels per group % 8 == 0");
  // ---- taps: (k-phase, shift) of every filter tap, per output phase
  struct Tap { int kph, sh, sw, r, s; };
  Tap taps[MAXY][MAXTAP];
  int hlo = 0, hhi = 0, wlo = 0, whi = 0;
  for (int y = 0; y < p.ny; ++y) {
    int n = 0;
    const int ya = y >> 1, yb = y & 1;
    for (int kph = 0; kph < p.nkph; ++kph)       // taps sorted by k-phase
      for (int r = 0; r < R; ++r)
        for (int q = 0; q < S; ++q) {
          int kp = 0, sh, sw;
          if (mode == 0) {
            const int dr = r - ph_, ds = q - pw_;
            if (st == 1) { sh = dr; sw = ds; }
            else {
              const int fh = dr & 1, fw = ds & 1;
              kp = fh * 2 + fw; sh = (dr - fh) / 2; sw = (ds - fw) / 2;
            }
          } else {
            if (st == 1) { sh = ph_ - r; sw = pw_ - q; }
            else {
              const int th = ya + ph_ - r, tw = yb + pw_ - q;
              if ((th & 1) || (tw & 1)) continue;
              sh = th / 2; sw = tw / 2;   // exact (even), also for negatives
            }
          }
          if (kp != kph) continue;
          if (n >= MAXTAP) return unsupported("more than 64 filter taps");
          taps[y][n++] = Tap{kph, sh, sw, r, q};
          hlo = std::max(hlo, -sh); hhi = std::max(hhi, sh); wlo = std::max(wlo, -sw); whi = std::max(whi, sw);
        }
    p.ntap[y] = n;
  }
  p.hlo = hlo; p.hhi = hhi; p.wlo = wlo; p.whi = whi;
  // ---- M tile: 128 consecutive positions of the zero-padded tile raster (tb, row, col)
  const int halo_w = wlo + whi;
  if (halo_w >= 96) return unsupported("filter too wide");
  // Column tiling: a tile is TH rows of Wt columns, rastered with the row pitch BW = Wt + halo, and its last valid position
  // must be < 128.  Narrower tiles often hold MORE valid positions (224 wide: 1 x 112 = 112 vs 4 x 28 = 112 with a third
  // of the halo rows; 32 wide: 3 x 32 = 96 vs 7 x 16 = 112) - every tile costs the same MMAs, and the halo rows are re-read
  // (THH * BW) / (TH * Wt) times.  cost = tiles per image * (1 + 0.25 * read amplification) * (1 + 3.2 / Wt)
  {
    const int ct_min = ceil_div(p.OWr, 128 - halo_w);
    double best = 1e30;
    // (measured, r2w / r2x: the single-product kernels gain from narrower tiles - 64 -> 64 3x3 @32: 62 -> 53 us - while the
    // segmented split-fp32 kernels lose 10 - 15 % unless the widest tiling re-reads its halo rows more than ~2.2 x, as on
    // 112- and 224-wide planes)
    int ct_max = std::min(p.OWr, ct_min + 14);
    if (p.npairs > 1) {
      const int wt0 = ceil_div(p.OWr, ct_min), bw0 = wt0 + halo_w;
      const int th0 = std::max(1, std::min(p.OHr, (128 - wt0) / bw0 + 1));
      if ((double)((th0 + hlo + hhi) * bw0) / (double)(th0 * wt0) <= 2.2) ct_max = ct_min;
    }
    for (int ct = ct_min; ct <= ct_max; ++ct) {
      const int wt = ceil_div(p.OWr, ct), bw = wt + halo_w;
      if (ceil_div(p.OWr, wt) != ct) continue;                       // same tiling as a smaller ct
      const int th = std::max(1, std::min(p.OHr, (128 - wt) / bw + 1));
      const double amp = (double)((th + hlo + hhi) * bw) / (double)(th * wt);
      // (+ a mild preference for long rows: the epilogue's fp32 stores cover Wt * 4 contiguous bytes per channel and row)
      const double cost = (double)ct * ceil_div(p.OHr, th) * (1.0 + 0.25 * amp) * (1.0 + 3.2 / wt);
      if (cost < best - 1e-9) { best = cost; p.col_tiles = ct; p.Wt = wt; p.BW = bw; p.TH = th; }
    }
    if (const char* e = getenv("MNB_PK_COLTILES")) {                 // experiments: force the number of column tiles
      const int ct = atoi(e);
      if (ct >= ct_min && ct <= p.OWr) {
        p.col_tiles = ct; p.Wt = ceil_div(p.OWr, ct); p.col_tiles = ceil_div(p.OWr, p.Wt); p.BW = p.Wt + halo_w;
        p.TH = std::max(1, std::min(p.OHr, (128 - p.Wt) / p.BW + 1));
      }
    }
  }
  p.THH = p.TH + hlo + hhi;
  p.TB = 1;
  if (p.TH == p.OHr && p.col_tiles == 1) {
    const int last = (p.TH - 1) * p.BW + p.Wt;             // rows used by the last image of a tile
    p.TB = std::max(1, std::min(p.B, (128 - last) / (p.THH * p.BW) + 1));
  }
  if (p.BW > 128 || p.THH > 256 || p.TB > 256) return unsupported("box dimension");
  p.npos = p.TB * p.THH * p.BW;
  p.row_tiles = ceil_div(p.OHr, p.TH);
  p.img_tiles = ceil_div(p.B, p.TB);
  p.n_mtiles = p.img_tiles * p.row_tiles * p.col_tiles;
  // ---- N tile
  const int ng16 = round_up(p.ng, 16);
  // Split fp32 operands (more than one piece product per K-step) run in SEGMENTED mode: tcgen05.mma truncates the running
  // fp32 accumulator after every instruction (a bias of ~2e-8 of |D| per MMA, measured: 3e-5 after 1700 chained MMAs),
  // so the K loop is cut into segments of <= ~64 MMAs, each into a fresh TMEM accumulator, and the epilogue warps add
  // the segments in registers with round-to-nearest adds.  That needs the whole N tile in registers: Nt <= 128, MT = 1.
  // A K loop that is short anyway needs no segments: the whole chain of one accumulator (taps x piece pairs x K-steps) is
  // then no longer than a segment would be, and the kernel keeps the rolled epilogue, MT > 1 and N tiles up to 256 (the
  // data gradients of NIN-GC's grouped layers: 16 / 36 MMAs per accumulator; r2z: the segmented form of the 256-channel 1x1
  // data gradient took 226 us against 95 us for the forward of the same tile shape).
  {
    int seg_target = 64;
    if (const char* e = getenv("MNB_PK_SEG_MMAS")) seg_target = std::max(1, atoi(e));
    int chain = 0;
    for (int y = 0; y < p.ny; ++y) chain = std::max(chain, p.ntap[y] * p.npairs * ceil_div(p.kg, 16));
    p.segmented = p.npairs > 1 && chain > seg_target;
  }
  if (ng16 <= 128) p.Nt = ng16;
  else if (ng16 % 128 == 0) p.Nt = 128;
  else if (ng16 <= 256 && !p.segmented) p.Nt = ng16;
  else if (ng16 <= 256) p.Nt = round_up(ceil_div(p.ng, 2), 16);
  else p.Nt = 128;
  p.n_ntiles = ceil_div(p.ng, p.Nt);
  // M tiles per work item: every item streams the WHOLE weight block of its (N tile, group) from L2 - measured floor of the
  // 64 -> 64 3x3 layer with the MMAs switched off (MNB_PK_DEBUG=2): 190 us for the split-fp32 forward at MT = 1, i.e. L2 ->
  // shared-memory bandwidth on the re-fetched weights.  MT M tiles share one weight fetch (TMEM: 2 x MT x Nt <= 512 columns;
  // segmented mode keeps MT x Nt <= 128 running sums per thread in registers).  The items are dealt to 148 persistent
  // CTAs, so a larger MT is taken only while it costs no wave efficiency.
  p.MT = 1;
  {
    auto wave_eff = [&](int mt) {
      const int64_t items = (int64_t)ceil_div(p.n_mtiles, mt) * p.n_ntiles * G;
      const int64_t ctas = std::max<int64_t>(1, MNB_NUM_SMS / p.ny);
      return (double)items / (double)(ceil_div((int)std::min<int64_t>(items, 1 << 30), (int)ctas) * ctas);
    };
    const int cap = p.segmented ? std::max(1, 128 / p.Nt) : std::max(1, 256 / p.Nt);
    for (int mt = 2; mt <= std::min(4, cap); mt *= 2) {
      if (p.n_mtiles < mt) break;
      if ((int64_t)ceil_div(p.n_mtiles, mt) * p.n_ntiles * G * p.ny < 120) break;
      if (wave_eff(mt) >= wave_eff(1) - 0.04) p.MT = mt;
    }
  }
  if (const char* e = getenv("MNB_PK_MT")) {
    const int v = atoi(e);
    if ((v == 1 || v == 2 || v == 4) && v * p.Nt <= (p.segmented ? 128 : 256)) p.MT = v;
  }
  p.n_mgroups = ceil_div(p.n_mtiles, p.MT);
  p.n_items = p.n_mgroups * p.n_ntiles * G;
  // ---- K chunking and tap groups: one stage = MT * TA boxes of CC channels + the weights of (chunk, tap group)
  const int nk16 = ceil_div(p.kg, 16);
  int maxtap_kph = 1;
  for (int y = 0; y < p.ny; ++y)
    for (int i = 0, run = 0; i < p.ntap[y]; ++i) {
      run = (i > 0 && taps[y][i].kph == taps[y][i - 1].kph) ? run + 1 : 1;
      maxtap_kph = std::max(maxtap_kph, run);
    }
  const int a16 = p.MT * TA * round_up(2 * p.npos * 16, 128);     // A bytes per 16 channels (2 octets)
  auto b16 = [&](int tg) { return TBk * tg * 2 * p.Nt * 16; };   // B bytes per 16 channels
  const int stage_target = 56 * 1024;
  int TG = std::min(maxtap_kph, 25);
  while (TG > 1 && a16 + b16(TG) > stage_target) --TG;
  if (a16 + b16(TG) > (kSmemBudget - 8192) / 2) return unsupported("one 16-channel stage does not fit in shared memory");
  int cc16 = std::max(1, std::min(nk16, stage_target / (a16 + b16(TG))));
  cc16 = std::min(cc16, 16);
  p.chunks = ceil_div(nk16, cc16);
  cc16 = ceil_div(nk16, p.chunks);            // balance the chunks
  p.CC = cc16 * 16; p.ksteps = cc16;
  p.a_box_bytes = (p.CC / 8) * p.npos * 16;
  p.a_bytes = round_up(p.a_box_bytes, 128);
  p.b_off = p.MT * TA * p.a_bytes;
  // ---- stage templates and the weight-image layout
  int64_t total = 0;
  int max_blk = 0;
  for (int y = 0; y < p.ny; ++y) {
    int nt = 0, off = 0;
    for (int i = 0; i < p.ntap[y];) {
      int j = i;
      while (j < p.ntap[y] && taps[y][j].kph == taps[y][i].kph && j - i < TG) ++j;
      if (nt >= MAXTMPL) return unsupported("too many tap groups");
      Tmpl& t = p.tmpl[y][nt++];
      t.kph = taps[y][i].kph; t.tap0 = i; t.ntap = j - i;
      t.blk_bytes = TBk * t.ntap * (p.CC / 8) * p.Nt * 16;
      t.blk_off = off;
      off += p.chunks * t.blk_bytes;
      max_blk = std::max(max_blk, t.blk_bytes);
      i = j;
    }
    p.ntmpl[y] = nt;
    p.img_bytes[y] = off;
    p.y_off[y] = (int)total;
    total += (int64_t)off * p.n_ntiles * G;
    if (total > (int64_t)1 << 30) return unsupported("weight image larger than 1 GiB");
    for (int i = 0; i < p.ntap[y]; ++i) {
      p.tap_aoff[y][i] = (taps[y][i].sh + hlo) * p.BW + (taps[y][i].sw + wlo);
      p.tap_r[y][i] = (short)taps[y][i].r; p.tap_s[y][i] = (short)taps[y][i].s;
    }
  }
  p.wimg_bytes = std::max<int64_t>(total, 16);
  p.seg_len = 1 << 30;
  if (p.segmented) {
    const int per_stage = TG * p.npairs * p.ksteps;     // MMAs per accumulator and stage (upper bound)
    int target = 64;
    if (const char* e = getenv("MNB_PK_SEG_MMAS")) target = std::max(1, atoi(e));
    p.seg_len = std::max(1, target / per_stage);
  }
  p.stage_bytes = round_up(p.b_off + max_blk, 1024);
  // slack behind the last stage: MMAs of invalid halo rows read up to 128 + max tap offset rows past a plane start
  const int slack = round_up((128 + (hlo + hhi) * p.BW + halo_w + 8) * 16, 1024);
  int nst = (kSmemBudget - slack) / p.stage_bytes;
  if (nst < 2) return unsupported("fewer than two pipeline stages fit");
  p.nstage = nst >= 8 ? 8 : (nst >= 4 ? 4 : 2);
  if (const char* e = getenv("MNB_PK_STAGES")) { const int v = atoi(e); if ((v == 2 || v == 4 || v == 8) && v <= nst) p.nstage = v; }
  p.st_log2 = p.nstage == 8 ? 3 : (p.nstage == 4 ? 2 : 1);
  p.smem_bytes = p.nstage * p.stage_bytes + slack;
  int cols = 32;
  while (cols < 2 * p.MT * p.Nt) cols <<= 1;
  if (cols > 512) return unsupported("accumulators exceed tensor memory");
  p.tmem_cols = cols;
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// operand packers
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// fp32 NCHW -> bf16 term planes [t][b][octet][h][w][8]; one thread = one pixel of one channel octet.
//   QUANT = 0: planes are the exact pieces of x (* ch_scale[c] when given)
//   QUANT = 1: plane 0.. hold the fake-quantized integer level e = code + a_off (+ zero point) (exact; two pieces when
//              |e| can exceed 256), bits8[b][c/8][h][w] bit j = STE pass flag of channel 8*(c/8) + j
// phase_split: octet index (h%2 * 2 + w%2) * C8 + c/8 of a [.., H/2, W/2] plane (stride-2 consumers)
template <int QUANT>
__global__ void __launch_bounds__(256) pack_act_kernel(const float* __restrict__ x, int B, int C, int H, int W, int C8,
                                                       int terms, const float* __restrict__ ch_scale, mnb_act_qparams qp,
                                                       int a_off, int phase_split, uint4* __restrict__ out,
                                                       int64_t plane_vecs, uint8_t* __restrict__ bits8, int relu) {
  MnbActQ q;
  float zp = 0.f;
  if (QUANT) {
    q = mnb_load_actq(qp);
    if (qp.mode == MNB_ACT_IAO && qp.zero_point) zp = __ldg(qp.zero_point);
  }
  // grid = (chunks of the H*W plane, B * C8 planes): 32-bit index arithmetic only (the first version decoded a flat
  // 64-bit index with five divisions per pixel and ran at 0.9 TB/s)
  const uint32_t HW = (uint32_t)H * (uint32_t)W;
  // block = (positions, planes): small images put several planes into one 256-thread block
  const uint32_t plane = blockIdx.y * blockDim.y + threadIdx.y;                 // b * C8 + c8
  if (plane >= (uint32_t)B * (uint32_t)C8) return;
  const uint32_t b = plane / (uint32_t)C8, c8 = plane - b * (uint32_t)C8;
  for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < HW; pos += gridDim.x * blockDim.x) {
    const int64_t idx = (int64_t)plane * HW + pos;
    float v[8];
    uint32_t passbits = 0;
    const float* src = x + ((int64_t)b * C + c8 * 8) * HW + pos;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = (int)c8 * 8 + j;
      float val = c < C ? __ldg(src + (int64_t)j * HW) : 0.f;
      if (relu) val = fmaxf(val, 0.f);          // a preceding nn.ReLU folded into the packer (inference graphs)
      if (!QUANT && ch_scale) val = c < C ? __fmul_rn(val, __ldg(ch_scale + c)) : 0.f;
      v[j] = val;
    }
    if (QUANT) {   // level itself (code + a_off) as a float, eight channels in straight-line code
      float lev[8];
      mnb_act_levels<8>(q, v, lev, passbits);
      uint32_t live = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool in = (int)c8 * 8 + j < C;
        v[j] = in ? lev[j] + zp : 0.f;
        live |= in ? (1u << j) : 0u;
      }
      passbits &= live;
    }
    int64_t dst;
    if (phase_split) {
      const uint32_t h = pos / (uint32_t)W, w = pos - h * (uint32_t)W;
      const uint32_t oct = ((h & 1u) * 2u + (w & 1u)) * (uint32_t)C8 + c8;
      dst = (((int64_t)b * 4 * C8 + oct) * (H >> 1) + (h >> 1)) * (W >> 1) + (w >> 1);
    } else {
      dst = idx;
    }
    for (int tm = 0; tm < terms; ++tm) {
      uint32_t pk4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        pk4[j] = pack2(v[2 * j], v[2 * j + 1]);
        v[2 * j] -= __uint_as_float(pk4[j] << 16);
        v[2 * j + 1] -= __uint_as_float(pk4[j] & 0xffff0000u);
      }
      out[(int64_t)tm * plane_vecs + dst] = make_uint4(pk4[0], pk4[1], pk4[2], pk4[3]);
    }
    if (QUANT && bits8) bits8[idx] = (uint8_t)passbits;
  }
}

// BatchNorm2d + ReLU + DoReFa activation quantizer + operand packing in ONE pass (SURVEY.md 8 f2 for the DoReFa blocks
// conv -> nn.BatchNorm2d -> nn.ReLU -> [channel_shuffle] -> QuantConv2d, nin_gc.py:53-59 + DF:36-46): reads the conv output
// once, writes the integer levels of the NEXT conv's activation quantizer as its packed bf16 plane (2 B / element, in the
// output channel order of the folded shuffle) and the combined STE mask  relu'(bn) * [0.1 bn <= 1]  as flat NCHW bits in the
// producer's own channel order - exactly what mnb_bn_sign_bwd consumes, so the backward needs no new kernel.  The fp32
// BatchNorm / ReLU outputs and the separate quantize + pack pass never touch HBM.
// one warp = 32 consecutive positions of one OUTPUT channel octet of one image
__global__ void __launch_bounds__(256) bn_relu_quant_pack_kernel(const float* __restrict__ x, int batch, int channels, int hw,
                                                                 int sg, const float* __restrict__ mean,
                                                                 const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                                 const float* __restrict__ beta, mnb_act_qparams qp,
                                                                 uint32_t* __restrict__ bits, uint4* __restrict__ xp) {
  const int lane = threadIdx.x & 31;
  const int c8n = channels / 8, p32n = hw / 32, cpg = channels / sg;
  const int64_t items = (int64_t)batch * c8n * p32n;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const MnbActQ q = mnb_load_actq(qp);
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < items; w += nwarps) {
    const int p32 = (int)(w % p32n);
    const int64_t t = w / p32n;
    const int oc8 = (int)(t % c8n), b = (int)(t / c8n);
    const int pos = p32 * 32 + lane;
    float lev[8], yv[8], bnv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int oc = oc8 * 8 + j;
      const int c = sg > 1 ? (oc % sg) * cpg + oc / sg : oc;   // inverse of out[:, a*sg + b] = in[:, b*cpg + a]
      const int64_t fi = ((int64_t)b * channels + c) * hw + pos;
      bnv[j] = fmaf(__ldg(x + fi) - __ldg(mean + c), __ldg(gamma + c) * __ldg(invstd + c), __ldg(beta + c));
      yv[j] = fmaxf(bnv[j], 0.f);                              // nn.ReLU
    }
    uint32_t passbits;
    mnb_act_levels<8>(q, yv, lev, passbits);                   // DoReFa: pass = 0 <= 0.1 y <= 1
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int oc = oc8 * 8 + j;
      const int c = sg > 1 ? (oc % sg) * cpg + oc / sg : oc;
      const int64_t fi = ((int64_t)b * channels + c) * hw + pos;
      const uint32_t word = __ballot_sync(0xffffffffu, ((passbits >> j) & 1u) && bnv[j] > 0.f);   // relu'(0) = 0
      if (lane == 0) bits[fi >> 5] = word;
    }
    xp[((int64_t)b * c8n + oc8) * hw + pos] = make_uint4(pack2(lev[0], lev[1]), pack2(lev[2], lev[3]), pack2(lev[4], lev[5]),
                                                          pack2(lev[6], lev[7]));
  }
}

// IAO QuantAdd of a frozen inference graph + the consuming conv's quantizer and operand packing in one pass (see
// mnb_quant_add_pack_fwd): one thread = one pixel of one channel octet, same arithmetic as quant_add_fwd_kernel
// (mnb_quant.cu) followed by pack_act_kernel<1>.
__global__ void __launch_bounds__(256) quant_add_pack_kernel(const float* __restrict__ a, const float* __restrict__ b, int B, int C,
                                                             int H, int W, int C8, mnb_act_qparams qadd, int relu,
                                                             float* __restrict__ out, mnb_act_qparams qnext, int next_relu,
                                                             int phase_split, uint4* __restrict__ out_pk) {
  const MnbActQ q = mnb_load_actq(qadd), qn = mnb_load_actq(qnext);
  const float zpn = (qnext.mode == MNB_ACT_IAO && qnext.zero_point) ? __ldg(qnext.zero_point) : 0.f;
  const uint32_t HW = (uint32_t)H * (uint32_t)W;
  const uint32_t plane = blockIdx.y * blockDim.y + threadIdx.y;                 // b * C8 + c8
  if (plane >= (uint32_t)B * (uint32_t)C8) return;
  const uint32_t bi = plane / (uint32_t)C8, c8 = plane - bi * (uint32_t)C8;
  for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < HW; pos += gridDim.x * blockDim.x) {
    const int64_t base = ((int64_t)bi * C + c8 * 8) * HW + pos;
    float va[8], vb[8], lev[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool live = (int)c8 * 8 + j < C;
      va[j] = live ? __ldg(a + base + (int64_t)j * HW) : 0.f;
      vb[j] = live ? __ldg(b + base + (int64_t)j * HW) : 0.f;
    }
    // Q(a), Q(b): the level as a float (IAO: clamp(round(x/s - zp)), value = (level + zp) * s; DoReFa: value = level * s)
    float la[8], lb[8], sum[8];
    uint32_t pbits;
    mnb_act_levels<8>(q, va, la, pbits);
    mnb_act_levels<8>(q, vb, lb, pbits);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool live = (int)c8 * 8 + j < C;
      float oa, ob;
      if (q.mode == MNB_ACT_DOREFA) { oa = __fmul_rn(la[j], q.s); ob = __fmul_rn(lb[j], q.s); }
      else { oa = __fmul_rn(__fadd_rn(la[j], q.zp), q.s); ob = __fmul_rn(__fadd_rn(lb[j], q.zp), q.s); }
      float t = __fadd_rn(oa, ob);
      if (relu) t = fmaxf(t, 0.f);
      if (live) out[base + (int64_t)j * HW] = t;
      sum[j] = next_relu ? fmaxf(t, 0.f) : t;
    }
    mnb_act_levels<8>(qn, sum, lev, pbits);
#pragma unroll
    for (int j = 0; j < 8; ++j) lev[j] = ((int)c8 * 8 + j < C) ? lev[j] + zpn : 0.f;
    int64_t dst;
    if (phase_split) {
      const uint32_t h = pos / (uint32_t)W, w = pos - h * (uint32_t)W;
      const uint32_t oct = ((h & 1u) * 2u + (w & 1u)) * (uint32_t)C8 + c8;
      dst = (((int64_t)bi * 4 * C8 + oct) * (H >> 1) + (h >> 1)) * (W >> 1) + (w >> 1);
    } else {
      dst = (int64_t)plane * HW + pos;
    }
    out_pk[dst] = make_uint4(pack2(lev[0], lev[1]), pack2(lev[2], lev[3]), pack2(lev[4], lev[5]), pack2(lev[6], lev[7]));
  }
}

template <int VEC> struct PkVec;
template <> struct PkVec<1> { typedef float type; };
template <> struct PkVec<2> { typedef float2 type; };
template <> struct PkVec<4> { typedef float4 type; };

// Second pass of the fused BatchNorm + binarizer backward (mnb_bn_sign_bwd: dgamma / dbeta already reduced) that writes the
// gradient of the PRODUCING convolution's output directly as that convolution's packed operand: `terms` exact bf16 pieces
// of  dx * ch_scale[c]  in the plane layout [t][b][c/8][h][w][8] (and, optionally, plain fp32 dx).  The conv's data- and
// weight-gradient kernels then start from TMA loads; the separate pack pass (read 4 B, write 4 B per element) is gone.
//   dx = gamma * invstd * (g * pass - dbeta / N - xhat * dgamma / N)            (training-mode BatchNorm, saturate STE)
// One warp = 32 * VEC consecutive pixels of one channel octet (the conv's own channel order; g is read in the shuffled
// order); a lane owns VEC consecutive pixels: 16-byte loads of g and x (VEC = 4), one word of pass bits per channel, VEC
// consecutive 16-byte pixels per piece plane.  (First version: one pixel per thread, 4-byte loads with the g load predicated
// on the bits load - 2.0 TB/s of its 12 B per element, 1.0 ms of the 6.6 ms headline step in the r2z launch list.)
template <int VEC>
__global__ void __launch_bounds__(256) bn_sign_bwd_pack_kernel(const float* __restrict__ g, const uint32_t* __restrict__ bits,
                                                               const float* __restrict__ x, int batch, int channels, int hw,
                                                               int sg, float inv_count, const float* __restrict__ mean,
                                                               const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                               const float* __restrict__ dgamma, const float* __restrict__ dbeta,
                                                               const float* __restrict__ ch_scale, int terms,
                                                               float* __restrict__ dx, uint4* __restrict__ out, int64_t plane_vecs) {
  typedef typename PkVec<VEC>::type T;
  const int lane = threadIdx.x & 31;
  const int c8n = channels / 8, cpg = channels / sg, chunks = hw / (32 * VEC);
  const int64_t items = (int64_t)batch * c8n * chunks;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < items; w += nwarps) {
    const int ch = (int)(w % chunks);
    const int64_t pl = w / chunks;                                // b * c8n + c8
    const int c8 = (int)(pl % c8n), b = (int)(pl / c8n);
    const int pos = (ch * 32 + lane) * VEC;
    T gv[8], xv[8];
    uint32_t bw[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = c8 * 8 + j;
      const int oc = sg > 1 ? (c % cpg) * sg + c / cpg : c;      // out[:, a*sg + b] = in[:, b*cpg + a]
      const int64_t fi = ((int64_t)b * channels + c) * hw + pos;
      gv[j] = __ldg(reinterpret_cast<const T*>(g + ((int64_t)b * channels + oc) * hw + pos));
      xv[j] = __ldg(reinterpret_cast<const T*>(x + fi));
      bw[j] = __ldg(bits + (fi >> 5)) >> (fi & 31);              // bit i = pass flag of pixel pos + i
    }
    float v[VEC][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = c8 * 8 + j;
      const float mu = __ldg(mean + c), is = __ldg(invstd + c), k = __ldg(gamma + c) * is;
      const float db = __ldg(dbeta + c) * inv_count, dg = __ldg(dgamma + c) * inv_count;
      const float sc = ch_scale ? __ldg(ch_scale + c) : 1.f;
      const float* gf = reinterpret_cast<const float*>(&gv[j]);
      const float* xf = reinterpret_cast<const float*>(&xv[j]);
      T dv;
      float* df = reinterpret_cast<float*>(&dv);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        float t = ((bw[j] >> i) & 1u) ? gf[i] : 0.f;
        t = t - db - ((xf[i] - mu) * is) * dg;
        t = k * t;
        df[i] = t;
        v[i][j] = ch_scale ? __fmul_rn(t, sc) : t;
      }
      if (dx) *reinterpret_cast<T*>(dx + ((int64_t)b * channels + c) * hw + pos) = dv;
    }
    const int64_t dst = pl * hw + pos;
    for (int tm = 0; tm < terms; ++tm) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        uint32_t pk4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          pk4[j] = pack2(v[i][2 * j], v[i][2 * j + 1]);
          v[i][2 * j] -= __uint_as_float(pk4[j] << 16);
          v[i][2 * j + 1] -= __uint_as_float(pk4[j] & 0xffff0000u);
        }
        out[(int64_t)tm * plane_vecs + dst + i] = make_uint4(pk4[0], pk4[1], pk4[2], pk4[3]);
      }
    }
  }
}

// The same for a producer with the 2x2 max-pool folded in (mnb_bn_sign_pool_*): second pass of its backward writing the
// full-resolution gradient of the producing conv's output as that conv's packed operand.  One lane = two horizontally
// adjacent pooling windows (4 x 2 pixels) of the 8 channels of one octet: per channel one float2 of the pooled gradient
// (read in the shuffled order), the two window arg-max bytes, the pass nibbles and two float4 of x; per piece plane two
// runs of 4 consecutive 16-byte pixels.  Layouts of arg / bits8 as written by bn_sign_pool_fwd_kernel (mnb_fused.cu).
__global__ void __launch_bounds__(256) bn_sign_pool_bwd_pack_kernel(const float2* __restrict__ g, const uchar2* __restrict__ arg,
                                                                    const uint8_t* __restrict__ bits8, const float4* __restrict__ x,
                                                                    int batch, int channels, int H, int W4, int sg, float inv_count,
                                                                    const float* __restrict__ mean, const float* __restrict__ invstd,
                                                                    const float* __restrict__ gamma, const float* __restrict__ dgamma,
                                                                    const float* __restrict__ dbeta, const float* __restrict__ ch_scale,
                                                                    int terms, uint4* __restrict__ out, int64_t plane_vecs) {
  const uint32_t OH = (uint32_t)H / 2u, OW2 = (uint32_t)W4, c8n = (uint32_t)channels / 8u, cpg = (uint32_t)channels / (uint32_t)sg;
  const uint32_t per_plane = OH * OW2;                                       // lane items per (image, channel) plane
  const int64_t total = (int64_t)batch * c8n * per_plane;
  for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t rem = (uint32_t)(it % per_plane);
    const int64_t pl = it / per_plane;                                      // b * c8n + c8
    const uint32_t c8 = (uint32_t)(pl % c8n), b = (uint32_t)(pl / c8n);
    const uint32_t oh = rem / OW2, j = rem - oh * OW2;
    float v[8][8];                                                            // [pixel e: row (e >> 2), column (e & 3)][channel]
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const uint32_t c = c8 * 8u + q;
      const uint32_t oc = sg > 1 ? (c % cpg) * (uint32_t)sg + c / cpg : c;
      const uint32_t plane = b * (uint32_t)channels + c;
      const float2 gv = __ldg(g + ((size_t)(b * (uint32_t)channels + oc) * OH + oh) * OW2 + j);
      const uchar2 a = arg[((size_t)plane * OH + oh) * OW2 + j];
      const uint32_t i0 = (plane * (uint32_t)H + 2u * oh) * (uint32_t)W4 + j, i1 = i0 + (uint32_t)W4;
      const uint32_t n0 = (bits8[i0 >> 1] >> (4u * (i0 & 1u))) & 15u, n1 = (bits8[i1 >> 1] >> (4u * (i1 & 1u))) & 15u;
      const float4 r0 = __ldg(x + i0), r1 = __ldg(x + i1);
      const float mu = __ldg(mean + c), is = __ldg(invstd + c), k = __ldg(gamma + c) * is;
      const float db = __ldg(dbeta + c) * inv_count, dg = __ldg(dgamma + c) * inv_count;
      const float sc = ch_scale ? __ldg(ch_scale + c) : 1.f;
      const uint32_t e0 = (a.x >> 1) * 4u + (a.x & 1u), e1 = (a.y >> 1) * 4u + 2u + (a.y & 1u);
      const uint32_t nib = n0 | (n1 << 4);
      const float xs[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float t = 0.f;
        if ((uint32_t)e == e0 && ((nib >> e) & 1u)) t = gv.x;
        if ((uint32_t)e == e1 && ((nib >> e) & 1u)) t = gv.y;
        t = t - db - ((xs[e] - mu) * is) * dg;
        t = k * t;
        v[e][q] = ch_scale ? __fmul_rn(t, sc) : t;
      }
    }
    const int64_t dst0 = (pl * H + 2 * oh) * (int64_t)(4 * W4) + 4 * j;     // pixel (2 oh, 4 j) of this octet plane
    for (int tm = 0; tm < terms; ++tm) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        uint32_t pk4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          pk4[q] = pack2(v[e][2 * q], v[e][2 * q + 1]);
          v[e][2 * q] -= __uint_as_float(pk4[q] << 16);
          v[e][2 * q + 1] -= __uint_as_float(pk4[q] & 0xffff0000u);
        }
        out[(int64_t)tm * plane_vecs + dst0 + (e >> 2) * (int64_t)(4 * W4) + (e & 3)] = make_uint4(pk4[0], pk4[1], pk4[2], pk4[3]);
      }
    }
  }
}

struct PackWParams {
  Plan pl;
  const int16_t* w_int; const float* w_f32; const float* kzero;   // kzero[k] == 0 -> the weights of channel k read as 0 (dgrad)
  int cin_g, cout_g;
};

// weights (int16 levels or fp32) -> bf16 image of the plan; one thread = one 16-byte vector (8 GEMM-K channels)
__global__ void __launch_bounds__(256) pack_weight_kernel(const __grid_constant__ PackWParams pp, uint4* __restrict__ out) {
  const Plan& p = pp.pl;
  const int64_t total = p.wimg_bytes / 16;
  const int RS = p.R * p.S;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += (int64_t)gridDim.x * blockDim.x) {
    int64_t byte = v * 16;
    int y = 0;
    for (int yy = 1; yy < p.ny; ++yy) if (byte >= p.y_off[yy]) y = yy;
    byte -= p.y_off[y];
    if (p.img_bytes[y] == 0) continue;
    const int ntg = (int)(byte / p.img_bytes[y]);
    int rem = (int)(byte - (int64_t)ntg * p.img_bytes[y]);
    if (ntg >= p.n_ntiles * p.G) continue;
    const int nt = ntg / p.G, g = ntg - nt * p.G;
    int t = 0;
    for (int tt = 1; tt < p.ntmpl[y]; ++tt) if (rem >= p.tmpl[y][tt].blk_off) t = tt;
    const Tmpl tp = p.tmpl[y][t];
    rem -= tp.blk_off;
    const int cc = rem / tp.blk_bytes;
    rem -= cc * tp.blk_bytes;
    const int per_tap = (p.CC / 8) * p.Nt * 16, per_term = tp.ntap * per_tap;
    const int term = rem / per_term;
    rem -= term * per_term;
    const int tapi = rem / per_tap;
    rem -= tapi * per_tap;
    const int c8l = rem / (p.Nt * 16), n = (rem - c8l * (p.Nt * 16)) / 16;
    const int r = p.tap_r[y][tp.tap0 + tapi], s = p.tap_s[y][tp.tap0 + tapi];
    const int nn = nt * p.Nt + n;                 // GEMM-N channel within the group
    float val[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int kk = cc * p.CC + c8l * 8 + e;     // GEMM-K channel within the group
      float x = 0.f;
      if (kk < p.kg && nn < p.ng) {
        int64_t src;
        int kout;
        if (p.mode == 0) { kout = g * pp.cout_g + nn; src = ((int64_t)kout * pp.cin_g + kk) * RS + r * p.S + s; }
        else { kout = g * pp.cout_g + kk; src = ((int64_t)kout * pp.cin_g + nn) * RS + r * p.S + s; }
        x = pp.w_int ? (float)__ldg(pp.w_int + src) : __ldg(pp.w_f32 + src);
        if (pp.kzero && __ldg(pp.kzero + kout) == 0.f) x = 0.f;
      }
      val[e] = x;
    }
    uint32_t pk4[4];
    for (int tm = 0; tm <= term; ++tm) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        pk4[j] = pack2(val[2 * j], val[2 * j + 1]);
        val[2 * j] -= __uint_as_float(pk4[j] << 16);
        val[2 * j + 1] -= __uint_as_float(pk4[j] & 0xffff0000u);
      }
    }
    out[v] = make_uint4(pk4[0], pk4[1], pk4[2], pk4[3]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// the convolution kernel (forward and data gradient)
// ---------------------------------------------------------------------------------------------------------
struct ConvParams {
  // private parameter block of the MMA-issue warp (uniform datapath: see mnb_conv_packed.cu for the rules)
  struct Mma {
    uint32_t n_items, chunks, ksteps, MT, Nt, npairs, st_mask, st_log2, stage16, a_mt16, a_term16, a_k16, b_off16,
        b_tap16, b_k16, idesc, a_lbo, b_lbo, seg_len;
    uint32_t ntmpl[MAXY];
    // The MMA "program": one 32-bit word per (filter tap, piece pair) of a stage template = A offset | B offset << 16
    // (16-byte units inside the stage); the issue loop is then  load word, two adds, MMA.  A single warp executes this
    // loop serially, so every instruction in it costs MMA issue rate (measured: 45 uniform-datapath instructions per
    // MMA = 420 cycles per MMA, tensor pipe 15 % busy).
    uint16_t tmpl_begin[MAXY][MAXTMPL], tmpl_cnt[MAXY][MAXTMPL];   // in groups of four words
    alignas(16) uint4 prog4[MAXPROG / 4];                          // padded with 0xffffffff to whole groups
  } m;
  // TMA role
  int n_items, n_ntiles, G, MT, TA, chunks, CC8, C8A, kg8, stage_bytes, a_bytes, a_box_bytes, b_off, st_mask, st_log2;
  int Wt, TH, TB, wlo, hlo, col_tiles, row_tiles, n_mtiles;
  int ntmpl[MAXY], tmpl_kph[MAXY][MAXTMPL], tmpl_blk_off[MAXY][MAXTMPL], tmpl_blk_bytes[MAXY][MAXTMPL];
  int img_bytes[MAXY], y_off[MAXY];
  const uint8_t* w_img;
  // epilogue
  int B, THH, BW, OHr, OWr, OH, OW, omul, ny, ng, Nt, NOUT, C8O, smem_bytes, tmem_cols, mode, zero_y[MAXY];
  int nseg[MAXY];           // accumulation segments per work item (1 unless segmented)
  int dbg;                  // MNB_PK_DEBUG (timing experiments only): 1 no epilogue stores, 2 no MMAs, 4 no TMEM loads
  const float* n_scale;     // [NOUT] per-output-channel scale or NULL
  const float* a_scale;     // device scalar multiplied into n_scale, or NULL
  float a_scale_const;
  const float* bias;        // [NOUT] or NULL
  const uint8_t* bits8;     // dgrad STE mask [B][C8O][OH][OW] or NULL
  float gain;               // dgrad: factor on passed gradients (DoReFa 0.1)
  float* out;               // fp32 NCHW result, or NULL when only the packed output below is wanted
  // fused consumer (inference graphs): the epilogue also applies [ReLU +] the NEXT conv's activation quantizer and writes
  // that conv's operand plane [b][c/8][h][w][8] bf16 (space-to-depth phase planes for a stride-2 consumer)
  uint4* post_out;
  mnb_act_qparams post_q;
  int post_relu, post_split;
  int* err;
};

struct alignas(16) ConvShared {
  uint64_t full[MAXST], empty[MAXST], acc_full[2], acc_empty[2];
  uint32_t tmem_slot, abort;
  alignas(16) float epi_scale[256];
  alignas(16) float epi_bias[256];
};

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

template <int NEPI>
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory"); }

// Epilogue warps: one warp can only read the 32 TMEM lanes of its own quarter (warp % 4), and a lone warp per scheduler
// issues its dependent tcgen05.ld -> fma -> st chains at ~0.3 instructions per cycle - ncu r3b: every forward / data-gradient
// launch of the family sat at 42 - 47 k instructions per epilogue warp in 160 - 173 k cycles, tensor pipe 7 - 9 % busy, DRAM
// 3.6 TB/s.  The un-segmented kernel therefore runs TWO warps per quarter (warps 4..7 take the even 16-column slots of an
// item, warps 8..11 the odd ones); the segmented kernel keeps one (its 128 running sums per thread need the registers).
// n = q * d + r for n < 2^22 through one float multiply (the compiler's 32-bit integer division is a ~25-instruction dependent
// chain; the TMA-issuing lane ran ~2100 instructions per work item, most of them these, at one instruction every four cycles -
// as long as a whole 3x3 g16 item takes: ncu r3b, source page).  q from the reciprocal is within +-1: corrected exactly.
struct FastDiv {
  uint32_t d; float inv;
  __device__ __forceinline__ explicit FastDiv(int dd) : d((uint32_t)dd), inv(1.0f / (float)dd) {}
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = __float2uint_rz(__uint2float_rz(n) * inv);
    r = n - q * d;
    if ((int32_t)r < 0) { --q; r += d; } else if (r >= d) { ++q; r -= d; }
  }
};

template <bool SEG> struct ConvCfg { static constexpr int EPIW = SEG ? 4 : 8, THREADS = 128 + 32 * EPIW; };

template <bool SEG>   // SEG: segmented accumulation (split fp32 operands), the epilogue keeps the N tile in registers
__global__ void __launch_bounds__(ConvCfg<SEG>::THREADS, 1)
pk_conv_kernel(const __grid_constant__ CUtensorMap tmap0, const __grid_constant__ CUtensorMap tmap1,
               const __grid_constant__ CUtensorMap tmap2, const __grid_constant__ ConvParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ ConvShared sh;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < MAXST; ++i) { tc::mbar_init(&sh.full[i], 1); tc::mbar_init(&sh.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&sh.acc_full[i], 1); tc::mbar_init(&sh.acc_empty[i], 32 * ConvCfg<SEG>::EPIW); }
    sh.abort = 0;
    tc::fence_barrier_init();
    tc::prefetch_tmap(&tmap0);
    if (p.TA > 1) tc::prefetch_tmap(&tmap1);
    if (p.TA > 2) tc::prefetch_tmap(&tmap2);
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&sh.tmem_slot)),
                 "r"((uint32_t)p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // rows behind a box that only invalid accumulator rows read must at least be finite
  for (int i = tid; i < p.smem_bytes / 16; i += ConvCfg<SEG>::THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sh.tmem_slot;

  if (warp == 0) {
    // ================================================================= TMA producer
    if (lane == 0) {
      const int y = blockIdx.y;
      uint32_t sc = 0;
      const FastDiv d_nt(p.n_ntiles), d_g(p.G), d_ct(p.col_tiles), d_rt(p.row_tiles);
      for (int it = blockIdx.x; it < p.n_items; it += gridDim.x) {
        uint32_t nt, r1, g, mg;
        d_nt.divmod((uint32_t)it, r1, nt);
        d_g.divmod(r1, mg, g);
        const uint8_t* wsrc = p.w_img + (size_t)p.y_off[y] + (size_t)(nt * p.G + g) * (size_t)p.img_bytes[y];
        for (int t = 0; t < p.ntmpl[y]; ++t) {
          const int kph = p.tmpl_kph[y][t];
          const uint32_t blk = (uint32_t)p.tmpl_blk_bytes[y][t];
          const uint8_t* bsrc = wsrc + p.tmpl_blk_off[y][t];
          for (int cc = 0; cc < p.chunks; ++cc, ++sc) {
            const uint32_t slot = sc & (uint32_t)p.st_mask, ph = (sc >> p.st_log2) & 1u;
            if (!tc::mbar_wait(&sh.empty[slot], ph ^ 1u, p.err, 701)) goto done;
            // MNB_PK_DEBUG bits 8 / 16 (timing experiments only): leave out the activation boxes / the weight block
            const bool ld_a = !(p.dbg & 8), ld_b = !(p.dbg & 16);
            tc::mbar_arrive_expect_tx(&sh.full[slot], (ld_a ? (uint32_t)(p.MT * p.TA * p.a_box_bytes) : 0u) + (ld_b ? blk : 0u));
            uint8_t* sbase = smem + (size_t)slot * p.stage_bytes;
            const int c8 = kph * p.C8A + g * p.kg8 + cc * p.CC8;
            for (int mt = 0; mt < (ld_a ? p.MT : 0); ++mt) {
              const uint32_t tile = mg * (uint32_t)p.MT + (uint32_t)mt;
              uint32_t ct, r2, rt, bt;
              d_ct.divmod(tile, r2, ct);
              d_rt.divmod(r2, bt, rt);
              const int cw = (int)ct * p.Wt - p.wlo, chh = (int)rt * p.TH - p.hlo, cb = (int)bt * p.TB;
              tc::tma_load_4d(sbase + (size_t)(mt * p.TA) * p.a_bytes, &tmap0, &sh.full[slot], 2 * cw, chh, cb, c8);
              if (p.TA > 1) tc::tma_load_4d(sbase + (size_t)(mt * p.TA + 1) * p.a_bytes, &tmap1, &sh.full[slot], 2 * cw, chh, cb, c8);
              if (p.TA > 2) tc::tma_load_4d(sbase + (size_t)(mt * p.TA + 2) * p.a_bytes, &tmap2, &sh.full[slot], 2 * cw, chh, cb, c8);
            }
            if (ld_b) tc::bulk_load_1d(sbase + p.b_off, bsrc + (size_t)cc * blk, blk, &sh.full[slot]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer (warp-converged, lane 0 issues)

    const uint32_t y = blockIdx.y;
    const uint64_t a_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(smem), p.m.a_lbo, 128);
    const uint64_t b_desc0 = tc::smem_desc_kmajor_noswz(tc::smem_u32(smem), p.m.b_lbo, 128) + (uint64_t)p.m.b_off16;
    const uint32_t a_lo0 = (uint32_t)a_desc0, a_hi = (uint32_t)(a_desc0 >> 32), b_lo0 = (uint32_t)b_desc0, b_hi = (uint32_t)(b_desc0 >> 32);
    uint32_t sc = 0, accq = 0;   // accq counts accumulator hand-offs (one per segment)
    for (uint32_t it = blockIdx.x; it < p.m.n_items; it += gridDim.x) {
      uint32_t started = 0, seg_pos = 0, open = 0;
      for (uint32_t t = 0; t < p.m.ntmpl[y]; ++t) {
        const uint32_t pb = p.m.tmpl_begin[y][t], pc = p.m.tmpl_cnt[y][t];
        for (uint32_t cc = 0; cc < p.m.chunks; ++cc, ++sc) {
          const uint32_t acc = accq & 1u, aph = (accq >> 1) & 1u;
          if (!open) {   // first stage of a segment: the accumulator must have been drained
            tc::mbar_wait_soft(&sh.acc_empty[acc], aph ^ 1u, p.err, 702, &sh.abort);
            open = 1; started = 0;
          }
          const uint32_t slot = sc & p.m.st_mask, ph = (sc >> p.m.st_log2) & 1u;
          tc::mbar_wait_soft(&sh.full[slot], ph, p.err, 703, &sh.abort);
          tc::tc_fence_after();
          const uint32_t s16 = slot * p.m.stage16;
          for (uint32_t mt = 0; mt < p.m.MT; ++mt) {
            const uint32_t d = tmem + (acc * p.m.MT + mt) * p.m.Nt;
            const uint32_t a_base = a_lo0 + s16 + mt * p.m.a_mt16, b_base = b_lo0 + s16;
            // flat program: one word per MMA of this stage template (tap x piece pair x K-step).  The first MMA of a
            // segment overwrites the accumulator; the rest is a straight unrolled stream of independent
            // load-word / add / add / MMA groups (a single warp issues them: dependent chains cost MMA rate)
            if (!(p.dbg & 2)) {
              tc::mma_f16_x4(d, a_base, a_hi, b_base, b_hi, p.m.idesc, p.m.prog4[pb], started);
#pragma unroll 2
              for (uint32_t e = 1; e < pc; ++e)
                tc::mma_f16_x4(d, a_base, a_hi, b_base, b_hi, p.m.idesc, p.m.prog4[pb + e], 1u);
            }
          }
          // MNB_PK_DEBUG bit 32 (with bit 2, timing experiments): plain mbarrier arrivals instead of tcgen05.commit
          if (p.dbg & 32) { if (lane == 0) tc::mbar_arrive(&sh.empty[slot]); } else tc::mma_commit_elect(&sh.empty[slot]);
          __syncwarp();
          started = 1;
          if (++seg_pos == p.m.seg_len) {   // segment complete: hand the accumulator to the epilogue
            if (p.dbg & 32) { if (lane == 0) tc::mbar_arrive(&sh.acc_full[acc]); } else tc::mma_commit_elect(&sh.acc_full[acc]);
            __syncwarp();
            seg_pos = 0; open = 0; ++accq;
          }
        }
      }
      if (open || p.m.ntmpl[y] == 0) {      // last (partial) segment, or an output phase without any filter tap
        const uint32_t acc = accq & 1u, aph = (accq >> 1) & 1u;
        if (!open) tc::mbar_wait_soft(&sh.acc_empty[acc], aph ^ 1u, p.err, 702, &sh.abort);
        if (p.dbg & 32) { if (lane == 0) tc::mbar_arrive(&sh.acc_full[acc]); } else tc::mma_commit_elect(&sh.acc_full[acc]);
        __syncwarp();
        ++accq;
      }
    }
  } else if (warp >= 4) {
    // ================================================================= epilogue: TMEM -> scale/bias or STE -> fp32 NCHW
    constexpr int NEPI = 32 * ConvCfg<SEG>::EPIW;
    const int q = (warp - 4) & 3, half = (warp - 4) >> 2, et = tid - 128;   // TMEM lane quarter, slot parity (8 epilogue warps)
    const int m = q * 32 + lane;                     // accumulator row = position of the zero-padded tile raster
    const int tb = m / (p.THH * p.BW);
    const int rem = m - tb * (p.THH * p.BW);
    const int th = rem / p.BW, wc = rem - th * p.BW;
    const bool row_ok = tb < p.TB && th < p.TH && wc < p.Wt;
    const int y = blockIdx.y, ya = p.ny == 4 ? (y >> 1) : 0, yb = p.ny == 4 ? (y & 1) : 0;
    const int64_t plane = (int64_t)p.OH * p.OW;
    const float a_sc = p.a_scale ? __ldg(p.a_scale) : p.a_scale_const;
    MnbActQ pq;
    float pzp = 0.f;
    if (p.post_out) {
      pq = mnb_load_actq(p.post_q);
      if (p.post_q.mode == MNB_ACT_IAO && p.post_q.zero_point) pzp = __ldg(p.post_q.zero_point);
    }
    uint32_t accq = 0;
    const FastDiv e_nt(p.n_ntiles), e_g(p.G), e_ct(p.col_tiles), e_rt(p.row_tiles);
    for (int it = blockIdx.x; it < p.n_items; it += gridDim.x) {
      uint32_t nt_u, r1_u, g_u, mg_u;
      e_nt.divmod((uint32_t)it, r1_u, nt_u);
      e_g.divmod(r1_u, mg_u, g_u);
      const int nt = (int)nt_u, g = (int)g_u, mg = (int)mg_u;
      const int n_base = g * p.ng + nt * p.Nt;                // first output channel of this N tile
      const int n_cnt = min(p.Nt, p.ng - nt * p.Nt);
      // per-channel constants of this N tile (the previous item's readers are done: barrier at the end of the loop body)
      for (int n = et; n < p.Nt; n += NEPI) {
        float sc = 1.f, bs = 0.f;
        if (n < n_cnt) {
          sc = p.n_scale ? __fmul_rn(a_sc, __ldg(p.n_scale + n_base + n)) : a_sc;
          if (p.bias) bs = __ldg(p.bias + n_base + n);
        }
        sh.epi_scale[n] = sc; sh.epi_bias[n] = bs;
      }
      epi_bar_sync<NEPI>();
      const int nseg = SEG ? p.nseg[y] : 1;
      // running sums of the item's accumulator columns (segmented mode only: MT * Nt <= 128 -> 8 slots of 16 columns;
      // slot = mt * (Nt / 16) + column chunk).  The slot loop is fully unrolled so that rs[][] stays in registers.
      float rs[SEG ? 8 : 1][16];
      const int nc16 = p.Nt >> 4, nslots = p.MT * nc16;
      for (int seg = 0; seg < nseg; ++seg, ++accq) {
        const uint32_t acc = accq & 1u, aph = (accq >> 1) & 1u;
        if (!tc::mbar_wait(&sh.acc_full[acc], aph, p.err, 704)) goto done;
        tc::tc_fence_after();
        const bool last = seg == nseg - 1;
        int mt_cur = -1;
        bool valid = false;
        float* orow = nullptr;
        const uint8_t* brow = nullptr;
        int64_t prow = 0;      // vector index of this thread's position in octet 0 of the consumer's operand plane
        // one slot = 16 accumulator columns of one M tile.  Segmented kernels need rs[slot] with a compile-time index (8 slots,
        // unrolled); the others run a ROLLED loop: unrolled 32 x, this body was 1 MB of SASS and the epilogue warps stalled
        // on instruction fetch
        auto do_slot = [&](const int slot, const int mt, const int c16, float (&rsl)[16]) {
          const int n0 = c16 * 16;
          if (mt != mt_cur) {   // output row of this thread in M tile mt
            mt_cur = mt;
            const int tile = mg * p.MT + mt;
            uint32_t ct_u, r2_u, rt_u, bt_u;
            e_ct.divmod((uint32_t)tile, r2_u, ct_u);
            e_rt.divmod(r2_u, bt_u, rt_u);
            const int ct = (int)ct_u, rt = (int)rt_u, bt = (int)bt_u;
            const int b = bt * p.TB + tb, i = rt * p.TH + th, j = ct * p.Wt + wc;
            valid = row_ok && tile < p.n_mtiles && b < p.B && i < p.OHr && j < p.OWr;
            const int oh = i * p.omul + ya, ow = j * p.omul + yb;
            orow = p.out ? p.out + ((int64_t)b * p.NOUT + n_base) * plane + (int64_t)oh * p.OW + ow : nullptr;
            brow = p.bits8 ? p.bits8 + (int64_t)b * p.C8O * plane + (int64_t)oh * p.OW + ow : nullptr;
            if (!SEG && p.post_out) {
              if (p.post_split)   // octet index (h%2 * 2 + w%2) * C8 + c/8 of a [.., OH/2, OW/2] plane
                prow = (((int64_t)b * 4 * p.C8O + ((oh & 1) * 2 + (ow & 1)) * p.C8O) * (p.OH >> 1) + (oh >> 1)) * (p.OW >> 1) + (ow >> 1);
              else
                prow = ((int64_t)b * p.C8O * p.OH + oh) * p.OW + ow;
            }
          }
          uint32_t r[16];
          if (!p.zero_y[y] && !(p.dbg & 4)) {
            tmem_ld_32x16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)((acc * p.MT + mt) * p.Nt + n0), r);
            tc::tmem_ld_wait();
          } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) r[k] = 0u;
          }
          if (SEG) {   // accumulate the segment (round-to-nearest fp32 adds), write only after the last one
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const float v = seg == 0 ? __uint_as_float(r[k]) : __fadd_rn(rsl[k], __uint_as_float(r[k]));
              rsl[k] = v;
              r[k] = __float_as_uint(v);
            }
            if (!last) return;
          }
          if (!valid || n0 >= n_cnt || (p.dbg & 1)) return;
          float sc[16], bs[16];
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const float4 a = *reinterpret_cast<const float4*>(&sh.epi_scale[n0 + 4 * v]);
            const float4 c = *reinterpret_cast<const float4*>(&sh.epi_bias[n0 + 4 * v]);
            sc[4 * v] = a.x; sc[4 * v + 1] = a.y; sc[4 * v + 2] = a.z; sc[4 * v + 3] = a.w;
            bs[4 * v] = c.x; bs[4 * v + 1] = c.y; bs[4 * v + 2] = c.z; bs[4 * v + 3] = c.w;
          }
          float* op = orow + (int64_t)n0 * plane;
          if (!SEG && p.post_out) {
            // forward conv of a frozen inference graph: y = acc * scale + bias [-> ReLU] -> consumer's quantizer -> bf16 levels
            float lev[16], yv[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const float v = fmaf(__uint_as_float(r[k]), sc[k], bs[k]);
              if (orow && n0 + k < n_cnt) op[(int64_t)k * plane] = v;
              yv[k] = p.post_relu ? fmaxf(v, 0.f) : v;
            }
            uint32_t passbits;
            mnb_act_levels<16>(pq, yv, lev, passbits);
#pragma unroll
            for (int k = 0; k < 16; ++k) lev[k] = n0 + k < n_cnt ? lev[k] + pzp : 0.f;
            const int64_t oct_stride = p.post_split ? (int64_t)(p.OH >> 1) * (p.OW >> 1) : plane;
            const int oc8 = (n_base + n0) >> 3;
            uint4* dst = p.post_out + prow + (int64_t)oc8 * oct_stride;
            dst[0] = make_uint4(pack2(lev[0], lev[1]), pack2(lev[2], lev[3]), pack2(lev[4], lev[5]), pack2(lev[6], lev[7]));
            if (n0 + 8 < n_cnt)
              dst[oct_stride] = make_uint4(pack2(lev[8], lev[9]), pack2(lev[10], lev[11]), pack2(lev[12], lev[13]), pack2(lev[14], lev[15]));
          } else if (p.mode == 0 || !brow) {
#pragma unroll
            for (int k = 0; k < 16; ++k, op += plane)
              if (n0 + k < n_cnt) *op = fmaf(__uint_as_float(r[k]), sc[k], bs[k]);
          } else {
            // STE of the activation quantizer that fed the forward conv: the reference computes ((g*s)*pass)/s (IAO) or
            // (((g*s)/s)*pass)*0.1 (DoReFa); (g*s)/s is g to within one ulp, so g itself is passed
            const int oc0 = (n_base + n0) >> 3;     // n_base + n0 is a multiple of 8 (checked on the host)
            const uint32_t m0 = __ldg(brow + (int64_t)oc0 * plane);
            const uint32_t m1 = (n0 + 8 < n_cnt) ? __ldg(brow + (int64_t)(oc0 + 1) * plane) : 0u;
            const uint32_t mask = m0 | (m1 << 8);
#pragma unroll
            for (int k = 0; k < 16; ++k, op += plane)
              if (n0 + k < n_cnt) *op = ((mask >> k) & 1u) ? __uint_as_float(r[k]) * p.gain : 0.f;
          }
                };
        if (SEG) {
          int mt = 0, c16 = 0;
#pragma unroll
          for (int slot = 0; slot < 8; ++slot) {
            if (slot < nslots) do_slot(slot, mt, c16, rs[SEG ? slot : 0]);
            if (++c16 == nc16) { c16 = 0; ++mt; }
          }
        } else {
#pragma unroll 1
          for (int mt = 0, slot = 0; mt < p.MT; ++mt)
#pragma unroll 1
            for (int c16 = 0; c16 < nc16; ++c16, ++slot)
              if (ConvCfg<SEG>::EPIW == 4 || (slot & 1) == half) do_slot(slot, mt, c16, rs[0]);
        }
        tc::tc_fence_before();
        tc::mbar_arrive(&sh.acc_empty[acc]);
      }
      epi_bar_sync<NEPI>();   // everyone is done with epi_scale / epi_bias of this item
    }
  }
done:
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc::tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols));
  }
}

// Map over term plane `t` of a packed tensor [b][octet][h][w][8 x bf16].  The TMA unit's cost is per box ROW (~12 cycles
// per row and SM whatever its length: with the 16-byte channel octet as innermost dimension a 170-position x 16-channel
// box took 4000 cycles), so the 16-byte pixels of one image row are declared as ONE dimension of 8-byte elements:
// dims (2*W, H, B, octets), box (2*BW, rows, images, octets) - same shared-memory image [octet][image][row][col][16 B],
// halo columns still zero-filled (start coordinate -2*wlo: a multiple of 16 bytes).
static int make_pk_tmap(CUtensorMap* m, const void* base, int64_t plane_bytes, int t, int B, int C8tot, int H, int W,
                        int bw, int bh, int bb, int bc8) {
  const uint64_t HW = (uint64_t)H * W;
  uint64_t dims[4] = {(uint64_t)W * 2, (uint64_t)H, (uint64_t)B, (uint64_t)C8tot};
  uint64_t strides[3] = {(uint64_t)W * 16, (uint64_t)C8tot * HW * 16, HW * 16};
  uint32_t box[4] = {(uint32_t)bw * 2, (uint32_t)bh, (uint32_t)bb, (uint32_t)bc8};
  return mnb_make_tmap_strided(m, reinterpret_cast<const uint8_t*>(base) + (int64_t)t * plane_bytes, 8, 4, dims, strides, box);
}

template <typename K>
static int set_max_smem(K kernel, int bytes) {
  // the attribute is a property of the function on a device: set it once per (function, device).  Keyed by the function
  // ADDRESS (instantiations of one template share their pointer TYPE, so a per-type static would cover only the first)
  static const void* seen_fn[32];
  static int seen_dev[32], nseen = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  const void* fn = reinterpret_cast<const void*>(kernel);
  for (int i = 0; i < nseen; ++i)
    if (seen_fn[i] == fn && seen_dev[i] == dev) return 0;
  cudaError_t ce = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (ce != cudaSuccess) return mnb_fail((int)ce, "cudaFuncSetAttribute: %s", cudaGetErrorString(ce));
  if (nseen < 32) { seen_fn[nseen] = fn; seen_dev[nseen] = dev; ++nseen; }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// weight gradient: dW[k][c][tap] = sum over positions of dy[pos][k] * x[pos + tap][c]   (MN-major operands)
// ---------------------------------------------------------------------------------------------------------
struct WgPlan {
  int B, G, R, S, stride, ntap;
  int P, Q, K8, HX, WX, C8X, nkph;      // dy dims / octets; x planes as stored
  int cin_g, cout_g, gm;       // channels per (merged) group; gm = original groups per merged group
  int hlo, hhi, wlo, whi, BW, TH, THH, rows_dy, rows_x, row_tiles;
  int Nc, n_ctiles, n_ktiles, tpg, n_tg, NI, nsub, nstg_total, splits, stg_per_split;
  int TA, TX, npairs, pair_a[MAXPAIR], pair_b[MAXPAIR];
  int tap_kph[MAXTAP], tap_off[MAXTAP];   // per tap: k-phase plane and start-row offset in the x block
  int kph_used[4], nkph_used, kph_slot[4];
  int dy_box_bytes, x_box_bytes, dy_bytes, x_bytes, sub_bytes, stage_bytes, nstage, st_log2, smem_bytes, tmem_cols;
  int64_t partial_floats;
};

static int make_wg_plan_nc(const mnb_conv_shape* s, int TA, int TX, WgPlan& p, int nc_cap) {
  MNB_REQUIRE(s != nullptr, "conv shape is NULL");
  memset(&p, 0, sizeof(p));
  const int C = s->in_c, K = s->out_c, G = s->groups, H = s->in_h, W = s->in_w, R = s->ker_h, S = s->ker_w;
  MNB_REQUIRE(s->batch > 0 && C > 0 && K > 0 && H > 0 && W > 0 && G > 0 && C % G == 0 && K % G == 0, "bad conv shape");
  if (s->dil_h != 1 || s->dil_w != 1) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: dilation != 1");
  if (s->stride_h != s->stride_w || (s->stride_h != 1 && s->stride_h != 2)) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: stride");
  const int st = s->stride_h, ph_ = s->pad_h, pw_ = s->pad_w;
  if (ph_ > R - 1 || pw_ > S - 1) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: padding larger than the filter");
  if (st == 2 && ((H | W) & 1)) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: stride 2 needs even H and W");
  if (R * S > MAXTAP) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: more than 64 taps");
  p.B = s->batch; p.G = G; p.R = R; p.S = S; p.stride = st; p.ntap = R * S;
  p.P = (H + 2 * ph_ - R) / st + 1; p.Q = (W + 2 * pw_ - S) / st + 1;
  if (p.P < 1 || p.Q < 1) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: empty output");
  p.cin_g = C / G; p.cout_g = K / G;
  if (G > 1 && ((p.cin_g % 8) || (p.cout_g % 8))) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: grouped conv needs channels per group % 8 == 0");
  // Small groups are MERGED: gm neighbouring groups form one 128-row accumulator block (rows = their output channels,
  // columns = their input channels); an MMA costs 61 cycles whether it is 128 x 16 or 128 x 64, so computing the discarded
  // off-diagonal blocks is free and the MMA count drops by gm.  The reduction kernel keeps the diagonal blocks only.
  p.gm = 1;
  while (G % (p.gm * 2) == 0 && p.gm * 2 * p.cout_g <= 128 && p.gm * 2 * p.cin_g <= 256) p.gm *= 2;
  if (const char* e = getenv("MNB_PK_WG_MERGE")) { if (atoi(e) == 0) p.gm = 1; }
  p.G = G / p.gm; p.cin_g *= p.gm; p.cout_g *= p.gm;
  p.K8 = ceil_div(K, 8); p.C8X = ceil_div(C, 8);
  p.nkph = st == 2 ? 4 : 1; p.HX = H / st; p.WX = W / st;
  p.TA = TA; p.TX = TX;
  { Plan tmp; memset(&tmp, 0, sizeof(tmp)); make_pairs(TA, TX, tmp); p.npairs = tmp.npairs;
    for (int i = 0; i < tmp.npairs; ++i) { p.pair_a[i] = tmp.pair_a[i]; p.pair_b[i] = tmp.pair_b[i]; } }
  int sh_[MAXTAP], sw_[MAXTAP];
  int hlo = 0, hhi = 0, wlo = 0, whi = 0;
  for (int i = 0; i < 4; ++i) p.kph_slot[i] = -1;
  for (int r = 0; r < R; ++r)
    for (int q = 0; q < S; ++q) {
      const int t = r * S + q, dr = r - ph_, ds = q - pw_;
      int kp = 0, sh = dr, sw = ds;
      if (st == 2) { const int fh = dr & 1, fw = ds & 1; kp = fh * 2 + fw; sh = (dr - fh) / 2; sw = (ds - fw) / 2; }
      p.tap_kph[t] = kp; sh_[t] = sh; sw_[t] = sw;
      if (p.kph_slot[kp] < 0) { p.kph_slot[kp] = p.nkph_used; p.kph_used[p.nkph_used++] = kp; }
      hlo = std::max(hlo, -sh); hhi = std::max(hhi, sh); wlo = std::max(wlo, -sw); whi = std::max(whi, sw);
    }
  p.hlo = hlo; p.hhi = hhi; p.wlo = wlo; p.whi = whi;
  // raster: rows of BW >= Q + halo columns; TH * BW must be a multiple of 16 (MMA K-steps of 16 positions)
  const int need = p.Q + wlo + whi;
  if (need > 128) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: row wider than 128 positions");
  // N tile over input channels and TAP GROUPS: one CTA accumulates tpg taps x Nc columns (<= 512 TMEM columns).  An MMA of
  // N <= 64 costs the same 61 cycles as one of N = 128, so the N tile is made as wide as the layer allows (up to 256) and
  // the taps are split over CTAs instead (each tap group re-reads the operands, mostly from L2): the MMA count is
  // positions/16 x taps x pairs x ceil(C / Nc) - with Nc = 48 a 256-channel 3x3 layer issued six N = 48 MMAs where two
  // tap groups of N = 256 do the same work at full tensor rate.
  int nc = std::min(nc_cap, round_up(p.cin_g, 16));
  if (const char* e = getenv("MNB_PK_WG_NC")) nc = std::max(16, std::min(nc, atoi(e) / 16 * 16));
  p.n_ctiles = ceil_div(p.cin_g, nc);
  p.Nc = round_up(ceil_div(p.cin_g, p.n_ctiles), 16);      // balance the tiles
  p.n_ctiles = ceil_div(p.cin_g, p.Nc);
  p.n_ktiles = ceil_div(p.cout_g, 128);
  p.tpg = std::max(1, std::min(p.ntap, 512 / p.Nc));
  p.n_tg = ceil_div(p.ntap, p.tpg);
  p.tpg = ceil_div(p.ntap, p.n_tg);                        // balance the groups
  int cols = 32;
  while (cols < p.tpg * p.Nc) cols <<= 1;
  if (cols > 512) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: accumulators exceed tensor memory");
  p.tmem_cols = cols;
  // stage = NI sub-blocks (one image row-tile each): dy [TA][16 octets][rows_dy], x [TX][k-phase][Nc/8][rows_x].
  // Pick the raster (BW, TH) with the best useful fraction whose sub-block fits four times (else twice).
  auto sub_bytes_of = [&](int bw, int th) {
    const int dyb = round_up(16 * th * bw * 16, 128);
    const int xb = round_up((p.Nc / 8) * (th + hlo + hhi) * bw * 16 + 16 * 16, 128);
    return TA * dyb + TX * p.nkph_used * xb;
  };
  int best_bw = 0, best_th = 0;
  double best_score = -1;
  for (int pass = 0; pass < 2 && !best_bw; ++pass) {
    const int limit = (kSmemBudget - 2048) / (pass == 0 ? 4 : 2);
    for (int bw = need; bw <= std::min(128, need + 15); ++bw)
      for (int th = 1; th <= p.P; ++th) {
        if ((th * bw) % 16) continue;
        if (th + hlo + hhi > 256 || sub_bytes_of(bw, th) > limit) continue;
        const double eff = (double)p.Q / bw, fill = std::min(1.0, (double)th * bw / 64.0);
        const double score = eff * (0.5 + 0.5 * fill);
        if (score > best_score) { best_score = score; best_bw = bw; best_th = th; }
      }
  }
  if (!best_bw) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: no raster fits shared memory (N tile %d)", p.Nc);
  p.BW = best_bw; p.TH = best_th; p.THH = p.TH + hlo + hhi;
  p.rows_dy = p.TH * p.BW; p.rows_x = p.THH * p.BW;
  p.row_tiles = ceil_div(p.P, p.TH);
  for (int t = 0; t < p.ntap; ++t) p.tap_off[t] = (sh_[t] + hlo) * p.BW + (sw_[t] + wlo);
  p.dy_box_bytes = 16 * p.rows_dy * 16;
  p.x_box_bytes = (p.Nc / 8) * p.rows_x * 16;
  p.dy_bytes = round_up(p.dy_box_bytes, 128);
  p.x_bytes = round_up(p.x_box_bytes + 16 * 16, 128);       // + slack rows read past the last plane (must stay finite: zeroed)
  p.sub_bytes = TA * p.dy_bytes + TX * p.nkph_used * p.x_bytes;
  p.nsub = p.B * p.row_tiles;
  const int stage_target = 52 * 1024;
  p.NI = std::max(1, std::min(std::min(p.nsub, 8), stage_target / p.sub_bytes));
  p.stage_bytes = round_up(p.NI * p.sub_bytes, 1024);
  const int nst = (kSmemBudget - 1024) / p.stage_bytes;
  if (nst < 2) return mnb_fail(MNB_E_UNSUPPORTED, "pk wgrad: fewer than two stages fit");
  p.nstage = nst >= 4 ? 4 : 2;
  p.st_log2 = p.nstage == 4 ? 2 : 1;
  p.smem_bytes = p.nstage * p.stage_bytes + 1024;
  p.nstg_total = ceil_div(p.nsub, p.NI);
  const int n_kc = p.n_ktiles * p.n_ctiles * p.G * p.n_tg;
  p.splits = std::max(1, std::min(p.nstg_total, std::max(1, MNB_NUM_SMS / n_kc)));
  // keep accumulation chains short: tcgen05.mma truncates the running fp32 sum after every instruction (a bias of
  // ~2e-8 of |D| per MMA), so one accumulator takes <= ~192 MMAs; the partial sums are added with RN adds
  const int chain_per_stage = p.NI * (p.rows_dy / 16) * p.npairs;
  int chain_max = 256;
  if (const char* e = getenv("MNB_PK_WG_CHAIN")) chain_max = std::max(1, atoi(e));
  while (p.splits < p.nstg_total && (int64_t)ceil_div(p.nstg_total, p.splits) * chain_per_stage > chain_max) ++p.splits;
  p.stg_per_split = ceil_div(p.nstg_total, p.splits);
  p.splits = ceil_div(p.nstg_total, p.stg_per_split);
  p.partial_floats = (int64_t)p.splits * p.G * p.n_ktiles * p.n_ctiles * p.ntap * p.Nc * 128;
  return 0;
}

// the widest N tile whose operand blocks fit shared memory next to the dy planes (split fp32 x and stride-2 phase planes are
// several times larger than one plane of integer levels)
static int make_wg_plan(const mnb_conv_shape* s, int TA, int TX, WgPlan& p) {
  int rc = MNB_E_UNSUPPORTED;
  for (int cap = 256; cap >= 16; cap /= 2) {
    rc = make_wg_plan_nc(s, TA, TX, p, cap);
    if (rc != MNB_E_UNSUPPORTED) return rc;
  }
  return rc;
}

struct WgParams {
  struct Mma {
    uint32_t stg_per_split, nstg_total, NI, ksteps, ntap, tpg, n_tg, Nc, npairs, st_mask, st_log2, stage16, sub16, dy_term16, x_off16,
        x_term16, x_kph16, idesc, dy_sbo, x_sbo, nsub;
    uint32_t pair_a16[MAXPAIR], pair_b16[MAXPAIR];   // piece-plane offsets of the pairs (16-byte units)
    // per (piece pair, tap group of this CTA, four taps): x-operand offsets = pair plane + k-phase slot + tap row offset,
    // 0xffffffff behind the last tap of a group (one 128-bit constant load and one election per four MMAs)
    alignas(16) uint4 progb4[MAXPAIR * MAXTAP / 4 + MAXPAIR * 16];
    uint32_t g4;                        // uint4 entries per (pair, tap group) = ceil(tpg / 4)
  } m;
  int G, n_ktiles, n_ctiles, n_tg, tpg, splits, stg_per_split, nstg_total, NI, nsub, row_tiles, TA, TX, nkph_used, kph_used[4];
  int K8, C8X, cout_g8, cin_g8, Nc8, TH, hlo, wlo, stage_bytes, sub_bytes, dy_bytes, x_bytes, dy_box_bytes, x_box_bytes,
      st_mask, st_log2, smem_bytes, tmem_cols, ntap, Nc, cout_g, cin_g;
  float* partial;
  int* err;
};

struct alignas(16) WgShared {
  uint64_t full[MAXST], empty[MAXST], acc_full;
  uint32_t tmem_slot, abort;
};

__global__ void __launch_bounds__(NTHREADS, 1)
pk_wgrad_kernel(const __grid_constant__ CUtensorMap dy0, const __grid_constant__ CUtensorMap dy1,
                const __grid_constant__ CUtensorMap dy2, const __grid_constant__ CUtensorMap x0,
                const __grid_constant__ CUtensorMap x1, const __grid_constant__ CUtensorMap x2,
                const __grid_constant__ WgParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ WgShared sh;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < MAXST; ++i) { tc::mbar_init(&sh.full[i], 1); tc::mbar_init(&sh.empty[i], 1); }
    tc::mbar_init(&sh.acc_full, 1);
    sh.abort = 0;
    tc::fence_barrier_init();
    tc::prefetch_tmap(&dy0); tc::prefetch_tmap(&x0);
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&sh.tmem_slot)),
                 "r"((uint32_t)p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // every row an MMA can read must be finite (positions are the reduction dimension here): zero everything once,
  // the TMA boxes never touch the slack rows
  for (int i = tid; i < p.smem_bytes / 16; i += NTHREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sh.tmem_slot;
  // work item of this CTA: blockIdx.x = (((g * n_ktiles + kt) * n_ctiles + ct) * n_tg + tap group), blockIdx.y = split
  const int split = blockIdx.y;
  const int tg = blockIdx.x % p.n_tg;
  const int r0 = blockIdx.x / p.n_tg;
  const int t0 = tg * p.tpg, tn = min(p.tpg, p.ntap - t0);    // this CTA's filter taps
  const int ct = r0 % p.n_ctiles;
  const int r1 = r0 / p.n_ctiles;
  const int kt = r1 % p.n_ktiles, g = r1 / p.n_ktiles;
  const int stg0 = split * p.stg_per_split, stg1 = min(p.nstg_total, stg0 + p.stg_per_split);

  if (warp == 0) {
    if (lane == 0) {
      uint32_t sc = 0;
      const int k8 = g * p.cout_g8 + kt * 16, c8 = g * p.cin_g8 + ct * p.Nc8;
      for (int stg = stg0; stg < stg1; ++stg, ++sc) {
        const uint32_t slot = sc & (uint32_t)p.st_mask, ph = (sc >> p.st_log2) & 1u;
        if (!tc::mbar_wait(&sh.empty[slot], ph ^ 1u, p.err, 711)) goto done;
        const int sub0 = stg * p.NI, nsubs = min(p.NI, p.nsub - sub0);
        tc::mbar_arrive_expect_tx(&sh.full[slot], (uint32_t)(nsubs * (p.TA * p.dy_box_bytes + p.TX * p.nkph_used * p.x_box_bytes)));
        for (int si = 0; si < nsubs; ++si) {
          const int sub = sub0 + si;
          const int b = sub / p.row_tiles, rt = sub - b * p.row_tiles;
          uint8_t* sb = smem + (size_t)slot * p.stage_bytes + (size_t)si * p.sub_bytes;
          const int h0 = rt * p.TH;
          tc::tma_load_4d(sb, &dy0, &sh.full[slot], 0, h0, b, k8);
          if (p.TA > 1) tc::tma_load_4d(sb + p.dy_bytes, &dy1, &sh.full[slot], 0, h0, b, k8);
          if (p.TA > 2) tc::tma_load_4d(sb + 2 * p.dy_bytes, &dy2, &sh.full[slot], 0, h0, b, k8);
          uint8_t* xb = sb + (size_t)p.TA * p.dy_bytes;
          for (int tx = 0; tx < p.TX; ++tx)
            for (int ks = 0; ks < p.nkph_used; ++ks) {
              const CUtensorMap* tm = tx == 0 ? &x0 : (tx == 1 ? &x1 : &x2);
              tc::tma_load_4d(xb + (size_t)(tx * p.nkph_used + ks) * p.x_bytes, tm, &sh.full[slot], -2 * p.wlo, h0 - p.hlo, b,
                              p.kph_used[ks] * p.C8X + c8);
            }
        }
        // sub-blocks of a short last stage keep their previous (finite) contents; the MMA loop skips them
      }
    }
  } else if (warp == 1) {

    const uint64_t a_desc0 = tc::smem_desc_mnmajor_noswz(tc::smem_u32(smem), 128, p.m.dy_sbo);
    const uint64_t b_desc0 = tc::smem_desc_mnmajor_noswz(tc::smem_u32(smem), 128, p.m.x_sbo) + (uint64_t)p.m.x_off16;
    const uint32_t a_lo0 = (uint32_t)a_desc0, a_hi = (uint32_t)(a_desc0 >> 32), b_lo0 = (uint32_t)b_desc0, b_hi = (uint32_t)(b_desc0 >> 32);
    const uint32_t split_u = blockIdx.y;
    const uint32_t tgm = blockIdx.x % p.m.n_tg;
    const uint32_t t0m = tgm * p.m.tpg, tnm = min(p.m.tpg, p.m.ntap - t0m);
    const uint32_t s0 = split_u * p.m.stg_per_split;
    const uint32_t s1 = min(p.m.nstg_total, s0 + p.m.stg_per_split);
    uint32_t sc = 0, accf = 0;
    for (uint32_t stg = s0; stg < s1; ++stg, ++sc) {
      const uint32_t slot = sc & p.m.st_mask, ph = (sc >> p.m.st_log2) & 1u;
      tc::mbar_wait_soft(&sh.full[slot], ph, p.err, 712, &sh.abort);
      tc::tc_fence_after();
      const uint32_t nsubs = min(p.m.NI, p.m.nsub - stg * p.m.NI);
      for (uint32_t si = 0; si < nsubs; ++si) {
        const uint32_t s16 = slot * p.m.stage16 + si * p.m.sub16;
        uint32_t arow = a_lo0 + s16, brow = b_lo0 + s16;
        for (uint32_t j = 0; j < p.m.ksteps; ++j, arow += 16u, brow += 16u) {
          for (uint32_t pr = 0; pr < p.m.npairs; ++pr) {
            const uint32_t ad = arow + p.m.pair_a16[pr];
            uint32_t d = tmem, e = (pr * p.m.n_tg + tgm) * p.m.g4;
#pragma unroll 2
            for (uint32_t t = 0; t < tnm; t += 4u, ++e, d += 4u * p.m.Nc)
              tc::mma_f16_x4_taps(d, p.m.Nc, ad, a_hi, brow, b_hi, p.m.idesc, p.m.progb4[e], accf);
            accf = 1u;   // every tap accumulator has been written once: accumulate from here on
          }
        }
      }
      tc::mma_commit_elect(&sh.empty[slot]);
      __syncwarp();
    }
    tc::mma_commit_elect(&sh.acc_full);
    __syncwarp();
  } else if (warp >= 4) {
    // partial[split][g][kt][ct][tap][c][k]: lanes = k -> coalesced
    const int q = warp - 4;
    const int kl = q * 32 + lane;
    if (!tc::mbar_wait(&sh.acc_full, 0, p.err, 713)) goto done;
    tc::tc_fence_after();
    float* dst = p.partial + ((((int64_t)split * p.G + g) * p.n_ktiles + kt) * p.n_ctiles + ct) * (int64_t)(p.ntap * p.Nc * 128) +
                 (int64_t)t0 * p.Nc * 128 + kl;
    const bool any = stg1 > stg0;
    for (int col = 0; col < tn * p.Nc; col += 16) {
      uint32_t r[16];
      tmem_ld_32x16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)col, r);
      tc::tmem_ld_wait();
#pragma unroll
      for (int k = 0; k < 16; ++k) dst[(int64_t)(col + k) * 128] = any ? __uint_as_float(r[k]) : 0.f;
    }
    tc::tc_fence_before();
  }
done:
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc::tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols));
  }
}

// dw[k][c][tap] = mul(k) * sum over splits (fixed order: deterministic); mul = a_scale / kdiv[k] (either may be NULL).
// G merged groups of gm original groups each: only the diagonal (same original group) blocks are read.
// One block = the 128 output channels of a k tile for ONE (input channel, tap): the partials are read along k, their
// contiguous dimension (512-byte runs per warp), four splits in flight per thread; |W| threads in total.
__global__ void __launch_bounds__(128) wg_reduce_kernel(const float* __restrict__ partial, int splits, int G, int gm, int n_ktiles,
                                                        int n_ctiles, int ntap, int Nc, int cout_g, int cin_g,
                                                        const float* __restrict__ a_scale, const float* __restrict__ kdiv,
                                                        float* __restrict__ dw) {
  // cout_g / cin_g: channels per ORIGINAL group.  grid = (cin_g * ntap, k tiles of the original group, original groups)
  const int go = blockIdx.z, ktile = blockIdx.y;
  const int c = blockIdx.x / ntap, tap = blockIdx.x - c * ntap;
  const int g = go / gm, gi = go - g * gm;
  const int kk = ktile * 128 + threadIdx.x;         // output channel inside the original group
  if (kk >= cout_g) return;
  const int64_t tile = (int64_t)ntap * Nc * 128;
  const int64_t split_stride = (int64_t)G * n_ktiles * n_ctiles * tile;
  const int km = gi * cout_g + kk, cm = gi * cin_g + c;     // row / column inside the merged group
  const int kt = km >> 7, kl = km & 127, ct = cm / Nc, cl = cm - ct * Nc;
  const float* src = partial + (((int64_t)g * n_ktiles + kt) * n_ctiles + ct) * tile + ((int64_t)tap * Nc + cl) * 128 + kl;
  float acc = 0.f;
  int s = 0;
  for (; s + 4 <= splits; s += 4) {
    const float v0 = __ldg(src + (int64_t)s * split_stride), v1 = __ldg(src + (int64_t)(s + 1) * split_stride),
                v2 = __ldg(src + (int64_t)(s + 2) * split_stride), v3 = __ldg(src + (int64_t)(s + 3) * split_stride);
    acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v0), v1), v2), v3);
  }
  for (; s < splits; ++s) acc = __fadd_rn(acc, __ldg(src + (int64_t)s * split_stride));
  const int kout = go * cout_g + kk;
  if (a_scale || kdiv) {
    const float as = a_scale ? __ldg(a_scale) : 1.f;
    acc = __fmul_rn(acc, kdiv ? __fdiv_rn(as, __ldg(kdiv + kout)) : as);
  }
  dw[((int64_t)kout * cin_g + c) * ntap + tap] = acc;
}

}  // namespace pk

// =========================================================================================================
// C-ABI
// =========================================================================================================
extern "C" int64_t mnb_pk_act_bytes(int32_t batch, int32_t channels, int32_t h, int32_t w, int32_t terms) {
  return (int64_t)terms * batch * ((channels + 7) / 8) * h * w * 16;
}

extern "C" int mnb_pk_pack_act(const float* x, int32_t batch, int32_t channels, int32_t h, int32_t w,
                               const mnb_act_qparams* qp, int32_t terms, const float* ch_scale, int32_t phase_split,
                               void* out_pk, uint8_t* bits8, mnb_stream_t stream) {
  return mnb_pk_pack_act_relu(x, batch, channels, h, w, qp, terms, ch_scale, phase_split, 0, out_pk, bits8, stream);
}

extern "C" int mnb_pk_pack_act_relu(const float* x, int32_t batch, int32_t channels, int32_t h, int32_t w,
                                    const mnb_act_qparams* qp, int32_t terms, const float* ch_scale, int32_t phase_split,
                                    int32_t relu, void* out_pk, uint8_t* bits8, mnb_stream_t stream) {
  MNB_REQUIRE(x && out_pk, "NULL pk_pack_act pointer");
  MNB_REQUIRE(batch > 0 && channels > 0 && h > 0 && w > 0 && terms >= 1 && terms <= 3, "bad pk_pack_act arguments");
  MNB_REQUIRE((reinterpret_cast<uintptr_t>(out_pk) & 15) == 0, "packed tensor must be 16-byte aligned");
  if (phase_split) MNB_REQUIRE(((h | w) & 1) == 0, "phase split needs even H and W");
  const int C8 = (channels + 7) / 8;
  const int64_t plane_vecs = (int64_t)batch * C8 * h * w;
  MNB_REQUIRE((int64_t)batch * C8 <= 65535 * 8 && (int64_t)h * w < (1ll << 31), "pk_pack_act: too many (image, octet) planes");
  const int hw = h * w;
  const int tx = std::min(256, (hw + 31) / 32 * 32), ty = 256 / tx;     // threads along positions / planes per block
  const int planes = batch * C8, gy = (planes + ty - 1) / ty;
  const int bx = std::max(1, std::min((hw + tx - 1) / tx, std::max(1, (MNB_NUM_SMS * 16) / std::max(1, gy))));
  if (gy > 65535) return mnb_fail(MNB_E_UNSUPPORTED, "pk_pack_act: %d (image, octet) planes exceed the grid", planes);
  const dim3 blocks(bx, gy), threads(tx, ty);
  cudaStream_t st = (cudaStream_t)stream;
  if (qp) {
    MNB_REQUIRE(qp->mode == MNB_ACT_DOREFA || qp->mode == MNB_ACT_IAO || qp->mode == MNB_ACT_SIGN, "unknown activation quantizer");
    if (qp->mode == MNB_ACT_DOREFA) MNB_REQUIRE(qp->bits >= 2 && qp->bits <= 8, "DoReFa a_bits must be in [2,8]");
    const int a_off = qp->mode == MNB_ACT_IAO ? qp->qmin : (qp->mode == MNB_ACT_SIGN ? -1 : 0);
    pk::pack_act_kernel<1><<<blocks, threads, 0, st>>>(x, batch, channels, h, w, C8, terms, nullptr, *qp, a_off, phase_split,
                                                   reinterpret_cast<uint4*>(out_pk), plane_vecs, bits8, relu);
  } else {
    mnb_act_qparams none{};
    pk::pack_act_kernel<0><<<blocks, threads, 0, st>>>(x, batch, channels, h, w, C8, terms, ch_scale, none, 0, phase_split,
                                                   reinterpret_cast<uint4*>(out_pk), plane_vecs, nullptr, relu);
  }
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_bn_sign_bwd_pack(const float* g, const uint32_t* pass_bits, const float* x, int32_t batch, int32_t channels,
                                    int32_t hw, const float* mean, const float* invstd, const float* gamma, const float* dgamma,
                                    const float* dbeta, int32_t out_shuffle_groups, const float* ch_scale, int32_t terms,
                                    float* dx, void* dy_packed, mnb_stream_t stream) {
  MNB_REQUIRE(g && pass_bits && x && mean && invstd && gamma && dgamma && dbeta && dy_packed, "NULL bn_sign_bwd_pack pointer");
  MNB_REQUIRE(batch > 0 && channels > 0 && hw > 0 && terms >= 1 && terms <= 3, "bad bn_sign_bwd_pack arguments");
  MNB_REQUIRE(out_shuffle_groups >= 1 && channels % out_shuffle_groups == 0, "shuffle groups %d do not divide %d channels",
              out_shuffle_groups, channels);
  if (channels % 8 || (reinterpret_cast<uintptr_t>(dy_packed) & 15))
    return mnb_fail(MNB_E_UNSUPPORTED, "packed BatchNorm backward needs channels %% 8 == 0 and a 16-byte aligned output");
  if (hw % 32) return mnb_fail(MNB_E_UNSUPPORTED, "packed BatchNorm backward needs H*W %% 32 == 0");
  const int c8n = channels / 8;
  auto al = [](const void* p, int a) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & (uintptr_t)(a - 1)) == 0; };
  const int vec = (hw % 128 == 0 && al(g, 16) && al(x, 16) && al(dx, 16)) ? 4 : ((hw % 64 == 0 && al(g, 8) && al(x, 8) && al(dx, 8)) ? 2 : 1);
  const int64_t warps = (int64_t)batch * c8n * (hw / (32 * vec));
  const int blocks = (int)std::min<int64_t>(mnb_ceil_div(warps, 8), (int64_t)MNB_NUM_SMS * 8);
  const float inv_count = 1.f / (float)((int64_t)batch * hw);
  uint4* outp = reinterpret_cast<uint4*>(dy_packed);
  const int64_t plane_vecs = (int64_t)batch * c8n * hw;
  cudaStream_t st = (cudaStream_t)stream;
#define MNB_BWD_PACK(V)                                                                                                      \
  pk::bn_sign_bwd_pack_kernel<V><<<blocks, 256, 0, st>>>(g, pass_bits, x, batch, channels, hw, out_shuffle_groups, inv_count, \
                                                         mean, invstd, gamma, dgamma, dbeta, ch_scale, terms, dx, outp, plane_vecs)
  if (vec == 4) MNB_BWD_PACK(4); else if (vec == 2) MNB_BWD_PACK(2); else MNB_BWD_PACK(1);
#undef MNB_BWD_PACK
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_bn_sign_pool_bwd_pack(const float* g, const uint32_t* pass_bits, const uint8_t* argmax, const float* x,
                                         int32_t batch, int32_t channels, int32_t H, int32_t W, const float* mean,
                                         const float* invstd, const float* gamma, const float* dgamma, const float* dbeta,
                                         int32_t out_shuffle_groups, const float* ch_scale, int32_t terms, void* dy_packed,
                                         mnb_stream_t stream) {
  MNB_REQUIRE(g && pass_bits && argmax && x && mean && invstd && gamma && dgamma && dbeta && dy_packed, "NULL bn_sign_pool_bwd_pack pointer");
  MNB_REQUIRE(batch > 0 && channels > 0 && H > 0 && W > 0 && terms >= 1 && terms <= 3, "bad bn_sign_pool_bwd_pack arguments");
  MNB_REQUIRE(out_shuffle_groups >= 1 && channels % out_shuffle_groups == 0, "shuffle groups %d do not divide %d channels",
              out_shuffle_groups, channels);
  if ((H & 1) || (W & 7) || channels % 8 || (int64_t)batch * channels * H * W >= (1ll << 31) ||
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy_packed)) & 15) || (reinterpret_cast<uintptr_t>(g) & 7))
    return mnb_fail(MNB_E_UNSUPPORTED, "packed pooled BatchNorm backward needs even H, W %% 8 == 0, channels %% 8 == 0, aligned tensors");
  const int c8n = channels / 8;
  const int64_t total = (int64_t)batch * c8n * (H / 2) * (W / 4);
  const int blocks = (int)std::min<int64_t>(mnb_ceil_div(total, 256), (int64_t)MNB_NUM_SMS * 8);
  pk::bn_sign_pool_bwd_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float2*>(g), reinterpret_cast<const uchar2*>(argmax), reinterpret_cast<const uint8_t*>(pass_bits),
      reinterpret_cast<const float4*>(x), batch, channels, H, W / 4, out_shuffle_groups, 1.f / (float)((int64_t)batch * H * W), mean,
      invstd, gamma, dgamma, dbeta, ch_scale, terms, reinterpret_cast<uint4*>(dy_packed), (int64_t)batch * c8n * H * W);
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_quant_add_pack_fwd(const float* a, const float* b, int32_t batch, int32_t channels, int32_t h, int32_t w,
                                      const mnb_act_qparams* qp, int32_t relu, float* out, const mnb_pk_post* post,
                                      mnb_stream_t stream) {
  MNB_REQUIRE(a && b && qp && out && post && post->q && post->out_pk, "NULL quant_add_pack pointer");
  MNB_REQUIRE(batch > 0 && channels > 0 && h > 0 && w > 0, "bad quant_add_pack shape");
  MNB_REQUIRE(qp->mode == MNB_ACT_DOREFA || qp->mode == MNB_ACT_IAO, "QuantAdd takes a DoReFa or IAO quantizer");
  MNB_REQUIRE(post->q->mode == MNB_ACT_DOREFA || post->q->mode == MNB_ACT_IAO, "consumer quantizer must be DoReFa or IAO");
  MNB_REQUIRE(post->q->bits >= 2 && post->q->bits <= 8 && qp->bits >= 2 && qp->bits <= 8, "quantizers must have 2..8 bits");
  MNB_REQUIRE((reinterpret_cast<uintptr_t>(post->out_pk) & 15) == 0, "packed tensor must be 16-byte aligned");
  if (post->phase_split) MNB_REQUIRE(((h | w) & 1) == 0, "phase split needs even H and W");
  const int C8 = (channels + 7) / 8;
  const int hw = h * w;
  const int tx = std::min(256, (hw + 31) / 32 * 32), ty = 256 / tx;
  const int planes = batch * C8, gy = (planes + ty - 1) / ty;
  const int bx = std::max(1, std::min((hw + tx - 1) / tx, std::max(1, (MNB_NUM_SMS * 16) / std::max(1, gy))));
  if (gy > 65535) return mnb_fail(MNB_E_UNSUPPORTED, "quant_add_pack: %d (image, octet) planes exceed the grid", planes);
  pk::quant_add_pack_kernel<<<dim3(bx, gy), dim3(tx, ty), 0, (cudaStream_t)stream>>>(
      a, b, batch, channels, h, w, C8, *qp, relu, out, *post->q, post->relu, post->phase_split,
      reinterpret_cast<uint4*>(post->out_pk));
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_bn_relu_quant_pack_fwd(const float* x, int32_t batch, int32_t channels, int32_t hw, const float* mean,
                                          const float* invstd, const float* gamma, const float* beta,
                                          const mnb_act_qparams* qp, int32_t out_shuffle_groups, void* x_packed,
                                          uint32_t* pass_bits, mnb_stream_t stream) {
  MNB_REQUIRE(x && mean && invstd && gamma && beta && qp && x_packed && pass_bits, "NULL bn_relu_quant_pack pointer");
  MNB_REQUIRE(batch > 0 && channels > 0 && hw > 0, "bad bn_relu_quant_pack shape");
  MNB_REQUIRE(qp->mode == MNB_ACT_DOREFA && qp->bits >= 2 && qp->bits <= 8, "the fused producer takes a DoReFa quantizer with 2..8 bits");
  MNB_REQUIRE(out_shuffle_groups >= 1 && channels % out_shuffle_groups == 0, "shuffle groups %d do not divide %d channels",
              out_shuffle_groups, channels);
  if (channels % 8 || hw % 32 || (reinterpret_cast<uintptr_t>(x_packed) & 15))
    return mnb_fail(MNB_E_UNSUPPORTED, "fused producer needs channels %% 8 == 0, H*W %% 32 == 0, 16-byte aligned output");
  const int64_t warps = (int64_t)batch * (channels / 8) * (hw / 32);
  const int blocks = (int)std::min<int64_t>(mnb_ceil_div(warps, 8), (int64_t)MNB_NUM_SMS * 16);
  pk::bn_relu_quant_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, batch, channels, hw, out_shuffle_groups, mean, invstd,
                                                                       gamma, beta, *qp, pass_bits,
                                                                       reinterpret_cast<uint4*>(x_packed));
  MNB_LAUNCHED(1);
  return 0;
}

// host only: out[16] = {wimg_bytes(lo), wimg_bytes(hi), Nt, n_ntiles, MT, CC, chunks, nstage, smem_bytes, tmem_cols, TH, TB,
//                       BW, n_mtiles, n_items, ny}
extern "C" int mnb_pk_conv_plan(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w, int32_t* out16) {
  pk::Plan p;
  if (int e = pk::make_plan(s, mode, terms_a, terms_w, p)) return e;
  if (out16) {
    const int v[16] = {(int)(p.wimg_bytes & 0x7fffffff), (int)(p.wimg_bytes >> 31), p.Nt, p.n_ntiles, p.MT, p.CC, p.chunks, p.nstage,
                       p.smem_bytes, p.tmem_cols, p.TH, p.TB, p.BW, p.n_mtiles, p.n_items, p.ny};
    for (int i = 0; i < 16; ++i) out16[i] = v[i];
  }
  return 0;
}

extern "C" int64_t mnb_pk_wimage_bytes(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w) {
  pk::Plan p;
  if (pk::make_plan(s, mode, terms_a, terms_w, p)) return -1;
  return p.wimg_bytes;
}

extern "C" int mnb_pk_pack_weight(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w,
                                  const int16_t* w_int, const float* w_f32, const float* kzero, void* w_img,
                                  mnb_stream_t stream) {
  MNB_REQUIRE((w_int != nullptr) != (w_f32 != nullptr), "exactly one of w_int / w_f32");
  MNB_REQUIRE(w_img && (reinterpret_cast<uintptr_t>(w_img) & 15) == 0, "weight image must be 16-byte aligned");
  pk::PackWParams pp;
  if (int e = pk::make_plan(s, mode, terms_a, terms_w, pp.pl)) return e;
  pp.w_int = w_int; pp.w_f32 = w_f32; pp.kzero = kzero;
  pp.cin_g = s->in_c / s->groups; pp.cout_g = s->out_c / s->groups;
  const int64_t vecs = pp.pl.wimg_bytes / 16;
  const int blocks = (int)std::min<int64_t>((vecs + 255) / 256, (int64_t)MNB_NUM_SMS * 8);
  pk::pack_weight_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(pp, reinterpret_cast<uint4*>(w_img));
  MNB_LAUNCHED(1);
  return 0;
}

static int pk_conv_impl(const mnb_conv_shape* s, int32_t mode, const void* a_pk, int32_t terms_a, const void* w_img,
                        int32_t terms_w, const float* n_scale, const float* a_scale, float a_scale_const,
                        const float* bias, const uint8_t* bits8, float gain, float* out, const mnb_pk_post* post,
                        int32_t* err_flag, mnb_stream_t stream) {
  using namespace pk;
  MNB_REQUIRE(s && a_pk && w_img && (out || post) && err_flag, "NULL pk_conv pointer");
  Plan pl;
  if (int e = make_plan(s, mode, terms_a, terms_w, pl)) return e;
  if (post) {
    MNB_REQUIRE(mode == 0 && !bits8, "pk conv: a fused consumer is a forward-only (inference) option");
    MNB_REQUIRE(post->q && post->out_pk && (reinterpret_cast<uintptr_t>(post->out_pk) & 15) == 0, "pk conv: consumer plane / quantizer");
    MNB_REQUIRE(post->q->mode == MNB_ACT_DOREFA || post->q->mode == MNB_ACT_IAO, "pk conv: consumer quantizer must be DoReFa or IAO");
    MNB_REQUIRE(post->q->bits >= 2 && post->q->bits <= 8, "pk conv: consumer levels must fit one bf16 piece (2..8 bits)");
    if (pl.G > 1 && (pl.ng % 8)) return unsupported("fused consumer of a grouped conv needs channels per group % 8 == 0");
    if (post->phase_split && ((pl.OH | pl.OW) & 1)) return unsupported("stride-2 consumer of an odd-sized plane");
  }
  if (bits8 && pl.G > 1 && (pl.ng % 8)) return unsupported("STE mask of a grouped conv needs channels per group % 8 == 0");
  static ConvParams p;   // large POD: filled per call (single host thread per process)
  memset(&p, 0, sizeof(p));
  ConvParams::Mma& m = p.m;
  m.n_items = pl.n_items; m.chunks = pl.chunks; m.ksteps = pl.ksteps; m.MT = pl.MT; m.Nt = pl.Nt; m.npairs = pl.npairs;
  m.st_mask = pl.nstage - 1; m.st_log2 = pl.st_log2; m.stage16 = pl.stage_bytes >> 4;
  m.a_term16 = pl.a_bytes >> 4; m.a_mt16 = (pl.TA * pl.a_bytes) >> 4; m.a_k16 = 2 * pl.npos;
  m.b_off16 = pl.b_off >> 4; m.b_tap16 = (pl.CC / 8) * pl.Nt; m.b_k16 = 2 * pl.Nt;
  m.idesc = tc::make_idesc(1, 1, 1, 128, (uint32_t)pl.Nt);
  m.a_lbo = (uint32_t)pl.npos * 16u; m.b_lbo = (uint32_t)pl.Nt * 16u;
  m.seg_len = (uint32_t)pl.seg_len;
  int nprog = 0;
  uint32_t* prog = reinterpret_cast<uint32_t*>(m.prog4);
  for (int i = 0; i < MAXPROG; ++i) prog[i] = 0xffffffffu;    // padding words: no MMA
  for (int y = 0; y < pl.ny; ++y) {
    m.ntmpl[y] = pl.ntmpl[y]; p.ntmpl[y] = pl.ntmpl[y];
    for (int t = 0; t < pl.ntmpl[y]; ++t) {
      const Tmpl& tp = pl.tmpl[y][t];
      p.tmpl_kph[y][t] = tp.kph; p.tmpl_blk_off[y][t] = tp.blk_off; p.tmpl_blk_bytes[y][t] = tp.blk_bytes;
      const int cnt = tp.ntap * pl.npairs * pl.ksteps;
      nprog = (nprog + 3) & ~3;                       // every template starts on a group of four words
      m.tmpl_begin[y][t] = (uint16_t)(nprog / 4); m.tmpl_cnt[y][t] = (uint16_t)((cnt + 3) / 4);
      if (nprog + ((cnt + 3) & ~3) > MAXPROG) return unsupported("MMA program longer than 512 entries");
      for (int pr = 0; pr < pl.npairs; ++pr)          // piece pairs outermost: small products first
        for (int i = 0; i < tp.ntap; ++i)
          for (int j = 0; j < pl.ksteps; ++j) {
            const uint32_t a16 = (uint32_t)pl.tap_aoff[y][tp.tap0 + i] + (uint32_t)pl.pair_a[pr] * m.a_term16 + (uint32_t)j * m.a_k16;
            const uint32_t b16 = (uint32_t)i * m.b_tap16 + (uint32_t)pl.pair_b[pr] * (uint32_t)tp.ntap * m.b_tap16 + (uint32_t)j * m.b_k16;
            if (a16 > 0xffffu || b16 > 0xffffu) return mnb_fail(MNB_E_ARG, "pk conv: MMA program offset overflow");
            prog[nprog++] = a16 | (b16 << 16);
          }
    }
    p.img_bytes[y] = pl.img_bytes[y]; p.y_off[y] = pl.y_off[y];
    p.zero_y[y] = pl.ntap[y] == 0;
    const int nstages = pl.ntmpl[y] * pl.chunks;
    p.nseg[y] = nstages == 0 ? 1 : (int)(((int64_t)nstages + pl.seg_len - 1) / pl.seg_len);
  }
  p.n_items = pl.n_items; p.n_ntiles = pl.n_ntiles; p.G = pl.G; p.MT = pl.MT; p.TA = pl.TA; p.chunks = pl.chunks;
  p.CC8 = pl.CC / 8; p.C8A = pl.C8A; p.kg8 = pl.kg / 8; p.stage_bytes = pl.stage_bytes; p.a_bytes = pl.a_bytes;
  p.a_box_bytes = pl.a_box_bytes; p.b_off = pl.b_off; p.st_mask = pl.nstage - 1; p.st_log2 = pl.st_log2;
  p.Wt = pl.Wt; p.TH = pl.TH; p.TB = pl.TB; p.wlo = pl.wlo; p.hlo = pl.hlo; p.col_tiles = pl.col_tiles; p.row_tiles = pl.row_tiles;
  p.n_mtiles = pl.n_mtiles;
  p.w_img = reinterpret_cast<const uint8_t*>(w_img);
  p.B = pl.B; p.THH = pl.THH; p.BW = pl.BW; p.OHr = pl.OHr; p.OWr = pl.OWr; p.OH = pl.OH; p.OW = pl.OW; p.omul = pl.omul; p.ny = pl.ny;
  p.ng = pl.ng; p.Nt = pl.Nt; p.NOUT = pl.NOUT; p.C8O = (pl.NOUT + 7) / 8; p.smem_bytes = pl.smem_bytes; p.tmem_cols = pl.tmem_cols;
  p.mode = mode;
  p.n_scale = n_scale; p.a_scale = a_scale; p.a_scale_const = a_scale_const; p.bias = bias; p.bits8 = bits8; p.gain = gain;
  p.out = out; p.err = err_flag;
  if (post) {
    p.post_out = reinterpret_cast<uint4*>(post->out_pk); p.post_q = *post->q; p.post_relu = post->relu; p.post_split = post->phase_split;
  }
  { static const int dbg = [] { const char* e = getenv("MNB_PK_DEBUG"); return e ? atoi(e) : 0; }(); p.dbg = dbg; }
  CUtensorMap tm[3];
  const int C8tot = pl.nkph * pl.C8A;
  const int64_t plane_bytes = (int64_t)pl.B * C8tot * pl.HA * pl.WA * 16;
  for (int t = 0; t < 3; ++t) {
    const int tt = t < pl.TA ? t : 0;
    if (int e = make_pk_tmap(&tm[t], a_pk, plane_bytes, tt, pl.B, C8tot, pl.HA, pl.WA, pl.BW, pl.THH, pl.TB, pl.CC / 8)) return e;
  }
  if (pl.n_items >= (1 << 22) || pl.n_mtiles >= (1 << 22))     // FastDiv's exact range (fp32 reciprocal + one correction step)
    return mnb_fail(MNB_E_UNSUPPORTED, "pk conv: %d work items / %d M tiles exceed the index arithmetic of the kernel", pl.n_items, pl.n_mtiles);
  const int gx = std::max(1, std::min(pl.n_items, MNB_NUM_SMS / pl.ny));
  if (pl.segmented) {
    if (pl.MT * pl.Nt > 128) return mnb_fail(MNB_E_ARG, "pk conv: segmented plan with Nt %d, MT %d", pl.Nt, pl.MT);
    if (int e = set_max_smem(pk_conv_kernel<true>, kSmemBudget)) return e;
    pk_conv_kernel<true><<<dim3(gx, pl.ny), ConvCfg<true>::THREADS, pl.smem_bytes, (cudaStream_t)stream>>>(tm[0], tm[1], tm[2], p);
  } else {
    if (int e = set_max_smem(pk_conv_kernel<false>, kSmemBudget)) return e;
    pk_conv_kernel<false><<<dim3(gx, pl.ny), ConvCfg<false>::THREADS, pl.smem_bytes, (cudaStream_t)stream>>>(tm[0], tm[1], tm[2], p);
  }
  MNB_LAUNCHED(1);
  return 0;
}

extern "C" int mnb_pk_conv(const mnb_conv_shape* s, int32_t mode, const void* a_pk, int32_t terms_a, const void* w_img,
                           int32_t terms_w, const float* n_scale, const float* a_scale, float a_scale_const,
                           const float* bias, const uint8_t* bits8, float gain, float* out, int32_t* err_flag,
                           mnb_stream_t stream) {
  MNB_REQUIRE(out, "NULL pk_conv output");
  return pk_conv_impl(s, mode, a_pk, terms_a, w_img, terms_w, n_scale, a_scale, a_scale_const, bias, bits8, gain, out, nullptr,
                      err_flag, stream);
}

extern "C" int mnb_pk_conv_post(const mnb_conv_shape* s, const void* a_pk, int32_t terms_a, const void* w_img, int32_t terms_w,
                                const float* n_scale, const float* a_scale, float a_scale_const, const float* bias,
                                float* out, const mnb_pk_post* post, int32_t* err_flag, mnb_stream_t stream) {
  MNB_REQUIRE(post, "NULL consumer description");
  return pk_conv_impl(s, 0, a_pk, terms_a, w_img, terms_w, n_scale, a_scale, a_scale_const, bias, nullptr, 1.f, out, post,
                      err_flag, stream);
}

extern "C" int64_t mnb_pk_wgrad_scratch_bytes(const mnb_conv_shape* s, int32_t terms_dy, int32_t terms_x) {
  pk::WgPlan p;
  if (pk::make_wg_plan(s, terms_dy, terms_x, p)) return -1;
  return p.partial_floats * 4;
}

// dw[k][c][r][s] = mul(k) * sum_{b,p,q} dy[b,k,p,q] * x[b,c,p*st+r-pad, q*st+s-pad];  mul(k) = a_scale[0] / kdiv[k]
// (a_scale: activation scale when x_pk holds integer levels; kdiv: the per-channel factor dy_pk was pre-multiplied with)
extern "C" int mnb_pk_wgrad(const mnb_conv_shape* s, const void* dy_pk, int32_t terms_dy, const void* x_pk, int32_t terms_x,
                            const float* a_scale, const float* kdiv, float* dw, void* scratch, int32_t* err_flag,
                            mnb_stream_t stream) {
  using namespace pk;
  MNB_REQUIRE(s && dy_pk && x_pk && dw && scratch && err_flag, "NULL pk_wgrad pointer");
  WgPlan pl;
  if (int e = make_wg_plan(s, terms_dy, terms_x, pl)) return e;
  static WgParams p;
  memset(&p, 0, sizeof(p));
  WgParams::Mma& m = p.m;
  m.stg_per_split = pl.stg_per_split; m.nstg_total = pl.nstg_total; m.NI = pl.NI; m.ksteps = pl.rows_dy / 16; m.ntap = pl.ntap;
  m.Nc = pl.Nc; m.tpg = pl.tpg; m.n_tg = pl.n_tg; m.npairs = pl.npairs; m.st_mask = pl.nstage - 1; m.st_log2 = pl.st_log2; m.stage16 = pl.stage_bytes >> 4;
  m.sub16 = pl.sub_bytes >> 4; m.dy_term16 = pl.dy_bytes >> 4; m.x_off16 = (pl.TA * pl.dy_bytes) >> 4;
  m.x_term16 = (pl.nkph_used * pl.x_bytes) >> 4; m.x_kph16 = pl.x_bytes >> 4;
  m.idesc = tc::make_idesc_major(1, 1, 1, 128, (uint32_t)pl.Nc, 1, 1);
  m.dy_sbo = (uint32_t)pl.rows_dy * 16u; m.x_sbo = (uint32_t)pl.rows_x * 16u; m.nsub = pl.nsub;
  for (int i = 0; i < pl.npairs; ++i) { m.pair_a16[i] = pl.pair_a[i] * m.dy_term16; m.pair_b16[i] = pl.pair_b[i] * m.x_term16; }
  {
    m.g4 = (uint32_t)ceil_div(pl.tpg, 4);
    if ((size_t)pl.npairs * pl.n_tg * m.g4 > sizeof(m.progb4) / sizeof(uint4)) return unsupported("wgrad issue program too long");
    uint32_t* prog = reinterpret_cast<uint32_t*>(m.progb4);
    for (size_t i = 0; i < sizeof(m.progb4) / 4; ++i) prog[i] = 0xffffffffu;
    for (int i = 0; i < pl.npairs; ++i)
      for (int tg = 0; tg < pl.n_tg; ++tg)
        for (int tt = 0; tt < pl.tpg && tg * pl.tpg + tt < pl.ntap; ++tt) {
          const int t = tg * pl.tpg + tt;
          prog[((size_t)(i * pl.n_tg + tg) * m.g4) * 4 + tt] = m.pair_b16[i] + pl.kph_slot[pl.tap_kph[t]] * m.x_kph16 + pl.tap_off[t];
        }
  }
  p.G = pl.G; p.n_ktiles = pl.n_ktiles; p.n_ctiles = pl.n_ctiles; p.n_tg = pl.n_tg; p.tpg = pl.tpg; p.splits = pl.splits; p.stg_per_split = pl.stg_per_split;
  p.nstg_total = pl.nstg_total; p.NI = pl.NI; p.nsub = pl.nsub; p.row_tiles = pl.row_tiles; p.TA = pl.TA; p.TX = pl.TX;
  p.nkph_used = pl.nkph_used;
  for (int i = 0; i < 4; ++i) p.kph_used[i] = pl.kph_used[i];
  p.K8 = pl.K8; p.C8X = pl.C8X; p.cout_g8 = pl.cout_g / 8; p.cin_g8 = pl.cin_g / 8; p.Nc8 = pl.Nc / 8; p.TH = pl.TH; p.hlo = pl.hlo;
  p.wlo = pl.wlo; p.stage_bytes = pl.stage_bytes; p.sub_bytes = pl.sub_bytes; p.dy_bytes = pl.dy_bytes; p.x_bytes = pl.x_bytes;
  p.dy_box_bytes = pl.dy_box_bytes; p.x_box_bytes = pl.x_box_bytes; p.st_mask = pl.nstage - 1; p.st_log2 = pl.st_log2;
  p.smem_bytes = pl.smem_bytes; p.tmem_cols = pl.tmem_cols; p.ntap = pl.ntap; p.Nc = pl.Nc; p.cout_g = pl.cout_g; p.cin_g = pl.cin_g;
  p.partial = reinterpret_cast<float*>(scratch); p.err = err_flag;
  CUtensorMap tdy[3], tx[3];
  const int64_t dy_plane = (int64_t)pl.B * pl.K8 * pl.P * pl.Q * 16;
  const int C8tot = pl.nkph * pl.C8X;
  const int64_t x_plane = (int64_t)pl.B * C8tot * pl.HX * pl.WX * 16;
  for (int t = 0; t < 3; ++t) {
    if (int e = make_pk_tmap(&tdy[t], dy_pk, dy_plane, t < pl.TA ? t : 0, pl.B, pl.K8, pl.P, pl.Q, pl.BW, pl.TH, 1, 16)) return e;
    if (int e = make_pk_tmap(&tx[t], x_pk, x_plane, t < pl.TX ? t : 0, pl.B, C8tot, pl.HX, pl.WX, pl.BW, pl.THH, 1, pl.Nc / 8)) return e;
  }
  if (int e = set_max_smem(pk_wgrad_kernel, kSmemBudget)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  pk_wgrad_kernel<<<dim3(pl.G * pl.n_ktiles * pl.n_ctiles * pl.n_tg, pl.splits), NTHREADS, pl.smem_bytes, st>>>(tdy[0], tdy[1], tdy[2], tx[0],
                                                                                                      tx[1], tx[2], p);
  {
    const int cout_o = pl.cout_g / pl.gm, cin_o = pl.cin_g / pl.gm;     // channels per original group
    const dim3 rgrid(cin_o * pl.ntap, (cout_o + 127) / 128, pl.G * pl.gm);
    wg_reduce_kernel<<<rgrid, 128, 0, st>>>(p.partial, pl.splits, pl.G, pl.gm, pl.n_ktiles, pl.n_ctiles, pl.ntap, pl.Nc, cout_o,
                                            cin_o, a_scale, kdiv, dw);
  }
  MNB_LAUNCHED(2);
  return 0;
}
