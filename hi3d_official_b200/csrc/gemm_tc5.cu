// Implicit-GEMM engine, Blackwell-native variant: TMA (cp.async.bulk.tensor) operand staging into
// SWIZZLE_128B shared tiles, tcgen05.mma (UTCHMMA, cta_group::1, M=128) with fp32 accumulators in TMEM,
// tcgen05.ld epilogue.  Same contract as hi3d_gemm (include/hi3d_b200.h); geometries this engine does not
// cover (stride-2 / upsample-fused convs, odd tile shapes, N < 32) are forwarded to the mma.sync engine.
//
// Persistent kernel: one CTA per SM walks output tiles (n-tile fastest, so the CTAs running together share the
// same A rows through L2).  A tile is 128 x BN with BN a runtime multiple of 32 (<= 256) chosen so that N is
// covered with the least padding (N=320 -> 2 x 160, N=960 -> 5 x 192, ...).  The 128 rows of a tile are
//   PLAIN    : 128 consecutive rows
//   CONV2D   : a (tn images) x (th rows) x (tw columns) patch, tn*th*tw = 128 -- the 3x3 taps are the same TMA box
//              shifted by (dy, dx) and the zero padding is TMA out-of-bounds fill
//   TEMPORAL : (tf frames) x (ts pixels), tf*ts = 128 -- the temporal taps shift the frame coordinate of a
//              [C, HW, T, B] view; clip boundaries zero-fill by OOB.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2..9 = epilogue (two warps per TMEM lane quarter, alternating 32-column chunks).  Two accumulator
// buffers (TMEM columns [0,256) and [256,512)) let the epilogue of tile i overlap the main loop of tile i+1.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tc5.cuh"

namespace hi3d {
int validate_gemm(const hi3d_gemm_params* p, const char* who);

constexpr int T5_BM = 128;
constexpr int T5_BK = 64;
constexpr int T5_EPI_WARPS = 8;
constexpr int T5_THREADS = 64 + 32 * T5_EPI_WARPS;
constexpr int T5_MAX_MAPS = 4;
constexpr int T5_MAX_STAGES = 8;
constexpr int T5_A_BYTES = T5_BM * 128;
constexpr int T5_SMEM_BUDGET = 192 * 1024;
constexpr int T5_SCR_BYTES = 32 * 80;                  // per-epilogue-warp transpose scratch

struct T5Seg {
  int map;       // index into amap[]
  int c_off, C;  // channel range
  int dy, dx, dt;
};

struct T5Params {
  CUtensorMap bmap;
  CUtensorMap amap[T5_MAX_MAPS];
  T5Seg seg[HI3D_MAX_SEGS];
  int nseg;
  int M, N, K, mode;
  int BN, stages, n_tiles, total_tiles;
  int dbg;   // HI3D_TC5_DBG bit mask for bottleneck experiments: 1 skip stores, 2 skip residual/blend/rowbias loads, 4 skip TMEM loads, 8 skip MMA, 16 skip A loads, 32 skip B loads
  // tile -> rows
  int tw, th, tn;      // CONV2D patch (PLAIN: tw = 128, th = tn = 1; TEMPORAL: tw = ts, th = tf)
  int Wo, Ho, Nimg;    // CONV2D: output W, H, images.  TEMPORAL: Wo = HW, Ho = T, Nimg = B
  int tiles_x, tiles_y;  // tiles along W and H (CONV2D) / along HW and T (TEMPORAL)
  int cstride;           // CONV2D input stride (1 | 2): TMA element strides, box origin = tile origin * cstride + tap
  int out_up, out_py, out_px;   // parity-class output mapping (see hi3d_gemm_params::out_up)
  int t_off;                    // TEMPORAL: frame offset of output frame 0 inside the (haloed) source clip
  // epilogue
  const float* bias;
  const __half* rowbias;
  int rb_div, rb_mod, rb_ld, act;
  const __half* residual;
  int res_ld;
  const __half* blend_x;
  int blend_ld;
  float alpha;
  __half* out;
  int out_ld;
  // GroupNorm statistics of the output (hi3d_gemm_params::gn_stats), added to the global table from the epilogue registers
  float* gn_stats;
  int gn_unit, gn_rows, gn_units, gn_nimg;   // channels per unit, GEMM-grid rows per image, units per image (N / unit), images
  int gelu_poly;                             // GEGLU gate: 1 = MUFU-free polynomial erf (gelu_poly2), 0 = Abramowitz-Stegun form
  // deterministic statistics (EPI_*_GN_DET): slot table [image][parity class][32-row block of the image][octet][4]
  float* gn_part;
  int gn_bpi;                                // 32-row blocks per image and parity class (gn_rows / 32)
};

// gelu(x) = 0.5 x (1 + erf(x / sqrt 2)) with erf from Abramowitz-Stegun 7.1.26 (|err| < 1.5e-7 + MUFU error, far
// below the fp16 rounding of the GEGLU output): 2 MUFU + ~13 FMA-class instructions per value.
HI3D_DEVINL float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
HI3D_DEVINL float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
HI3D_DEVINL float gelu_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float t = rcp_approx(fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  const float ex = ex2_approx(z * z * -1.4426950408889634f);
  const float e = copysignf(fmaf(-p, ex, 1.0f), x);
  const float hx = 0.5f * x;
  return fmaf(hx, e, hx);
}

// Two gates at once on the packed-fp32 pipe (FFMA2 / FMUL2): the GEGLU epilogue is instruction-issue bound, not
// MUFU bound, and this form needs ~10 issue slots per gate instead of ~17.
HI3D_DEVINL float2 gelu_fast2(float2 x) {
  const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 z = __fmul2_rn(ax, make_float2(0.70710678118654752f, 0.70710678118654752f));
  const float2 den = __ffma2_rn(make_float2(0.3275911f, 0.3275911f), z, make_float2(1.0f, 1.0f));
  const float2 t = make_float2(rcp_approx(den.x), rcp_approx(den.y));
  float2 p = __ffma2_rn(make_float2(1.061405429f, 1.061405429f), t, make_float2(-1.453152027f, -1.453152027f));
  p = __ffma2_rn(p, t, make_float2(1.421413741f, 1.421413741f));
  p = __ffma2_rn(p, t, make_float2(-0.284496736f, -0.284496736f));
  p = __ffma2_rn(p, t, make_float2(0.254829592f, 0.254829592f));
  p = __fmul2_rn(p, t);
  const float2 arg = __fmul2_rn(__fmul2_rn(z, z), make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 ex = make_float2(ex2_approx(arg.x), ex2_approx(arg.y));
  const float2 em = __ffma2_rn(p, ex, make_float2(-1.0f, -1.0f));          // -(erf|z|), <= 0
  const float2 e = make_float2(copysignf(em.x, x.x), copysignf(em.y, x.y));  // erf(x / sqrt 2)
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, e, hx);
}

// The same gate without the MUFU pipe: erf(z) = z P(w), w = 2 z^2 / Z^2 - 1, on |z| <= Z = 3.4 (weighted least-squares fit
// of degree 10 in w; beyond Z the clamp makes erf = +-(1 - 1.5e-6)).  |gelu error| <= 5e-6 over all x (checked in fp32
// against the exact function, tools/gelu_fit.py) -- two orders below the fp16 rounding of the GEGLU output.  The clamp is
// a saturating FMA: t = sat(z / 2Z + 1/2), z_c = 2Z t - Z.  18 issue slots per pair of gates, none of them MUFU
// (gelu_fast2: 21 including 4 MUFU).  Measured on the GEGLU C = 320 GEMM: 1.029 ms with either gate -- the epilogue is bound by
// dependency and shared-memory latency spread over the whole chunk (profiles/r02_ncu_gemm_epilogue_notes.txt), not by the
// gate's arithmetic -- so gelu_fast2 stays the default and this one is selectable (HI3D_TC5_GELU=poly).
HI3D_DEVINL float fma_sat(float a, float b, float c) {
  float r;
  asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
HI3D_DEVINL float2 gelu_poly2(float2 x) {
  constexpr float Z = 3.4f;
  const float kz = 0.70710678118654752f * 0.5f / Z;
  const float2 t = make_float2(fma_sat(x.x, kz, 0.5f), fma_sat(x.y, kz, 0.5f));
  const float2 zc = __ffma2_rn(t, make_float2(2.f * Z, 2.f * Z), make_float2(-Z, -Z));
  const float2 zs = __fmul2_rn(zc, make_float2(2.f / (Z * Z), 2.f / (Z * Z)));
  const float2 w = __ffma2_rn(zs, zc, make_float2(-1.f, -1.f));
  float2 p = __ffma2_rn(make_float2(0.004088203888386488f, 0.004088203888386488f), w, make_float2(-0.012048999778926373f, -0.012048999778926373f));
  p = __ffma2_rn(p, w, make_float2(0.015636751428246498f, 0.015636751428246498f));
  p = __ffma2_rn(p, w, make_float2(-0.021256500855088234f, -0.021256500855088234f));
  p = __ffma2_rn(p, w, make_float2(0.03925583139061928f, 0.03925583139061928f));
  p = __ffma2_rn(p, w, make_float2(-0.06293924897909164f, -0.06293924897909164f));
  p = __ffma2_rn(p, w, make_float2(0.08708704262971878f, 0.08708704262971878f));
  p = __ffma2_rn(p, w, make_float2(-0.11474799364805222f, -0.11474799364805222f));
  p = __ffma2_rn(p, w, make_float2(0.14947132766246796f, 0.14947132766246796f));
  p = __ffma2_rn(p, w, make_float2(-0.20609460771083832f, -0.20609460771083832f));
  p = __ffma2_rn(p, w, make_float2(0.41566580533981323f, 0.41566580533981323f));
  const float2 e = __fmul2_rn(zc, p);                      // erf(x / sqrt 2)
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, e, hx);
}

struct T5Tile {
  int x0, y0, z0;   // TMA origin coordinates (CONV2D: x, y, image; TEMPORAL: pixel, frame, clip)
};

HI3D_DEVINL T5Tile t5_origin(const T5Params& p, int mt) {
  T5Tile t{0, 0, 0};
  if (p.mode != HI3D_ROWS_PLAIN) {
    const int tx = mt % p.tiles_x, rest = mt / p.tiles_x;
    t.x0 = tx * p.tw;
    t.y0 = (rest % p.tiles_y) * p.th;
    t.z0 = (rest / p.tiles_y) * p.tn;
  }
  return t;
}
// tile-local row -> global output row (or -1)
HI3D_DEVINL long long t5_row(const T5Params& p, int mt, const T5Tile& o, int r) {
  if (p.mode == HI3D_ROWS_PLAIN) {
    const long long m = (long long)mt * T5_BM + r;
    return m < p.M ? m : -1;
  }
  const int x = o.x0 + r % p.tw;
  const int y = o.y0 + (r / p.tw) % p.th;
  const int n = o.z0 + r / (p.tw * p.th);
  if (x >= p.Wo || y >= p.Ho || n >= p.Nimg) return -1;
  return ((long long)n * p.Ho + y) * p.Wo + x;
}

// base row (row of the Ho x Wo GEMM grid) -> row of the output tensor
HI3D_DEVINL long long t5_map(const T5Params& p, long long m) {
  if (!p.out_up || m < 0) return m;
  const int hw = p.Ho * p.Wo;
  const int n = (int)(m / hw), rem = (int)(m - (long long)n * hw);
  const int y = rem / p.Wo, x = rem - y * p.Wo;
  return ((long long)n * 2 * p.Ho + 2 * y + p.out_py) * (2 * p.Wo) + 2 * x + p.out_px;
}

// NCTA = 2: the two CTAs of a cluster own the two 128-row halves of a 256-row tile and half of the B tile each;
// CTA 0 issues tcgen05.mma.cta_group::2 for the pair (operands are read from both CTAs' shared memory, so every B
// byte is fetched from L2 once per PAIR), each CTA runs the epilogue of its own 128 accumulator rows.
// EPI specialises the epilogue at compile time.  The generic epilogue (EPI_GENERIC: every option a run-time branch on a
// kernel parameter) was profiled at 12 % instruction-cache misses and 6 % branch stalls on the short-K GEMMs, whose epilogue
// IS the kernel (ncu source page, profiles/r02_ncu_gemm_epilogue_notes.txt): the options that cost code and branches inside the
// chunk loop -- GEGLU, residual, blend, GroupNorm statistics -- are template constants in the specialised kernels.
// The *_GN_DET variants store the statistics partials into per-warp slots instead of adding them with RED (deterministic mode,
// hi3d_gemm_tc5_det): separate instantiations, so that the default ones keep their registers and code.
enum { EPI_GENERIC = 0, EPI_GEGLU = 1, EPI_BIAS = 2, EPI_RES = 3, EPI_RESBLEND = 4, EPI_BIAS_GN = 5, EPI_RES_GN = 6, EPI_RESBLEND_GN = 7,
       EPI_BIAS_GN_DET = 8, EPI_RES_GN_DET = 9, EPI_RESBLEND_GN_DET = 10 };

// EW = epilogue warps (8 or 16).  Sixteen (four per TMEM lane quarter, every fourth 32-column chunk each) double the
// epilogue's issue slots and loads / stores in flight for the short-K GEMMs whose epilogue is the bound; the register-light
// specialisations (<= 112 registers) fit 576 threads.
template <int NCTA, int EPI, int EW>
__global__ void __launch_bounds__(64 + 32 * EW, 1) gemm_tc5_kernel(const __grid_constant__ T5Params p) {
  constexpr bool kGen = (EPI == EPI_GENERIC);
  // compile-time constants in the specialised kernels, run-time tests in the generic one
  const bool kGeglu = kGen ? (p.act == HI3D_ACT_GEGLU) : (EPI == EPI_GEGLU);
  const bool kRes = kGen ? (p.residual != nullptr) : (EPI == EPI_RES || EPI == EPI_RESBLEND || EPI == EPI_RES_GN || EPI == EPI_RESBLEND_GN ||
                                                      EPI == EPI_RES_GN_DET || EPI == EPI_RESBLEND_GN_DET);
  const bool kBlend = kGen ? (p.blend_x != nullptr) : (EPI == EPI_RESBLEND || EPI == EPI_RESBLEND_GN || EPI == EPI_RESBLEND_GN_DET);
  constexpr bool kDet = (EPI >= EPI_BIAS_GN_DET);
  const bool kSilu = kGen ? (p.act == HI3D_ACT_SILU) : false;
  const bool kGn = kGen ? (p.gn_stats != nullptr && p.act != HI3D_ACT_GEGLU) : (EPI >= EPI_BIAS_GN);
  const int kDbg = kGen ? p.dbg : 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;          // SWIZZLE_128B atoms need 1024-byte alignment
  uint8_t* smem = smem_raw + (base - raw);
  const int BN = p.BN, STAGES = p.stages;
  const uint32_t stage_bytes = T5_A_BYTES + (BN / NCTA) * 128;   // per CTA
  const uint32_t rank = (NCTA == 2) ? cluster_ctarank() : 0u;
  const int unit0 = blockIdx.x / NCTA, nunits = gridDim.x / NCTA;  // a unit = one CTA (pair); units walk (pair-)tiles
  const uint32_t bar_base = base + STAGES * stage_bytes;
  const uint32_t bar_full = bar_base;                      // STAGES x 8
  const uint32_t bar_empty = bar_base + 8 * T5_MAX_STAGES;
  const uint32_t bar_acc_full = bar_empty + 8 * T5_MAX_STAGES;   // 2 x 8
  const uint32_t bar_acc_empty = bar_acc_full + 16;              // 2 x 8
  const uint32_t tmem_slot = bar_acc_empty + 16;
  volatile uint32_t* tmem_slot_g =
      reinterpret_cast<volatile uint32_t*>(smem + STAGES * stage_bytes + 16 * T5_MAX_STAGES + 32);
  float* sbias = reinterpret_cast<float*>(smem + STAGES * stage_bytes + 16 * T5_MAX_STAGES + 64);   // [2][256]
  uint8_t* scratch = smem + STAGES * stage_bytes + 16 * T5_MAX_STAGES + 64 + 2048;                  // [EPI_WARPS][32 x 80]

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform role index
  const int KT = p.K / T5_BK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(bar_full + 8 * s, 1);        // the (leader's) expect_tx arrive; a pair counts both CTAs' bytes on CTA 0
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int b = 0; b < 2; b++) {
      mbar_init(bar_acc_full + 8 * b, 1);
      mbar_init(bar_acc_empty + 8 * b, EW * NCTA);   // pair: both CTAs' epilogue warps report to the leader
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    if (NCTA == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();   // barrier inits visible to the peer before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_g;

  if (warp == 0) {
    // ======================= TMA producer =======================
    // The whole warp walks the loop with warp-uniform values and one elected lane issues: addresses stay in uniform
    // registers.  (A lane-0-only loop made every TMA / MMA operand go through R2UR waterfall code and the two
    // single-thread issue loops -- ~600 cycles per k-block -- were the slowest part of the kernel.)
    uint32_t s = 0, ph = 0;
    const uint32_t lead_full = (NCTA == 2) ? mapa_cluster(bar_full, 0) : bar_full;   // pair: bytes count on CTA 0
    const uint32_t txb = ((kDbg & 16) ? 0u : (uint32_t)T5_A_BYTES) + ((kDbg & 32) ? 0u : (uint32_t)(BN / NCTA) * 128u);
    for (int tile = unit0; tile < p.total_tiles; tile += nunits) {
      const int mu = tile / p.n_tiles, nt = tile - mu * p.n_tiles;
      const int mt = mu * NCTA + (int)rank;
      const T5Tile o = t5_origin(p, mt);
      const int n0 = nt * BN + (int)rank * (BN / NCTA);     // pair: this CTA stages its half of the B rows
      int si = 0, so = 0;
      T5Seg sg = p.seg[0];
      const CUtensorMap* am = &p.amap[sg.map];
      for (int kt = 0; kt < KT; kt++) {
        mbar_wait(bar_empty + 8 * s, ph ^ 1);
        if (elect_one()) {
          const uint32_t sA = base + s * stage_bytes;
          const uint32_t sB = sA + T5_A_BYTES;
          const int c = sg.c_off + so;
          if (NCTA == 2) {
            // The peer does not arrive on the leader's barrier: its bytes may land before the leader arms the phase (the
            // tx-count goes negative for a moment), and a release.cluster arrive per k-block serialises the producer.
            const uint32_t full = lead_full + 8 * s;
            if (rank == 0) mbar_expect_tx(bar_full + 8 * s, 2 * txb);
            if (kDbg & 16) {
            } else if (p.mode == HI3D_ROWS_PLAIN)
              tma_load_2d_cg2(sA, am, full, c, mt * T5_BM);
            else if (p.mode == HI3D_ROWS_CONV2D)
              tma_load_4d_cg2(sA, am, full, c, o.x0 * p.cstride + sg.dx, o.y0 * p.cstride + sg.dy, o.z0);
            else
              tma_load_4d_cg2(sA, am, full, c, o.x0, o.y0 + p.t_off + sg.dt, o.z0);
            if (!(kDbg & 32)) tma_load_2d_cg2(sB, &p.bmap, full, kt * T5_BK, n0);
          } else {
            const uint32_t full = bar_full + 8 * s;
            mbar_expect_tx(full, txb);
            if (kDbg & 16) {
            } else if (p.mode == HI3D_ROWS_PLAIN)
              tma_load_2d(sA, am, full, c, mt * T5_BM);
            else if (p.mode == HI3D_ROWS_CONV2D)
              tma_load_4d(sA, am, full, c, o.x0 * p.cstride + sg.dx, o.y0 * p.cstride + sg.dy, o.z0);
            else
              tma_load_4d(sA, am, full, c, o.x0, o.y0 + p.t_off + sg.dt, o.z0);
            if (!(kDbg & 32)) tma_load_2d(sB, &p.bmap, full, kt * T5_BK, n0);
          }
        }
        __syncwarp();
        so += T5_BK;
        if (so >= sg.C && kt + 1 < KT) { si++; so = 0; sg = p.seg[si]; am = &p.amap[sg.map]; }
        if (++s == (uint32_t)STAGES) { s = 0; ph ^= 1; }
      }
    }
    if (NCTA == 2) {
      // drain: every multicast commit aimed at this CTA's empty barriers has landed before the CTA may exit
      for (int j = 0; j < STAGES; j++) {
        // slot s is the oldest outstanding one; a slot never filled keeps its initial phase and passes at once
        mbar_wait(bar_empty + 8 * s, ph ^ 1);
        if (++s == (uint32_t)STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer (pair: leader CTA only) =======================
    if (rank == 0) {
      // instruction descriptor: D = f32, A = B = f16, both K-major, N = BN, M = 128 (per CTA; 256 for the pair)
      const uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((T5_BM * NCTA) >> 4) << 24);
      const uint64_t ad0 = umma_desc_sw128(base), bd0 = umma_desc_sw128(base + T5_A_BYTES);
      const uint32_t stage16 = stage_bytes >> 4;             // descriptor address field is in 16-byte units
      uint32_t s = 0, ph = 0, at = 0;
      for (int tile = unit0; tile < p.total_tiles; tile += nunits, at++) {
        const uint32_t buf = at & 1;
        mbar_wait(bar_acc_empty + 8 * buf, ((at >> 1) & 1) ^ 1);   // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tacc = tmem_base + buf * 256;
        for (int kt = 0; kt < KT; kt++) {
          mbar_wait(bar_full + 8 * s, ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t ad = ad0 + (uint64_t)(s * stage16), bd = bd0 + (uint64_t)(s * stage16);
            if (!(kDbg & 8)) {
#pragma unroll
              for (int k = 0; k < T5_BK / 16; k++) {   // +32 bytes along K inside the 128-byte swizzle atom
                if (NCTA == 2) tc_mma_f16_cg2(tacc, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kt | k) ? 1u : 0u);
                else tc_mma_f16(tacc, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kt | k) ? 1u : 0u);
              }
            }
            // frees the smem slot (in both CTAs of a pair) when these MMAs retire
            if (NCTA == 2) tc_commit_cg2(bar_empty + 8 * s, 3); else tc_commit(bar_empty + 8 * s);
          }
          __syncwarp();
          if (++s == (uint32_t)STAGES) { s = 0; ph ^= 1; }
        }
        // accumulator complete
        if (elect_one()) {
          if (NCTA == 2) tc_commit_cg2(bar_acc_full + 8 * buf, 3); else tc_commit(bar_acc_full + 8 * buf);
        }
        __syncwarp();
      }
    }
  } else {
    // ======================= epilogue warps: T5_EPI_WARPS/4 per TMEM lane quarter =======================
    // A thread owns one accumulator row (its TMEM lane).  Global traffic is NOT issued row-per-thread (16-byte pieces
    // of 32 different rows per instruction are partial-sector writes and were 4x slower than the MMA main loop):
    // every 32 x 32 chunk goes through a per-warp shared-memory transpose so that 4 lanes cover 64 contiguous bytes of
    // one row (full 32-byte sectors) for the output stores and for the residual / blend loads alike.
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int ew = warp - 2;                     // epilogue warp index
    const int wsel = ew >> 2;                    // this warp takes 32-column chunks wsel, wsel + EPI/4, ...
    const bool geglu = kGeglu;
    const int rl = q * 32 + lane;                // tile-local row == TMEM lane
    uint8_t* scr = scratch + ew * T5_SCR_BYTES;  // 32 rows x 80 bytes (64 data + 16 pad)
    const int crow = lane >> 2, cchk = lane & 3; // coalesced pattern: rows crow + 8 i, 16-byte chunk cchk
    uint32_t at = 0;
    const uint32_t lead_acc_empty = (NCTA == 2) ? mapa_cluster(bar_acc_empty, 0) : bar_acc_empty;
    const int et = tid - 64;                     // epilogue thread index; threads 0..255 stage the bias slice
    // bias slice of the first tile; later tiles are fetched one tile ahead (a global-load latency plus a 256-thread
    // barrier per tile was on the critical path of every epilogue warp)
    if (unit0 < p.total_tiles) {
      const int nb = (unit0 % p.n_tiles) * BN + et;
      if (et < 256) sbias[et] = (p.bias != nullptr && et < BN && nb < p.N) ? __ldg(p.bias + nb) : 0.f;
    }
    const bool gn_on = kGn;

    for (int tile = unit0; tile < p.total_tiles; tile += nunits, at++) {
      const int mu = tile / p.n_tiles, nt = tile - mu * p.n_tiles;
      const int mt = mu * NCTA + (int)rank;
      const T5Tile o = t5_origin(p, mt);
      const int n0 = nt * BN;
      const long long m = t5_row(p, mt, o, rl);
      long long mrow[4];                         // global rows of the rows this lane touches in the coalesced pattern
#pragma unroll
      for (int i = 0; i < 4; i++) mrow[i] = t5_map(p, __shfl_sync(0xffffffffu, m, crow + 8 * i));
      // GroupNorm statistics: image (sample) of this warp's rows relative to the first image the tile can touch
      int gn_s0 = 0, gn_wsmp = -1, gn_srow[4] = {-1, -1, -1, -1};
      bool gn_uniform = true;
      if (gn_on) {
        if (p.mode == HI3D_ROWS_CONV2D) gn_s0 = o.z0;
        else if (p.mode == HI3D_ROWS_TEMPORAL) gn_s0 = o.z0 * p.Ho + o.y0;
        else gn_s0 = (int)(((long long)mt * T5_BM) / p.gn_rows);
        const int sl = (m >= 0) ? (int)(m / p.gn_rows) - gn_s0 : -1;
        const int smax = __reduce_max_sync(0xffffffffu, sl);
        const int smin = __reduce_min_sync(0xffffffffu, sl < 0 ? 0x7fffffff : sl);
        gn_uniform = (smax < 0) || (smin == smax);
        gn_wsmp = smax;                            // the warp's image when uniform (-1: no valid row)
#pragma unroll
        for (int i = 0; i < 4; i++) gn_srow[i] = __shfl_sync(0xffffffffu, sl, crow + 8 * i);
      }
      // deterministic mode: this warp's slot row = (image, parity class, block of the image).  The host takes this path only
      // when every warp block lies inside one image: PLAIN gn_rows % 32 == 0, CONV2D tw * th >= 32, TEMPORAL ts >= 32.
      float* gn_slot = nullptr;
      if (kDet && gn_wsmp >= 0) {
        int loc;
        if (p.mode == HI3D_ROWS_PLAIN) {
          loc = (int)((((long long)mt * T5_BM + q * 32) % p.gn_rows) / 32);
        } else {
          // blocks of one image inside a tile: CONV2D a tw x th patch, TEMPORAL ts = tw pixels of one frame
          const int bpf = ((p.mode == HI3D_ROWS_CONV2D) ? p.tw * p.th : p.tw) / 32;
          const int tx = mt % p.tiles_x, ty = (mt / p.tiles_x) % p.tiles_y;
          loc = (p.mode == HI3D_ROWS_CONV2D) ? (ty * p.tiles_x + tx) * bpf + q % bpf : tx * bpf + q % bpf;
        }
        const int npar = p.out_up ? 4 : 1, par = p.out_up ? 2 * p.out_py + p.out_px : 0;
        gn_slot = p.gn_part + ((long long)((gn_s0 + gn_wsmp) * npar + par) * p.gn_bpi + loc) * (long long)(p.N / 2);
      }
      const __half* rbp = nullptr;
      if (p.rowbias != nullptr && m >= 0) rbp = p.rowbias + (long long)((m / p.rb_div) % p.rb_mod) * p.rb_ld;
      const uint32_t buf = at & 1;
      // every epilogue warp has finished the previous tile (its bias buffer may be overwritten) and this tile's slice,
      // written during the previous tile, is visible
      asm volatile("bar.sync 1, %0;\n" ::"n"(32 * EW) : "memory");
      float bnext = 0.f;
      {
        const int tnext = tile + nunits;
        const int nb = (tnext % p.n_tiles) * BN + et;
        if (tnext < p.total_tiles && p.bias != nullptr && et < BN && nb < p.N) bnext = __ldg(p.bias + nb);
      }
      const float* sb = sbias + buf * 256;
      mbar_wait(bar_acc_full + 8 * buf, (at >> 1) & 1);
      tc_fence_after();
      const uint32_t tacc = tmem_base + buf * 256 + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c0 = wsel * 32; c0 < BN; c0 += 8 * EW) {
        uint32_t v[32];
        if (!(kDbg & 4)) tmem_ld32(tacc + (uint32_t)c0, v);       // asynchronous: completes at tmem_ld_wait()
        const int n = n0 + c0;
        const bool live = (m >= 0) && (n < p.N);
        const bool colok = (n + cchk * 8) < p.N;                   // this lane's 16-byte column group exists
        // issue every global load of this chunk (coalesced pattern) while the TMEM read is in flight
        Half8 rb8[4], rsg[4], bxg[4];
        if (!(kDbg & 2)) {
          if (rbp != nullptr && live) {
#pragma unroll
            for (int j = 0; j < 4; j++)
              if (n + 8 * j < p.N) rb8[j] = *reinterpret_cast<const Half8*>(rbp + n + 8 * j);
          }
          if (kRes) {
#pragma unroll
            for (int i = 0; i < 4; i++)
              if (mrow[i] >= 0 && colok) rsg[i] = *reinterpret_cast<const Half8*>(p.residual + mrow[i] * p.res_ld + n + cchk * 8);
          }
          if (kBlend) {
#pragma unroll
            for (int i = 0; i < 4; i++)
              if (mrow[i] >= 0 && colok) bxg[i] = *reinterpret_cast<const Half8*>(p.blend_x + mrow[i] * p.blend_ld + n + cchk * 8);
          }
        }
        tmem_ld_wait(v);
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + j);
          f[j] = __uint_as_float(v[j]) + b4.x; f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
          f[j + 2] = __uint_as_float(v[j + 2]) + b4.z; f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
        }
        if (rbp != nullptr && live) {
#pragma unroll
          for (int j = 0; j < 4; j++) {
            if (n + 8 * j >= p.N) break;
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const float2 t = __half22float2(rb8[j].h[k]);
              f[8 * j + 2 * k] += t.x; f[8 * j + 2 * k + 1] += t.y;
            }
          }
        }
        if (geglu) {
          // 32 accumulator columns = 16 (value, gate) pairs -> 16 outputs = 32 bytes per row
          Half8 o8[2];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const float2 gin = make_float2(f[2 * j + 1], f[2 * j + 3]);
            const float2 gl = p.gelu_poly ? gelu_poly2(gin) : gelu_fast2(gin);
            const float2 o = __fmul2_rn(make_float2(f[2 * j], f[2 * j + 2]), gl);
            o8[j >> 3].h[(j & 7) >> 1] = __floats2half2_rn(o.x, o.y);
          }
          *reinterpret_cast<Half8*>(scr + lane * 80) = o8[0];
          *reinterpret_cast<Half8*>(scr + lane * 80 + 16) = o8[1];
          __syncwarp();
          // 2 lanes per row: rows (lane >> 1) + 16 i
#pragma unroll
          for (int i = 0; i < 2; i++) {
            const int rr = (lane >> 1) + 16 * i, ck = lane & 1;
            const long long mr = __shfl_sync(0xffffffffu, m, rr);
            const Half8 w8 = *reinterpret_cast<const Half8*>(scr + rr * 80 + ck * 16);
            if (mr >= 0 && n + 16 * ck < p.N && !(kDbg & 1))
              *reinterpret_cast<Half8*>(p.out + mr * p.out_ld + (n >> 1) + 8 * ck) = w8;
          }
          __syncwarp();
        } else {
          if (kSilu) {
#pragma unroll
            for (int j = 0; j < 32; j++) f[j] = silu_f(f[j]);
          }
          // row-per-thread values -> shared -> coalesced pattern
#pragma unroll
          for (int c = 0; c < 4; c++) {
            Half8 o8;
#pragma unroll
            for (int k = 0; k < 4; k++) o8.h[k] = __floats2half2_rn(f[8 * c + 2 * k], f[8 * c + 2 * k + 1]);
            *reinterpret_cast<Half8*>(scr + lane * 80 + 16 * c) = o8;
          }
          __syncwarp();
          const float al = p.alpha, be = 1.f - p.alpha;
          Half8 w8s[4];                          // distinct registers: a reused one serialises on the previous store
#pragma unroll
          for (int i = 0; i < 4; i++) w8s[i] = *reinterpret_cast<const Half8*>(scr + (crow + 8 * i) * 80 + cchk * 16);
#pragma unroll
          for (int i = 0; i < 4; i++) {
            Half8& w8 = w8s[i];
            if (mrow[i] < 0 || !colok) continue;
            if (kRes && !(kDbg & 2)) {
#pragma unroll
              for (int k = 0; k < 4; k++) {
                const float2 a = __half22float2(w8.h[k]), b = __half22float2(rsg[i].h[k]);
                w8.h[k] = __floats2half2_rn(a.x + b.x, a.y + b.y);
              }
            }
            if (kBlend && !(kDbg & 2)) {
#pragma unroll
              for (int k = 0; k < 4; k++) {
                const float2 a = __half22float2(w8.h[k]), b = __half22float2(bxg[i].h[k]);
                w8.h[k] = __floats2half2_rn(al * b.x + be * a.x, al * b.y + be * a.y);
              }
            }
            if (!(kDbg & 1)) *reinterpret_cast<Half8*>(p.out + mrow[i] * p.out_ld + n + cchk * 8) = w8;
          }
          __syncwarp();
          if (gn_on) {
            // (sum, sumsq) of the values just stored (fp16-rounded: exactly what a statistics pass over the tensor sees), per
            // image and per unit of gn_unit channels, added to the global table with fire-and-forget RED.ADD.F32.
            // This lane: rows crow + 8 i (i < 4), channels n + 8 cchk .. + 7.  (First version: a per-CTA shared-memory table
            // flushed once per tile -- shared float atomics are compare-and-swap loops and the flush needed a 256-thread
            // barrier per tile; it cost the GEMMs more than the statistics pass it replaced.)
            const int cbase = n + cchk * 8;
            if (kDet || (gn_uniform && p.gn_unit >= 4)) {
              float2 s2[4], q2[4];                 // packed fp32: channel pairs (2k, 2k+1) summed over this lane's rows
#pragma unroll
              for (int k = 0; k < 4; k++) s2[k] = q2[k] = make_float2(0.f, 0.f);
#pragma unroll
              for (int i = 0; i < 4; i++) {
                if (mrow[i] < 0 || !colok) continue;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  const float2 f = __half22float2(w8s[i].h[k]);
                  s2[k] = __fadd2_rn(s2[k], f);
                  q2[k] = __ffma2_rn(f, f, q2[k]);
                }
              }
              // 8 consecutive channels (cbase is a multiple of 8) touch at most two units when gn_unit >= 4: split at the boundary
              const int ua = cbase / p.gn_unit;
              const int nb = (ua + 1) * p.gn_unit - cbase;          // channels of this lane that belong to unit ua (1..8)
              float sA = 0.f, qA = 0.f, sT = 0.f, qT = 0.f;
#pragma unroll
              for (int k = 0; k < 4; k++) {
                sT += s2[k].x + s2[k].y; qT += q2[k].x + q2[k].y;
                sA += (2 * k < nb ? s2[k].x : 0.f) + (2 * k + 1 < nb ? s2[k].y : 0.f);
                qA += (2 * k < nb ? q2[k].x : 0.f) + (2 * k + 1 < nb ? q2[k].y : 0.f);
              }
              float sB = sT - sA, qB = qT - qA;
              // sum over the 8 row groups (lanes with the same cchk: lane bits 2..4)
#pragma unroll
              for (int off = 4; off < 32; off <<= 1) {
                sA += __shfl_xor_sync(0xffffffffu, sA, off); qA += __shfl_xor_sync(0xffffffffu, qA, off);
                sB += __shfl_xor_sync(0xffffffffu, sB, off); qB += __shfl_xor_sync(0xffffffffu, qB, off);
              }
              if (kDet) {
                // slot (warp block, octet): written by exactly one lane of one warp, read by hi3d_groupnorm_fold
                if (lane < 4 && gn_slot != nullptr && colok)
                  *reinterpret_cast<float4*>(gn_slot + (cbase / 8) * 4) = make_float4(sA, qA, sB, qB);
              } else if (lane < 4 && gn_wsmp >= 0 && colok) {
                float* dst = p.gn_stats + ((long long)(gn_s0 + gn_wsmp) * p.gn_units + ua) * 2;
                atomicAdd(dst, sA); atomicAdd(dst + 1, qA);                       // results unused -> RED
                if (nb < 8 && ua + 1 < p.gn_units) { atomicAdd(dst + 2, sB); atomicAdd(dst + 3, qB); }
              }
            } else {
              // tiny models (units narrower than 4 channels: model_channels < 128) or rows of several images inside one warp
              // (images smaller than 32 pixels): one RED per stored pair -- only test-sized shapes come here.  (The 128-channel
              // VAE has 4-channel units: sending ITS 1024^2 tensors down this path cost 6 s per video in one measured build.)
#pragma unroll
              for (int i = 0; i < 4; i++) {
                if (mrow[i] < 0 || !colok || gn_srow[i] < 0) continue;
                float* row = p.gn_stats + (long long)(gn_s0 + gn_srow[i]) * p.gn_units * 2;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  const float2 f = __half22float2(w8s[i].h[k]);
                  const int c0 = cbase + 2 * k;
                  const int u0_ = c0 / p.gn_unit, u1_ = (c0 + 1) / p.gn_unit;
                  if (u0_ == u1_) {
                    atomicAdd(row + u0_ * 2, f.x + f.y); atomicAdd(row + u0_ * 2 + 1, f.x * f.x + f.y * f.y);
                  } else {
                    atomicAdd(row + u0_ * 2, f.x); atomicAdd(row + u0_ * 2 + 1, f.x * f.x);
                    atomicAdd(row + u1_ * 2, f.y); atomicAdd(row + u1_ * 2 + 1, f.y * f.y);
                  }
                }
              }
            }
          }
        }
      }
      if (et < 256) sbias[(buf ^ 1) * 256 + et] = bnext;      // next tile's slice -> the buffer nobody reads until the next bar.sync
      // this warp is done reading the accumulator buffer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NCTA == 2) mbar_arrive_cluster(lead_acc_empty + 8 * buf); else mbar_arrive(bar_acc_empty + 8 * buf);
      }
    }
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (NCTA == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
  }
}

// ---- host: tensor maps ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  }
  return fn;
}

int encode_map(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, const cuuint32_t* elem_strides) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("hi3d_gemm_tc5: cuTensorMapEncodeTiled entry point unavailable"); return -1; }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if (elem_strides) for (int i = 0; i < rank; i++) estr[i] = elem_strides[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides_bytes, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("hi3d_gemm_tc5: cuTensorMapEncodeTiled failed (%d) rank=%d dims=%llu,%llu box=%u,%u", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return -1;
  }
  return 0;
}

static bool pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

// experiment knobs, read from the environment ONCE per process (not per call: getenv on every eager launch was measurable
// in the un-graphed frame-sharded mode); hi3d_gemm_tc5_set_pair_mode overrides the pair knob for tests
static int g_pair_mode = -2;      // -2 unread, -1 auto, 0 single CTA, 1 CTA pairs
static int g_dbg = -1;            // -1 unread
static int g_ew_mode = -2;        // -2 unread, -1 auto, 8 / 16 forced (HI3D_TC5_EW)
static int g_gelu_poly = -1;      // -1 unread; HI3D_TC5_GELU=poly selects the MUFU-free gate (measured: same speed, so the default stays A-S)
constexpr int T5_EW16_MAX_K = 640;
static void read_env_once() {
  if (g_pair_mode == -2) { const char* e = getenv("HI3D_TC5_PAIR"); g_pair_mode = e ? atoi(e) : -1; }
  if (g_dbg < 0) { const char* e = getenv("HI3D_TC5_DBG"); g_dbg = e ? atoi(e) : 0; }
  if (g_gelu_poly < 0) { const char* e = getenv("HI3D_TC5_GELU"); g_gelu_poly = (e && e[0] == 'p') ? 1 : 0; }
  if (g_ew_mode == -2) { const char* e = getenv("HI3D_TC5_EW"); g_ew_mode = e ? atoi(e) : -1; if (g_ew_mode != 8 && g_ew_mode != 16) g_ew_mode = -1; }
}

template <int NCTA, int EPI, int EW>
static int launch_tc5_one(const T5Params& tp, int smem, int smem_total, int units, int sm_count, cudaStream_t st) {
  static bool attr_done[HI3D_MAX_DEVICES];
  if (ensure_dyn_smem(gemm_tc5_kernel<NCTA, EPI, EW>, smem_total, attr_done, "hi3d_gemm_tc5")) return -1;
  constexpr int THREADS = 64 + 32 * EW;
  if (NCTA == 2) {
    const int grid = 2 * (tp.total_tiles < units ? tp.total_tiles : units);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc5_kernel<2, EPI, EW>, tp);
    if (e != cudaSuccess) { set_error("hi3d_gemm_tc5: pair launch: %s", cudaGetErrorString(e)); return -1; }
  } else {
    const int grid = tp.total_tiles < sm_count ? tp.total_tiles : sm_count;
    gemm_tc5_kernel<1, EPI, EW><<<grid, THREADS, smem, st>>>(tp);
  }
  return 0;
}

template <int NCTA>
static int launch_tc5_n(int epi, int ew, const T5Params& tp, int smem, int smem_total, int units, int sm_count, cudaStream_t st) {
  if (ew == 16) {      // only the register-light specialisations exist with 16 epilogue warps
    if (epi == EPI_GEGLU) return launch_tc5_one<NCTA, EPI_GEGLU, 16>(tp, smem, smem_total, units, sm_count, st);
    if (epi == EPI_BIAS) return launch_tc5_one<NCTA, EPI_BIAS, 16>(tp, smem, smem_total, units, sm_count, st);
    if (epi == EPI_RES) return launch_tc5_one<NCTA, EPI_RES, 16>(tp, smem, smem_total, units, sm_count, st);
  }
  switch (epi) {
    case EPI_GEGLU: return launch_tc5_one<NCTA, EPI_GEGLU, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_BIAS: return launch_tc5_one<NCTA, EPI_BIAS, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RES: return launch_tc5_one<NCTA, EPI_RES, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RESBLEND: return launch_tc5_one<NCTA, EPI_RESBLEND, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_BIAS_GN: return launch_tc5_one<NCTA, EPI_BIAS_GN, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RES_GN: return launch_tc5_one<NCTA, EPI_RES_GN, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RESBLEND_GN: return launch_tc5_one<NCTA, EPI_RESBLEND_GN, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_BIAS_GN_DET: return launch_tc5_one<NCTA, EPI_BIAS_GN_DET, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RES_GN_DET: return launch_tc5_one<NCTA, EPI_RES_GN_DET, 8>(tp, smem, smem_total, units, sm_count, st);
    case EPI_RESBLEND_GN_DET: return launch_tc5_one<NCTA, EPI_RESBLEND_GN_DET, 8>(tp, smem, smem_total, units, sm_count, st);
    default: return launch_tc5_one<NCTA, EPI_GENERIC, 8>(tp, smem, smem_total, units, sm_count, st);
  }
}

static int launch_tc5(int ncta, int epi, int ew, const T5Params& tp, int smem, int smem_total, int units, int sm_count,
                      cudaStream_t st) {
  return ncta == 2 ? launch_tc5_n<2>(epi, ew, tp, smem, smem_total, units, sm_count, st)
                   : launch_tc5_n<1>(epi, ew, tp, smem, smem_total, units, sm_count, st);
}

}  // namespace hi3d

using namespace hi3d;

extern "C" int hi3d_gemm_tc5_set_pair_mode(int mode) {
  if (mode < -1 || mode > 1) { set_error("hi3d_gemm_tc5_set_pair_mode: mode must be -1 (auto), 0 or 1"); return -2; }
  read_env_once();
  g_pair_mode = mode;
  return 0;
}

extern "C" int hi3d_gemm_tc5_set_epilogue_warps(int warps) {
  if (warps != -1 && warps != 8 && warps != 16) { set_error("hi3d_gemm_tc5_set_epilogue_warps: -1 (auto), 8 or 16"); return -2; }
  read_env_once();
  g_ew_mode = warps;
  return 0;
}

// partials != NULL: deterministic GroupNorm statistics (hi3d_gemm_tc5_det); geometries this engine does not cover go to
// hi3d_gemm / hi3d_gemm_det accordingly
static int gemm_tc5(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream) {
  int rc = validate_gemm(p, "hi3d_gemm_tc5");
  if (rc) return rc;
  auto fallback = [&]() { return partials ? hi3d_gemm_det(p, partials, partials_floats, stream) : hi3d_gemm(p, stream); };
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // ---- geometry this engine covers; everything else goes to the mma.sync engine (same results) ----
  T5Params tp;
  memset(&tp, 0, sizeof(tp));
  tp.M = p->M; tp.N = p->N; tp.K = p->K; tp.mode = p->mode; tp.nseg = p->nseg;
  tp.cstride = (p->mode == HI3D_ROWS_CONV2D) ? p->stride : 1;
  tp.out_up = p->out_up; tp.out_py = p->out_py; tp.out_px = p->out_px;
  tp.t_off = p->t_off;
  int m_tiles = 0;
  bool ok = (p->N >= 32) && (p->N % 8 == 0);
  // the vectorised epilogue needs 16-byte aligned rows / bias
  ok = ok && (p->rowbias == nullptr || ((uintptr_t)p->rowbias % 16 == 0 && p->rb_ld % 8 == 0));
  if (p->mode == HI3D_ROWS_PLAIN) {
    tp.tw = 128; tp.th = 1; tp.tn = 1;
    m_tiles = (p->M + T5_BM - 1) / T5_BM;
  } else if (p->mode == HI3D_ROWS_CONV2D) {
    ok = ok && p->ups == 0 && ((p->stride == 1 && p->Ho == p->Hs && p->Wo == p->Ws) ||
                               (p->stride == 2 && p->Hs == 2 * p->Ho && p->Ws == 2 * p->Wo && !p->out_up));
    const int Nimg = ok ? p->M / (p->Ho * p->Wo) : 0;
    int tw = 1;
    while (tw * 2 <= 16 && (p->Wo % (tw * 2)) == 0) tw *= 2;
    int th = 1;
    while (tw * th * 2 <= 128 && (p->Ho % (th * 2)) == 0) th *= 2;
    int tn = ok ? 128 / (tw * th) : 1;
    ok = ok && pow2(tn) && tw * th * tn == 128 && (Nimg % tn) == 0;
    tp.tw = tw; tp.th = th; tp.tn = tn; tp.Wo = p->Wo; tp.Ho = p->Ho; tp.Nimg = Nimg;
    tp.tiles_x = p->Wo / tw; tp.tiles_y = p->Ho / th;
    m_tiles = ok ? tp.tiles_x * tp.tiles_y * (Nimg / tn) : 0;
  } else {
    const int HW = p->Ho * p->Wo, T = p->T, B = p->M / (HW * T);
    int ts = 1;
    while (ts * 2 <= 128 && (HW % (ts * 2)) == 0) ts *= 2;
    int tf = 128 / ts;
    ok = ok && (T % tf) == 0;
    tp.tw = ts; tp.th = tf; tp.tn = 1; tp.Wo = HW; tp.Ho = T; tp.Nimg = B;
    tp.tiles_x = HW / ts; tp.tiles_y = ok ? T / tf : 1;
    m_tiles = ok ? tp.tiles_x * tp.tiles_y * B : 0;
  }
  // distinct A sources -> tensor maps
  const void* srcs[T5_MAX_MAPS];
  int lds[T5_MAX_MAPS];
  int nmaps = 0;
  for (int i = 0; ok && i < p->nseg; i++) {
    const hi3d_seg& s = p->seg[i];
    int mi = -1;
    for (int j = 0; j < nmaps; j++)
      if (srcs[j] == s.src && lds[j] == s.ld) mi = j;
    if (mi < 0) {
      if (nmaps == T5_MAX_MAPS) { ok = false; break; }
      srcs[nmaps] = s.src; lds[nmaps] = s.ld; mi = nmaps++;
    }
    tp.seg[i].map = mi; tp.seg[i].c_off = s.c_off; tp.seg[i].C = s.C;
    tp.seg[i].dy = s.dy; tp.seg[i].dx = s.dx; tp.seg[i].dt = s.dt;
  }
  if (!ok) return fallback();

  // tile-N: multiple of 32 in [32, 256].  Cost model = rounds of the persistent grid x time per tile, where a tile
  // costs its MMA columns plus a fixed term (A-operand traffic / epilogue set-up); this accounts both for the padding
  // of N and for wave quantisation over the SMs (e.g. N = 1280 with 64 row-tiles: 5 x 256 -> 3 rounds, 8 x 160 -> 4
  // rounds of much shorter tiles).  Ties go to the wider tile.
  const int g_sm_count = device_sm_count();
  read_env_once();
  // CTA pairs (cta_group::2, 256-row tiles) halve the B bytes each SM pulls from L2 -- the conv / linear main loops are
  // L2 -> SM bandwidth bound, not tensor bound -- but leave half as many schedulable units: used when there is enough
  // work to fill the pairs (HI3D_TC5_PAIR=0|1 forces it for experiments).
  const int pair_env = g_pair_mode;
  int ncta = 1;
  // measured (profiles/r01_microbench_pair.txt): pairs win 5-15 % once the main loop dominates (K >= ~2000: 3x3 convs,
  // wide temporal convs, ff2 at C >= 640) and lose on short-K, epilogue-bound GEMMs (both epilogues gate one accumulator).
  if (pair_env == 1 || (pair_env < 0 && p->K >= 1920 && (long long)m_tiles * ((p->N + 255) / 256) >= 2LL * g_sm_count)) ncta = 2;
  const int m_units = (m_tiles + ncta - 1) / ncta, units = g_sm_count / ncta;
  int BN = 256;
  {
    long long best = -1;
    for (int cand = 256; cand >= 32; cand -= 32) {
      if (p->act == HI3D_ACT_GEGLU && (cand % 64)) continue;     // keep GEGLU output chunks 32-byte aligned
      const long long ntl = (p->N + cand - 1) / cand;
      const long long rounds = ((long long)m_units * ntl + units - 1) / units;
      const long long cost = rounds * (cand + 48);
      if (best < 0 || cost < best) { best = cost; BN = cand; }
    }
  }
  // GroupNorm statistics in the epilogue
  const int gn_tab_bytes = 0;
  if (p->gn_stats != nullptr) {
    const int hw = (p->mode == HI3D_ROWS_PLAIN) ? p->gn_rows : p->Ho * p->Wo;
    if (p->gn_unit <= 0 || (p->N % p->gn_unit) || p->gn_rows <= 0 || (p->M % p->gn_rows) || p->act == HI3D_ACT_GEGLU ||
        (p->mode != HI3D_ROWS_PLAIN && p->gn_rows != hw)) {
      set_error("hi3d_gemm_tc5: bad gn_stats arguments (unit %d, rows %d, N %d, M %d)", p->gn_unit, p->gn_rows, p->N, p->M);
      return -2;
    }
    tp.gn_stats = p->gn_stats; tp.gn_unit = p->gn_unit; tp.gn_rows = p->gn_rows;
    tp.gn_units = p->N / p->gn_unit; tp.gn_nimg = p->M / p->gn_rows;
  }
  tp.gelu_poly = g_gelu_poly;
  // deterministic statistics (hi3d_gemm_tc5_det): per-warp slots from the specialised epilogues when every 32-row
  // warp block lies inside one image and an octet reaches into at most two units; otherwise no epilogue statistics and a
  // deterministic statistics pass over the stored tensor after the launch
  const bool has_res = p->residual != nullptr, has_blend = p->blend_x != nullptr;
  const bool det = p->gn_stats != nullptr && partials != nullptr;
  const int det_npar = p->out_up ? 4 : 1;
  bool det_slots = false;
  if (det) {
    const bool one_image = (p->mode == HI3D_ROWS_PLAIN) ? (p->gn_rows % 32 == 0)
                           : (p->mode == HI3D_ROWS_CONV2D) ? (tp.tw * tp.th >= 32) : (tp.tw >= 32);
    det_slots = one_image && (p->gn_unit == 4 || p->gn_unit >= 8) && g_dbg == 0 && p->act == HI3D_ACT_NONE &&
                !(has_blend && !has_res);
    const int64_t need = det_slots ? (int64_t)tp.gn_nimg * det_npar * (p->gn_rows / 32) * (p->N / 8) * 4 : 0;
    if (partials_floats < need || (!det_slots && p->out_ld != p->N)) {
      set_error("hi3d_gemm_tc5: deterministic statistics need %lld partials floats (have %lld) and out_ld == N (%d, %d)",
                (long long)need, (long long)partials_floats, p->out_ld, p->N);
      return -2;
    }
    if (det_slots) { tp.gn_part = partials; tp.gn_bpi = p->gn_rows / 32; }
    else tp.gn_stats = nullptr;
  }
  const bool has_gn = tp.gn_stats != nullptr;
  // epilogue specialisation and epilogue warp count (decided here: the scratch of 16 warps comes out of the stage budget)
  int epi = EPI_GENERIC;
  if (g_dbg == 0 && p->act != HI3D_ACT_SILU && !(has_blend && !has_res)) {
    if (p->act == HI3D_ACT_GEGLU) epi = (has_res || has_blend || has_gn) ? EPI_GENERIC : EPI_GEGLU;
    else if (has_blend) epi = has_gn ? (det_slots ? EPI_RESBLEND_GN_DET : EPI_RESBLEND_GN) : EPI_RESBLEND;
    else if (has_res) epi = has_gn ? (det_slots ? EPI_RES_GN_DET : EPI_RES_GN) : EPI_RES;
    else epi = has_gn ? (det_slots ? EPI_BIAS_GN_DET : EPI_BIAS_GN) : EPI_BIAS;
  }
  // 16 epilogue warps when the epilogue is the bound: short K (main loop of a tile shorter than its epilogue)
  int ew = 8;
  if ((epi == EPI_GEGLU || epi == EPI_BIAS || epi == EPI_RES) && (g_ew_mode == 16 || (g_ew_mode < 0 && p->K <= T5_EW16_MAX_K))) ew = 16;
  const int extra_scr = (ew - T5_EPI_WARPS) * T5_SCR_BYTES;
  const int stage_bytes = T5_A_BYTES + (BN / ncta) * 128;
  int stages = (T5_SMEM_BUDGET - gn_tab_bytes - extra_scr) / stage_bytes;
  if (stages > T5_MAX_STAGES) stages = T5_MAX_STAGES;
  if (stages < 2) { return fallback(); }
  tp.BN = BN; tp.stages = stages;
  tp.n_tiles = (p->N + BN - 1) / BN;
  tp.total_tiles = m_units * tp.n_tiles;      // (pair-)tiles

  for (int j = 0; j < nmaps; j++) {
    const cuuint64_t ld = (cuuint64_t)lds[j];
    if (p->mode == HI3D_ROWS_PLAIN) {
      cuuint64_t dims[2] = {ld, (cuuint64_t)p->M};
      cuuint64_t str[1] = {ld * 2};
      cuuint32_t box[2] = {64, 128};
      if (encode_map(&tp.amap[j], srcs[j], 2, dims, str, box, nullptr)) return -1;
    } else if (p->mode == HI3D_ROWS_CONV2D) {
      cuuint64_t dims[4] = {ld, (cuuint64_t)p->Ws, (cuuint64_t)p->Hs, (cuuint64_t)tp.Nimg};
      cuuint64_t str[3] = {ld * 2, ld * 2 * p->Ws, ld * 2 * p->Ws * p->Hs};
      const cuuint32_t cs = (cuuint32_t)tp.cstride;   // stride 2: box spans 2*tw x 2*th input pixels, every 2nd loaded
      cuuint32_t box[4] = {64, (cuuint32_t)tp.tw * cs, (cuuint32_t)tp.th * cs, (cuuint32_t)tp.tn};
      cuuint32_t est[4] = {1, cs, cs, 1};
      if (encode_map(&tp.amap[j], srcs[j], 4, dims, str, box, est)) return -1;
    } else {
      const cuuint64_t HW = (cuuint64_t)tp.Wo, T = (cuuint64_t)(p->Tin > 0 ? p->Tin : tp.Ho);   // source frames per clip
      cuuint64_t dims[4] = {ld, HW, T, (cuuint64_t)tp.Nimg};
      cuuint64_t str[3] = {ld * 2, ld * 2 * HW, ld * 2 * HW * T};
      cuuint32_t box[4] = {64, (cuuint32_t)tp.tw, (cuuint32_t)tp.th, 1};
      if (encode_map(&tp.amap[j], srcs[j], 4, dims, str, box, nullptr)) return -1;
    }
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)p->K, (cuuint64_t)p->N};
    cuuint64_t str[1] = {(cuuint64_t)p->K * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(BN / ncta)};
    if (encode_map(&tp.bmap, p->W, 2, dims, str, box, nullptr)) return -1;
  }
  tp.bias = p->bias; tp.rowbias = (const __half*)p->rowbias; tp.rb_div = p->rb_div; tp.rb_mod = p->rb_mod;
  tp.rb_ld = p->rb_ld; tp.act = p->act; tp.residual = (const __half*)p->residual; tp.res_ld = p->res_ld;
  tp.blend_x = (const __half*)p->blend_x; tp.blend_ld = p->blend_ld; tp.alpha = p->alpha;
  tp.out = (__half*)p->out; tp.out_ld = p->out_ld;
  tp.dbg = g_dbg;

  const int smem_total = T5_SMEM_BUDGET + 16 * T5_MAX_STAGES + 64 + 2048 + T5_EPI_WARPS * T5_SCR_BYTES + 1024;
  const int smem = stages * stage_bytes + 16 * T5_MAX_STAGES + 64 + 2048 + ew * T5_SCR_BYTES + gn_tab_bytes + 1024;
  rc = launch_tc5(ncta, epi, ew, tp, smem, smem_total, units, g_sm_count, st);
  if (rc) return rc;
  rc = check_launch("hi3d_gemm_tc5");
  // deterministic statistics: fold the slots (or run the pass) once the tensor is complete -- after the last parity launch
  if (rc || !det || (p->out_up && !(p->out_py == 1 && p->out_px == 1))) return rc;
  if (det_slots)
    return hi3d_groupnorm_fold(partials, tp.gn_nimg, det_npar * (p->gn_rows / 32), 1, p->N, p->gn_unit, p->gn_stats, stream);
  return hi3d_groupnorm_unit_stats_det(p->out, p->N, tp.gn_nimg, (int64_t)p->gn_rows * det_npar, p->gn_unit, p->gn_stats,
                                       partials, partials_floats, stream);
}

extern "C" int hi3d_gemm_tc5(const hi3d_gemm_params* p, void* stream) { return gemm_tc5(p, nullptr, 0, stream); }

extern "C" int hi3d_gemm_tc5_det(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream) {
  if (!partials) { set_error("hi3d_gemm_tc5_det: null partials table"); return -2; }
  return gemm_tc5(p, partials, partials_floats, stream);
}
