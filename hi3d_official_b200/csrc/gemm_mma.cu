// Implicit-GEMM engine, first engine: cp.async multistage pipeline + ldmatrix + mma.sync (HMMA) with
// fp32 accumulation.  The A operand is gathered on the fly from NHWC fp16 tensors (conv taps, temporal
// taps, virtual channel-concat, fused nearest-upsample, fused 1x1 skip) -- see include/hi3d_b200.h.
//
// Tile: 128 x BN x 64 per CTA, 256 threads (8 warps), STAGES-deep cp.async ring.  Shared tiles use the
// 128-byte XOR swizzle (common.cuh::swz128) which is also the tcgen05 SWIZZLE_128B K-major layout, so
// the gather/loader code is shared with the tcgen05 engine (gemm_tc5.cu).
#include <stdarg.h>
#include <stdio.h>

#include <atomic>

#include "common.cuh"

namespace hi3d {

// ---------------------------------------------------------------------------------------------
// host-side error / accounting plumbing (shared by all translation units)
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= HI3D_MAX_DEVICES) d = 0;
  return d;
}
int device_sm_count() {
  static int cnt[HI3D_MAX_DEVICES];     // zero-initialised; benign race (idempotent)
  const int d = current_device();
  if (cnt[d] <= 0) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d);
    cnt[d] = v > 0 ? v : 148;
  }
  return cnt[d];
}
int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return -1;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 256;

template <int BN, int STAGES>
struct GemmSmem {
  static constexpr int A_BYTES = BM * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TOTAL = STAGES * STAGE_BYTES;
};

template <int MODE, int BN, int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_mma_kernel(const __grid_constant__ hi3d_gemm_params p) {
  constexpr int WARPS_N = (BN == 128) ? 4 : 2;
  constexpr int WARPS_M = 8 / WARPS_N;
  constexpr int WM = BM / WARPS_M;  // 64 or 32
  constexpr int WN = BN / WARPS_N;  // 32
  constexpr int MT = WM / 16;
  constexpr int NT = WN / 8;
  using SM = GemmSmem<BN, STAGES>;

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int wm = warp / WARPS_N, wn = warp % WARPS_N;
  const int m0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int KT = p.K / BK;

  // ---- loader state ------------------------------------------------------------------------
  const int chunk = tid & 7;
  const int row_base = tid >> 3;  // 0..31
  bool rvalid[4];
  int ra[4], rb[4], rc[4];  // CONV: n*Hs, oy*stride, ox*stride ; TEMPORAL: t ; PLAIN: unused
  const int HW = p.Ho * p.Wo;
  const int Hin = p.Hs << p.ups, Win = p.Ws << p.ups;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int m = m0 + row_base + 32 * i;
    rvalid[i] = m < p.M;
    int mm = rvalid[i] ? m : 0;
    if (MODE == HI3D_ROWS_CONV2D) {
      int n = mm / HW, rem = mm - n * HW;
      int oy = rem / p.Wo, ox = rem - oy * p.Wo;
      ra[i] = n * p.Hs;
      rb[i] = oy * p.stride;
      rc[i] = ox * p.stride;
    } else if (MODE == HI3D_ROWS_TEMPORAL) {
      const int fr = mm / HW;                 // output frame index (b * T + t)
      ra[i] = fr % p.T + p.t_off;             // frame position inside the source clip
      rb[i] = (fr / p.T) * (p.Tin > 0 ? p.Tin : p.T);   // first source frame of this clip
      rc[i] = mm - fr * HW;                   // pixel
    } else {
      ra[i] = rb[i] = rc[i] = 0;
    }
  }
  int si = 0, so = 0, kglob = 0;
  const __half* Wp = reinterpret_cast<const __half*>(p.W);

  auto load_tile = [&](int stage) {
    const hi3d_seg& sg = p.seg[si];
    const __half* sbase = reinterpret_cast<const __half*>(sg.src) + sg.c_off + so + chunk * 8;
    const uint32_t sA = smem_base + stage * SM::STAGE_BYTES;
    const uint32_t sB = sA + SM::A_BYTES;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int r = row_base + 32 * i;
      bool v = rvalid[i];
      long long pix;
      if (MODE == HI3D_ROWS_CONV2D) {
        int iy = rb[i] + sg.dy, ix = rc[i] + sg.dx;
        v = v && ((unsigned)iy < (unsigned)Hin) && ((unsigned)ix < (unsigned)Win);
        pix = (long long)(ra[i] + (iy >> p.ups)) * p.Ws + (ix >> p.ups);
      } else if (MODE == HI3D_ROWS_TEMPORAL) {
        int tt = ra[i] + sg.dt;
        v = v && ((unsigned)tt < (unsigned)(p.Tin > 0 ? p.Tin : p.T));
        pix = (long long)(rb[i] + tt) * HW + rc[i];
      } else {
        pix = m0 + r;
      }
      const __half* src = v ? (sbase + pix * sg.ld) : reinterpret_cast<const __half*>(sg.src);
      cp_async16(sA + swz128(r, chunk), src, v);
    }
#pragma unroll
    for (int i = 0; i < BN / 32; i++) {
      const int r = row_base + 32 * i;
      const int n = n0 + r;
      const bool v = n < p.N;
      const __half* src = v ? (Wp + (long long)n * p.K + kglob + chunk * 8) : Wp;
      cp_async16(sB + swz128(r, chunk), src, v);
    }
    kglob += BK;
    so += BK;
    if (so >= sg.C) {
      si++;
      so = 0;
    }
  };

  float acc[MT][NT][4];
#pragma unroll
  for (int i = 0; i < MT; i++)
#pragma unroll
    for (int j = 0; j < NT; j++)
#pragma unroll
      for (int k = 0; k < 4; k++) acc[i][j][k] = 0.f;

  // ---- prologue ------------------------------------------------------------------------------
#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < KT) load_tile(s);
    cp_async_commit();
  }

  // ---- main loop -----------------------------------------------------------------------------
  for (int kt = 0; kt < KT; kt++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nk = kt + STAGES - 1;
      if (nk < KT) load_tile(nk % STAGES);
      cp_async_commit();
    }
    const uint32_t sA = smem_base + (kt % STAGES) * SM::STAGE_BYTES;
    const uint32_t sB = sA + SM::A_BYTES;
#pragma unroll
    for (int k16 = 0; k16 < BK / 16; k16++) {
      uint32_t a[MT][4], b[NT][2];
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
        ldmatrix_x4(a[mt][0], a[mt][1], a[mt][2], a[mt][3],
                    sA + swz128(wm * WM + mt * 16 + (lane & 15), k16 * 2 + (lane >> 4)));
#pragma unroll
      for (int np = 0; np < NT / 2; np++)
        ldmatrix_x4(b[2 * np][0], b[2 * np][1], b[2 * np + 1][0], b[2 * np + 1][1],
                    sB + swz128(wn * WN + np * 16 + (lane & 7) + ((lane >> 4) << 3), k16 * 2 + ((lane >> 3) & 1)));
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
#pragma unroll
        for (int nt = 0; nt < NT; nt++) mma_16816(acc[mt][nt], a[mt], b[nt][0], b[nt][1]);
    }
  }
  cp_async_wait<0>();
  __syncthreads();

  // ---- epilogue phase 1: registers -> (bias, rowbias, activation) -> fp16 staging tile in smem ----
  const bool geglu = (p.act == HI3D_ACT_GEGLU);
  const int BNo = geglu ? BN / 2 : BN;          // staged tile width
  const int pitch = BN + 8;                     // halfs
  __half* sC = reinterpret_cast<__half*>(smem);
  const int g = lane >> 2, t4 = lane & 3;
  const __half* rowbias = reinterpret_cast<const __half*>(p.rowbias);
#pragma unroll
  for (int mt = 0; mt < MT; mt++) {
#pragma unroll
    for (int hh = 0; hh < 2; hh++) {
      const int rl = wm * WM + mt * 16 + g + 8 * hh;
      const int m = m0 + rl;
      const __half* rbp = nullptr;
      if (rowbias != nullptr && m < p.M) rbp = rowbias + (long long)((m / p.rb_div) % p.rb_mod) * p.rb_ld;
#pragma unroll
      for (int nt = 0; nt < NT; nt++) {
        const int cl = wn * WN + nt * 8 + 2 * t4;
        const int n = n0 + cl;
        float v0 = acc[mt][nt][2 * hh], v1 = acc[mt][nt][2 * hh + 1];
        if (n < p.N) {
          if (p.bias != nullptr) {
            v0 += __ldg(p.bias + n);
            v1 += __ldg(p.bias + n + 1);
          }
          if (rbp != nullptr) {
            __half2 rbv = *reinterpret_cast<const __half2*>(rbp + n);
            v0 += __low2float(rbv);
            v1 += __high2float(rbv);
          }
        }
        if (geglu) {
          sC[rl * pitch + (cl >> 1)] = __float2half_rn(v0 * gelu_erf_f(v1));
        } else {
          if (p.act == HI3D_ACT_SILU) {
            v0 = silu_f(v0);
            v1 = silu_f(v1);
          }
          *reinterpret_cast<uint32_t*>(sC + rl * pitch + cl) = pack_half2(v0, v1);
        }
      }
    }
  }
  __syncthreads();

  // ---- epilogue phase 2: coalesced 16-byte stores with residual / blend ---------------------------
  const int cpr = BNo / 8;  // 16-byte chunks per staged row
  const int Nout = geglu ? p.N / 2 : p.N;
  const int nout0 = geglu ? n0 / 2 : n0;
  const __half* res = reinterpret_cast<const __half*>(p.residual);
  const __half* bx = reinterpret_cast<const __half*>(p.blend_x);
  __half* out = reinterpret_cast<__half*>(p.out);
  for (int idx = tid; idx < BM * cpr; idx += GEMM_THREADS) {
    const int r = idx / cpr, c = idx - r * cpr;
    const int m = m0 + r;
    const int nc = nout0 + c * 8;
    if (m >= p.M || nc >= Nout) continue;
    long long mo = m;                       // output row (differs from m only for the parity-class upsample convs)
    if (p.out_up) {
      const int n_ = m / HW, rem_ = m - n_ * HW;
      const int y_ = rem_ / p.Wo, x_ = rem_ - y_ * p.Wo;
      mo = ((long long)n_ * 2 * p.Ho + 2 * y_ + p.out_py) * (2 * p.Wo) + 2 * x_ + p.out_px;
    }
    Half8 v = *reinterpret_cast<const Half8*>(sC + r * pitch + c * 8);
    if (res != nullptr) {
      Half8 rr = *reinterpret_cast<const Half8*>(res + mo * p.res_ld + nc);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        float2 a = __half22float2(v.h[q]), b = __half22float2(rr.h[q]);
        v.h[q] = __floats2half2_rn(a.x + b.x, a.y + b.y);
      }
    }
    if (bx != nullptr) {
      Half8 xx = *reinterpret_cast<const Half8*>(bx + mo * p.blend_ld + nc);
      const float al = p.alpha, be = 1.f - p.alpha;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        float2 a = __half22float2(v.h[q]), b = __half22float2(xx.h[q]);
        v.h[q] = __floats2half2_rn(al * b.x + be * a.x, al * b.y + be * a.y);
      }
    }
    *reinterpret_cast<Half8*>(out + mo * p.out_ld + nc) = v;
  }
}

template <int MODE, int BN>
static int launch_gemm(const hi3d_gemm_params& p, cudaStream_t st) {
  constexpr int STAGES = 3;
  using SM = GemmSmem<BN, STAGES>;
  static bool attr_done[HI3D_MAX_DEVICES];  // per device; benign race: idempotent
  auto kern = gemm_mma_kernel<MODE, BN, STAGES>;
  if (ensure_dyn_smem(kern, SM::TOTAL, attr_done, "hi3d_gemm")) return -1;
  dim3 grid((p.M + BM - 1) / BM, (p.N + BN - 1) / BN);
  kern<<<grid, GEMM_THREADS, SM::TOTAL, st>>>(p);
  return check_launch("hi3d_gemm");
}

int validate_gemm(const hi3d_gemm_params* p, const char* who) {
  if (p == nullptr) { set_error("%s: null params", who); return -2; }
  if (p->M <= 0 || p->N <= 0 || p->K <= 0) { set_error("%s: bad M/N/K %d/%d/%d", who, p->M, p->N, p->K); return -2; }
  if (p->N % 8) { set_error("%s: N=%d must be a multiple of 8", who, p->N); return -2; }
  if (p->nseg <= 0 || p->nseg > HI3D_MAX_SEGS) { set_error("%s: nseg=%d out of range", who, p->nseg); return -2; }
  long long ksum = 0;
  for (int i = 0; i < p->nseg; i++) {
    const hi3d_seg& s = p->seg[i];
    if (s.src == nullptr || s.C <= 0 || s.C % 64 || s.ld % 8 || s.c_off % 8 || ((uintptr_t)s.src & 15)) {
      set_error("%s: bad segment %d (src=%p C=%d ld=%d c_off=%d)", who, i, s.src, s.C, s.ld, s.c_off);
      return -2;
    }
    ksum += s.C;
  }
  if (ksum != p->K) { set_error("%s: sum of segment channels %lld != K %d", who, ksum, p->K); return -2; }
  if (p->W == nullptr || p->out == nullptr || ((uintptr_t)p->W & 15) || ((uintptr_t)p->out & 15) || p->out_ld % 8) {
    set_error("%s: W/out null or misaligned (out_ld=%d)", who, p->out_ld);
    return -2;
  }
  if (p->residual && (((uintptr_t)p->residual & 15) || p->res_ld % 8)) { set_error("%s: residual misaligned", who); return -2; }
  if (p->blend_x && (((uintptr_t)p->blend_x & 15) || p->blend_ld % 8)) { set_error("%s: blend_x misaligned", who); return -2; }
  if (p->rowbias && (p->rb_div <= 0 || p->rb_mod <= 0 || p->rb_ld % 2)) { set_error("%s: bad rowbias div/mod/ld", who); return -2; }
  if (p->act == HI3D_ACT_GEGLU && (p->N % 16)) { set_error("%s: GEGLU needs N %% 16 == 0", who); return -2; }
  if (p->mode == HI3D_ROWS_CONV2D) {
    if (p->Ho <= 0 || p->Wo <= 0 || p->Hs <= 0 || p->Ws <= 0 || (p->stride != 1 && p->stride != 2) ||
        (p->ups != 0 && p->ups != 1) || (p->M % (p->Ho * p->Wo))) {
      set_error("%s: bad conv geometry Ho=%d Wo=%d Hs=%d Ws=%d stride=%d ups=%d M=%d", who, p->Ho, p->Wo, p->Hs,
                p->Ws, p->stride, p->ups, p->M);
      return -2;
    }
    if (p->out_up && (p->stride != 1 || p->ups != 0 || (p->out_py & ~1) || (p->out_px & ~1))) {
      set_error("%s: out_up needs stride 1, ups 0 and parities in {0,1}", who);
      return -2;
    }
  } else if (p->out_up) {
    set_error("%s: out_up is a CONV2D option", who);
    return -2;
  } else if (p->mode == HI3D_ROWS_TEMPORAL) {
    if (p->T <= 0 || p->Ho * p->Wo <= 0 || (p->M % (p->T * p->Ho * p->Wo)) || p->Tin < 0 || p->t_off < 0 ||
        (p->Tin > 0 && p->t_off + p->T > p->Tin)) {
      set_error("%s: bad temporal geometry T=%d HW=%d M=%d", who, p->T, p->Ho * p->Wo, p->M);
      return -2;
    }
  } else if (p->mode != HI3D_ROWS_PLAIN) {
    set_error("%s: unknown row mode %d", who, p->mode);
    return -2;
  }
  return 0;
}

}  // namespace hi3d

using namespace hi3d;

// partials != NULL: deterministic GroupNorm statistics (hi3d_gemm_det)
static int gemm_mma(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream) {
  int rc = validate_gemm(p, "hi3d_gemm");
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // tile-N choice: padded work with a 15% penalty for the narrower (lower-intensity) tile
  const double c128 = (double)((p->N + 127) / 128) * 128.0;
  const double c64 = (double)((p->N + 63) / 64) * 64.0 * 1.15;
  const bool wide = c128 <= c64;
  switch (p->mode) {
    case HI3D_ROWS_PLAIN:
      rc = wide ? launch_gemm<HI3D_ROWS_PLAIN, 128>(*p, st) : launch_gemm<HI3D_ROWS_PLAIN, 64>(*p, st);
      break;
    case HI3D_ROWS_CONV2D:
      rc = wide ? launch_gemm<HI3D_ROWS_CONV2D, 128>(*p, st) : launch_gemm<HI3D_ROWS_CONV2D, 64>(*p, st);
      break;
    default:
      rc = wide ? launch_gemm<HI3D_ROWS_TEMPORAL, 128>(*p, st) : launch_gemm<HI3D_ROWS_TEMPORAL, 64>(*p, st);
  }
  if (rc || p->gn_stats == nullptr) return rc;
  // hi3d_gemm_params::gn_stats on this (first, mma.sync) engine: a separate statistics pass over the stored tensor.  The
  // four parity-class launches of an up-conv fill one tensor: the pass runs after the last one.
  if (p->gn_unit <= 0 || (p->N % p->gn_unit) || p->gn_rows <= 0 || (p->M % p->gn_rows) || p->act == HI3D_ACT_GEGLU ||
      p->out_ld != p->N) {
    set_error("hi3d_gemm: bad gn_stats arguments (unit %d, rows %d, N %d, out_ld %d)", p->gn_unit, p->gn_rows, p->N, p->out_ld);
    return -2;
  }
  if (p->out_up && !(p->out_py == 1 && p->out_px == 1)) return 0;
  if (partials != nullptr)
    return hi3d_groupnorm_unit_stats_det(p->out, p->N, p->M / p->gn_rows, (int64_t)p->gn_rows * (p->out_up ? 4 : 1), p->gn_unit,
                                         p->gn_stats, partials, partials_floats, stream);
  return hi3d_groupnorm_unit_stats(p->out, p->N, p->M / p->gn_rows, (int64_t)p->gn_rows * (p->out_up ? 4 : 1), p->gn_unit,
                                   p->gn_stats, stream);
}

extern "C" int hi3d_gemm(const hi3d_gemm_params* p, void* stream) { return gemm_mma(p, nullptr, 0, stream); }

extern "C" int hi3d_gemm_det(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream) {
  if (!partials) { set_error("hi3d_gemm_det: null partials table"); return -2; }
  return gemm_mma(p, partials, partials_floats, stream);
}

extern "C" const char* hi3d_last_error(void) { return hi3d::g_err; }
extern "C" int64_t hi3d_launch_count(void) { return (int64_t)hi3d::g_launches.load(); }
extern "C" int hi3d_abi_version(void) { return 2; }   // 2: hi3d_gemm_params gained gn_stats / gn_unit / gn_rows

extern "C" int hi3d_device_info(int* sm_count, int* cc_major, int* cc_minor, int* max_smem_optin) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return -1; }
  cudaDeviceProp pr;
  e = cudaGetDeviceProperties(&pr, dev);
  if (e != cudaSuccess) { set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e)); return -1; }
  if (sm_count) *sm_count = pr.multiProcessorCount;
  if (cc_major) *cc_major = pr.major;
  if (cc_minor) *cc_minor = pr.minor;
  if (max_smem_optin) *max_smem_optin = (int)pr.sharedMemPerBlockOptin;
  return 0;
}
