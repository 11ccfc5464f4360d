// GroupNorm(32) [+SiLU] and LayerNorm for channels-last fp16 activations.  Statistics in fp32 (final
// combine in fp64), matching the reference's fp32 GroupNorm32 / autocast-fp32 LayerNorm (SURVEY App. E).
// Both are pure HBM streams: every thread owns fixed 16-byte channel columns, keeps its per-channel
// constants in registers and walks rows with several independent 16-byte loads in flight; grids are sized to a
// few full waves of the 148 SMs.
#include "common.cuh"

namespace hi3d {

constexpr int GN_MAX_CHUNKS = 512;
constexpr int GN_GROUPS = 32;
constexpr int GN_UNROLL = 4;
constexpr int GN_TARGET_CTAS = 148 * 4 * 4;   // ~4 waves at 4 CTAs/SM

HI3D_DEVINL Half8 ld_stream(const __half* p) {
  Half8 v;
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "l"(p));
  *reinterpret_cast<uint4*>(&v) = u;
  return v;
}

// ---- pass 1: per-(sample, chunk, group) partial sum / sum of squares -------------------------------
// grid (chunks, n_samples); blockDim = RL * CV where CV = C/8 vector-columns.
// DET: the per-CTA group sums are formed in a fixed order (per-thread channel sums staged in shared memory, then one thread per
// (group, sum | sumsq) adds them channel-major, row-lane-minor) instead of shared-memory float atomics.
template <bool DET>
__global__ void __launch_bounds__(512)
gn_stats_kernel(const __half* __restrict__ x1, int C1, const __half* __restrict__ x2, int C2, long long rows_per_sample,
                long long rows_per_chunk, float* __restrict__ ws) {
  __shared__ float sg[GN_GROUPS * 2];
  const int C = C1 + C2, CV = C >> 3, cpg = C / GN_GROUPS;
  const int tid = threadIdx.x;
  if (tid < GN_GROUPS * 2) sg[tid] = 0.f;
  __syncthreads();
  const int cv = tid % CV, rl = tid / CV, RL = blockDim.x / CV;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const long long r0 = (long long)chunk * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > rows_per_sample) r1 = rows_per_sample;
  const int c0 = cv * 8;
  const __half* base;
  int ld;
  if (c0 < C1) { base = x1 + c0; ld = C1; } else { base = x2 + (c0 - C1); ld = C2; }
  base += (long long)n * rows_per_sample * ld;
  float s[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; e++) s[e] = q[e] = 0.f;
  long long r = r0 + rl;
  for (; r + (long long)(GN_UNROLL - 1) * RL < r1; r += (long long)GN_UNROLL * RL) {
    Half8 v[GN_UNROLL];
#pragma unroll
    for (int u = 0; u < GN_UNROLL; u++) v[u] = ld_stream(base + (r + (long long)u * RL) * ld);
#pragma unroll
    for (int u = 0; u < GN_UNROLL; u++)
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float2 f = __half22float2(v[u].h[k]);
        s[2 * k] += f.x; q[2 * k] += f.x * f.x;
        s[2 * k + 1] += f.y; q[2 * k + 1] += f.y * f.y;
      }
  }
  for (; r < r1; r += RL) {
    const Half8 v = ld_stream(base + r * ld);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const float2 f = __half22float2(v.h[k]);
      s[2 * k] += f.x; q[2 * k] += f.x * f.x;
      s[2 * k + 1] += f.y; q[2 * k + 1] += f.y * f.y;
    }
  }
  if constexpr (DET) {
    __shared__ float sch[2][512 * 8];           // [s | q][rl * C + channel]
#pragma unroll
    for (int e = 0; e < 8; e++) { sch[0][rl * C + c0 + e] = s[e]; sch[1][rl * C + c0 + e] = q[e]; }
    __syncthreads();
    if (tid < GN_GROUPS * 2) {
      const int g = tid >> 1, which = tid & 1;
      float acc = 0.f;
      for (int c = g * cpg; c < (g + 1) * cpg; c++)
        for (int l = 0; l < RL; l++) acc += sch[which][l * C + c];
      ws[((long long)n * GN_MAX_CHUNKS + chunk) * (GN_GROUPS * 2) + tid] = acc;
    }
    return;
  }
  // fold the 8 channels into their groups (a vector may straddle a group boundary when cpg % 8 != 0)
  int gcur = c0 / cpg;
  float as = 0.f, aq = 0.f;
#pragma unroll
  for (int e = 0; e < 8; e++) {
    const int gi = (c0 + e) / cpg;
    if (gi != gcur) {
      atomicAdd(&sg[2 * gcur], as); atomicAdd(&sg[2 * gcur + 1], aq);
      as = aq = 0.f; gcur = gi;
    }
    as += s[e]; aq += q[e];
  }
  atomicAdd(&sg[2 * gcur], as); atomicAdd(&sg[2 * gcur + 1], aq);
  __syncthreads();
  if (tid < GN_GROUPS * 2) ws[((long long)n * GN_MAX_CHUNKS + chunk) * (GN_GROUPS * 2) + tid] = sg[tid];
}

// ---- pass 1b: combine the chunk partials of one sample into (sum, sum of squares) per group ----------------
// grid (n_samples), 1024 threads; result at fin[n][32][2].  (Frame-sharded runs all-reduce `fin` across ranks here.)
// DET: the 16 per-thread partials of a value are added in thread order instead of with shared-memory atomics.
template <bool DET>
__global__ void __launch_bounds__(1024)
gn_finalize_kernel(const float* __restrict__ ws, int nchunks, float* __restrict__ fin) {
  __shared__ float stot[GN_GROUPS * 2];
  const int tid = threadIdx.x, n = blockIdx.x;
  if (tid < GN_GROUPS * 2) stot[tid] = 0.f;
  __syncthreads();
  const float* w = ws + (long long)n * GN_MAX_CHUNKS * (GN_GROUPS * 2);
  // thread owns value index tid % 64 and chunks tid/64, +16, ...; 4 independent loads in flight per thread
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int c = tid >> 6;
  for (; c + 48 < nchunks; c += 64) {
    a0 += w[c * (GN_GROUPS * 2) + (tid & 63)];
    a1 += w[(c + 16) * (GN_GROUPS * 2) + (tid & 63)];
    a2 += w[(c + 32) * (GN_GROUPS * 2) + (tid & 63)];
    a3 += w[(c + 48) * (GN_GROUPS * 2) + (tid & 63)];
  }
  for (; c < nchunks; c += 16) a0 += w[c * (GN_GROUPS * 2) + (tid & 63)];
  if constexpr (DET) {
    __shared__ float spart[16][GN_GROUPS * 2];
    spart[tid >> 6][tid & 63] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (tid < GN_GROUPS * 2) {
      float acc = 0.f;
      for (int k = 0; k < 16; k++) acc += spart[k][tid];
      fin[(long long)n * (GN_GROUPS * 2) + tid] = acc;
    }
    return;
  }
  atomicAdd(&stot[tid & 63], (a0 + a1) + (a2 + a3));
  __syncthreads();
  if (tid < GN_GROUPS * 2) fin[(long long)n * (GN_GROUPS * 2) + tid] = stot[tid];
}

// ---- pass 2: y = [silu]((x - mean) * rstd * gamma + beta) ------------------------------------------
// grid (row_slabs, n_samples), blockDim = RL * CV.
template <bool HALO>      // HALO = haloed output with peer stores / boundary zero fill (frame-sharded temporal GroupNorm only):
                          // a template so that the dense kernel keeps its 64 registers (2 CTAs per SM)
__global__ void __launch_bounds__(512)
gn_apply_kernel(const __half* __restrict__ x1, int C1, const __half* __restrict__ x2, int C2, long long rows_per_sample,
                long long rows_per_cta, const float* __restrict__ fin, double count, float eps,
                const float* __restrict__ gamma, const float* __restrict__ beta, int apply_silu, __half* __restrict__ y,
                long long y_sample_rows, long long y_row_off, __half* __restrict__ y_prev, __half* __restrict__ y_next,
                long long frame_rows, int zero_lead, int zero_trail, const float* __restrict__ stats1,
                const float* __restrict__ stats2, int unit, int ips) {
  __shared__ float smean[GN_GROUPS], srstd[GN_GROUPS];
  __shared__ float ssum[GN_GROUPS * 2];
  const int C = C1 + C2, CV = C >> 3, cpg = C / GN_GROUPS;
  const int tid = threadIdx.x, n = blockIdx.y;
  if (stats1 != nullptr) {
    // statistics from the unit tables the producing GEMM epilogues accumulated (hi3d_gemm_params::gn_stats): group g of
    // sample n = units [g cpg / unit, (g+1) cpg / unit) of the channel concat, over the `ips` images of the sample.
    // 64 threads, one per (group, sum | sumsq), each adding its <= ips * upg table entries in registers (independent loads).
    if (tid < GN_GROUPS * 2) {
      const int g = tid >> 1, which = tid & 1;
      const int upg = cpg / unit, u1 = C1 / unit, u2 = C2 / unit;
      float acc = 0.f;
      for (int img = 0; img < ips; img++) {
        const long long im = (long long)n * ips + img;
        for (int uu = 0; uu < upg; uu++) {
          const int u = g * upg + uu;
          acc += (u < u1) ? __ldg(stats1 + (im * u1 + u) * 2 + which) : __ldg(stats2 + (im * u2 + (u - u1)) * 2 + which);
        }
      }
      ssum[tid] = acc;
    }
    __syncthreads();
    fin = ssum - (long long)n * (GN_GROUPS * 2);                   // so that the indexing below reads ssum[...]
  }
  if (tid < GN_GROUPS) {      // `count` = elements per (sample, group) over ALL ranks
    const double mean = (double)fin[(long long)n * (GN_GROUPS * 2) + 2 * tid] / count;
    double var = (double)fin[(long long)n * (GN_GROUPS * 2) + 2 * tid + 1] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    smean[tid] = (float)mean;
    srstd[tid] = (float)(1.0 / sqrt(var + (double)eps));
  }
  __syncthreads();
  const int cv = tid % CV, rl = tid / CV, RL = blockDim.x / CV;
  const int c0 = cv * 8;
  float A[8], B[8];
#pragma unroll
  for (int e = 0; e < 8; e++) {
    const int c = c0 + e, g = c / cpg;
    A[e] = srstd[g] * gamma[c];
    B[e] = beta[c] - smean[g] * A[e];
  }
  const __half* base;
  int ld;
  if (c0 < C1) { base = x1 + c0; ld = C1; } else { base = x2 + (c0 - C1); ld = C2; }
  const long long srow0 = (long long)n * rows_per_sample;
  base += srow0 * ld;
  __half* yb = y + ((long long)n * y_sample_rows + y_row_off) * C + c0;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta;
  if (r1 > rows_per_sample) r1 = rows_per_sample;
  // (A variant with one shared reciprocal per four sigmoids -- 1.25 MUFU operations per element instead of 2 -- was measured
  // SLOWER: 128 us vs 76 us per launch in the ncu launch list of profiles/r02_*: the kernel is latency-bound at ~50 % issue /
  // MUFU / DRAM utilisation, and the extra multiplies plus the register squeeze cost more than the MUFU slots they free.)
  auto xform = [&](Half8 v) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      float2 f = __half22float2(v.h[k]);
      f.x = f.x * A[2 * k] + B[2 * k];
      f.y = f.y * A[2 * k + 1] + B[2 * k + 1];
      if (apply_silu) { f.x = silu_f(f.x); f.y = silu_f(f.y); }
      v.h[k] = __floats2half2_rn(f.x, f.y);
    }
    return v;
  };
  // Frame-sharded temporal GroupNorm (SURVEY 8e): y is a haloed [n, T_local + 2, frame_rows, C] buffer.  The first local
  // frame is ALSO stored into the trailing halo slot of the previous rank's buffer and the last local frame into the leading
  // halo slot of the next rank's (peer stores over NVLink): the one-frame halo exchange of the (3,1,1) conv rides on this
  // kernel's stores.  y_prev / y_next are the peers' buffer bases (NULL at the clip boundary: that slot stays zero = padding).
  const long long last0 = rows_per_sample - frame_rows;
  __half* yp = (HALO && y_prev) ? y_prev + ((long long)n * y_sample_rows + (y_sample_rows - frame_rows)) * C + c0 : nullptr;
  __half* yn = (HALO && y_next) ? y_next + ((long long)n * y_sample_rows - last0) * C + c0 : nullptr;
  // At a clip boundary (no previous / next rank) the halo slot of THIS rank is the Conv3d zero padding: the buffer is
  // shared by layers of different geometry, so it is re-zeroed here by the threads that own the matching boundary frame.
  __half* zl = (HALO && zero_lead) ? y + ((long long)n * y_sample_rows) * C + c0 : nullptr;                     // slot 0
  __half* zt = (HALO && zero_trail) ? y + ((long long)n * y_sample_rows + (y_sample_rows - frame_rows) - last0) * C + c0 : nullptr;
  Half8 zero8;
  zero8.u = make_uint4(0u, 0u, 0u, 0u);
  bool remote = false;
  auto put = [&](long long rr, const Half8& o) {
    *reinterpret_cast<Half8*>(yb + rr * C) = o;
    if (!HALO) return;
    if (rr < frame_rows) {
      if (yp != nullptr) { *reinterpret_cast<Half8*>(yp + rr * C) = o; remote = true; }
      if (zl != nullptr) *reinterpret_cast<Half8*>(zl + rr * C) = zero8;
    }
    if (rr >= last0) {
      if (yn != nullptr) { *reinterpret_cast<Half8*>(yn + rr * C) = o; remote = true; }
      if (zt != nullptr) *reinterpret_cast<Half8*>(zt + rr * C) = zero8;
    }
  };
  long long r = r0 + rl;
  for (; r + (long long)(GN_UNROLL - 1) * RL < r1; r += (long long)GN_UNROLL * RL) {
    Half8 v[GN_UNROLL];
#pragma unroll
    for (int u = 0; u < GN_UNROLL; u++) v[u] = ld_stream(base + (r + (long long)u * RL) * ld);
#pragma unroll
    for (int u = 0; u < GN_UNROLL; u++) put(r + (long long)u * RL, xform(v[u]));
  }
  for (; r < r1; r += RL) put(r, xform(ld_stream(base + r * ld)));
  if (remote) __threadfence_system();
}

// ---- LayerNorm: LPR lanes per row (32/LPR rows per warp pass), VPL 16-byte vectors per lane ------------------
// C = 8 * VPL * LPR exactly (C = 320 -> VPL 5, LPR 8; 640 -> 5 x 16; 1280 -> 5 x 32; 64 -> 1 x 8; 2560 -> 10 x 32).
template <int VPL, int LPR>
__global__ void __launch_bounds__(256)
layernorm_kernel(const __half* __restrict__ x, const __half* __restrict__ addvec, int add_div, int add_mod, long long M,
                 int C, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                 __half* __restrict__ y) {
  constexpr int RPW = 32 / LPR;                      // rows per warp pass
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR, rsel = lane / LPR;
  const long long wrow0 = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * RPW;
  const long long m = wrow0 + rsel;
  const bool live = m < M;
  const float invC = 1.f / (float)C;
  Half8 raw[VPL];
  if (live) {
#pragma unroll
    for (int i = 0; i < VPL; i++) raw[i] = ld_stream(x + m * C + (sub + LPR * i) * 8);
  }
  float v[VPL][8];
  float sum = 0.f;
  if (live) {
    const __half* av = addvec ? addvec + (long long)((m / add_div) % add_mod) * C : nullptr;
#pragma unroll
    for (int i = 0; i < VPL; i++) {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float2 f = __half22float2(raw[i].h[k]);
        v[i][2 * k] = f.x; v[i][2 * k + 1] = f.y;
      }
      if (av) {
        const Half8 a = *reinterpret_cast<const Half8*>(av + (sub + LPR * i) * 8);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float2 f = __half22float2(a.h[k]);
          v[i][2 * k] += f.x; v[i][2 * k + 1] += f.y;
        }
      }
#pragma unroll
      for (int e = 0; e < 8; e++) sum += v[i][e];
    }
  } else {
#pragma unroll
    for (int i = 0; i < VPL; i++)
#pragma unroll
      for (int e = 0; e < 8; e++) v[i][e] = 0.f;
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * invC;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; i++)
#pragma unroll
    for (int e = 0; e < 8; e++) { const float d = v[i][e] - mean; sq += d * d; }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq * invC + eps);
  if (live) {
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      const int c0 = (sub + LPR * i) * 8;
      Half8 o;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float2 gm = *reinterpret_cast<const float2*>(gamma + c0 + 2 * k);
        const float2 bt = *reinterpret_cast<const float2*>(beta + c0 + 2 * k);
        o.h[k] = __floats2half2_rn((v[i][2 * k] - mean) * rstd * gm.x + bt.x, (v[i][2 * k + 1] - mean) * rstd * gm.y + bt.y);
      }
      *reinterpret_cast<Half8*>(y + m * C + c0) = o;
    }
  }
}

// generic fallback: one warp per row, up to 10 vectors per lane with masking (any C % 8 == 0, C <= 2560)
template <int VPL>
__global__ void __launch_bounds__(256)
layernorm_generic_kernel(const __half* __restrict__ x, const __half* __restrict__ addvec, int add_div, int add_mod,
                         long long M, int C, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                         __half* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long m = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  const int CV = C >> 3;
  const __half* av = addvec ? addvec + (long long)((m / add_div) % add_mod) * C : nullptr;
  float v[VPL][8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    const int cv = lane + 32 * i;
#pragma unroll
    for (int e = 0; e < 8; e++) v[i][e] = 0.f;
    if (cv < CV) {
      const Half8 h = ld_stream(x + m * C + cv * 8);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float2 f = __half22float2(h.h[k]);
        v[i][2 * k] = f.x; v[i][2 * k + 1] = f.y;
      }
      if (av) {
        const Half8 a = *reinterpret_cast<const Half8*>(av + cv * 8);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float2 f = __half22float2(a.h[k]);
          v[i][2 * k] += f.x; v[i][2 * k + 1] += f.y;
        }
      }
#pragma unroll
      for (int e = 0; e < 8; e++) sum += v[i][e];
    }
  }
  const float mean = warp_sum(sum) / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; i++)
    if (lane + 32 * i < CV) {
#pragma unroll
      for (int e = 0; e < 8; e++) { const float d = v[i][e] - mean; sq += d * d; }
    }
  const float rstd = rsqrtf(warp_sum(sq) / (float)C + eps);
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    const int cv = lane + 32 * i;
    if (cv < CV) {
      Half8 o;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int c = cv * 8 + 2 * k;
        o.h[k] = __floats2half2_rn((v[i][2 * k] - mean) * rstd * gamma[c] + beta[c],
                                   (v[i][2 * k + 1] - mean) * rstd * gamma[c + 1] + beta[c + 1]);
      }
      *reinterpret_cast<Half8*>(y + m * C + cv * 8) = o;
    }
  }
}

}  // namespace hi3d

using namespace hi3d;

extern "C" int64_t hi3d_groupnorm_ws_floats(int n_samples) {
  return (int64_t)n_samples * (GN_MAX_CHUNKS + 1) * GN_GROUPS * 2;     // chunk partials + final (mean, rstd)
}

static int gn_check(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample, const char* who) {
  const int C = C1 + C2;
  if (!x1 || n_samples <= 0 || rows_per_sample <= 0 || C1 <= 0 || (C1 % 8) || (C2 % 8) || (C % GN_GROUPS) || C > 4096 ||
      ((uintptr_t)x1 & 15) || (x2 && ((uintptr_t)x2 & 15)) || n_samples > 65535) {
    set_error("%s: bad arguments (C1=%d C2=%d n=%d rows=%lld)", who, C1, C2, n_samples, (long long)rows_per_sample);
    return -2;
  }
  return 0;
}

// (sum, sum of squares) per (sample, group) of the LOCAL rows -> sums[n_samples][32][2] (fp32)
template <bool DET>
static int groupnorm_sums(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample, float* sums,
                          float* ws, void* stream) {
  if (!x2) C2 = 0;
  int rc = gn_check(x1, C1, x2, C2, n_samples, rows_per_sample, "hi3d_groupnorm_sums");
  if (rc) return rc;
  if (!sums || !ws) { set_error("hi3d_groupnorm_sums: null output / workspace"); return -2; }
  cudaStream_t st = (cudaStream_t)stream;
  const int C = C1 + C2, CV = C / 8;
  const int threads = (512 / CV) * CV;
  const int RL = threads / CV;
  const long long min_rows = (long long)RL * GN_UNROLL;     // one unrolled sweep per thread at least
  long long chunks = (GN_TARGET_CTAS + n_samples - 1) / n_samples;
  const long long max_by_rows = (rows_per_sample + min_rows - 1) / min_rows;
  if (chunks > max_by_rows) chunks = max_by_rows;
  if (chunks > GN_MAX_CHUNKS) chunks = GN_MAX_CHUNKS;
  if (chunks < 1) chunks = 1;
  long long rpc = (rows_per_sample + chunks - 1) / chunks;
  rpc = (rpc + RL - 1) / RL * RL;
  chunks = (rows_per_sample + rpc - 1) / rpc;
  gn_stats_kernel<DET><<<dim3((unsigned)chunks, n_samples), threads, 0, st>>>((const __half*)x1, C1, (const __half*)x2, C2,
                                                                        rows_per_sample, rpc, ws);
  rc = check_launch("hi3d_groupnorm_sums(stats)");
  if (rc) return rc;
  gn_finalize_kernel<DET><<<n_samples, 1024, 0, st>>>(ws, (int)chunks, sums);
  return check_launch("hi3d_groupnorm_sums(finalize)");
}

extern "C" int hi3d_groupnorm_sums(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                                   float* sums, float* ws, void* stream) {
  return groupnorm_sums<false>(x1, C1, x2, C2, n_samples, rows_per_sample, sums, ws, stream);
}

extern "C" int hi3d_groupnorm_sums_det(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                                       float* sums, float* ws, void* stream) {
  return groupnorm_sums<true>(x1, C1, x2, C2, n_samples, rows_per_sample, sums, ws, stream);
}

// hi3d_groupnorm_apply_stats routes through the same launcher; its extra arguments travel in these thread-locals
static thread_local const float* g_apply_stats1 = nullptr;
static thread_local const float* g_apply_stats2 = nullptr;
static thread_local int g_apply_unit = 0, g_apply_ips = 1;

// y = [silu]((x - mean) * rstd * gamma + beta) with mean / rstd from `sums` over `count_rows` rows per sample
// (count_rows = rows_per_sample for a single GPU, the GLOBAL row count when the sums were all-reduced over ranks).
// Sample n of y starts at row n * y_sample_rows + y_row_off (haloed temporal buffers); 0, 0 -> dense like x.
extern "C" int hi3d_groupnorm_apply(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                                    const float* sums, int64_t count_rows, const float* gamma, const float* beta, float eps,
                                    int apply_silu, void* y, int64_t y_sample_rows, int64_t y_row_off, void* stream) {
  return hi3d_groupnorm_apply_halo(x1, C1, x2, C2, n_samples, rows_per_sample, sums, count_rows, gamma, beta, eps, apply_silu,
                                   y, y_sample_rows, y_row_off, nullptr, nullptr, 0, stream);
}

extern "C" int hi3d_groupnorm_apply_halo(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                                         const float* sums, int64_t count_rows, const float* gamma, const float* beta, float eps,
                                         int apply_silu, void* y, int64_t y_sample_rows, int64_t y_row_off, void* y_prev_rank,
                                         void* y_next_rank, int64_t frame_rows, void* stream) {
  // frame_rows > 0 selects the haloed form: a NULL neighbour then means "clip boundary", whose local halo slot is zero-filled
  if (!x2) C2 = 0;
  int rc = gn_check(x1, C1, x2, C2, n_samples, rows_per_sample, "hi3d_groupnorm_apply");
  if (rc) return rc;
  if ((y_prev_rank || y_next_rank || frame_rows > 0) &&
      (frame_rows <= 0 || rows_per_sample % frame_rows || y_sample_rows != rows_per_sample + 2 * frame_rows ||
       y_row_off != frame_rows || ((uintptr_t)y_prev_rank & 15) || ((uintptr_t)y_next_rank & 15))) {
    set_error("hi3d_groupnorm_apply_halo: the peer halo stores need y = [n, T_local + 2, frame_rows, C] with y_row_off = "
              "frame_rows (rows %lld, frame_rows %lld, y_sample_rows %lld, y_row_off %lld)", (long long)rows_per_sample,
              (long long)frame_rows, (long long)y_sample_rows, (long long)y_row_off);
    return -2;
  }
  if ((!sums && !g_apply_stats1) || !gamma || !beta || !y || ((uintptr_t)y & 15) || count_rows <= 0) {
    set_error("hi3d_groupnorm_apply: bad arguments");
    return -2;
  }
  if (y_sample_rows <= 0) { y_sample_rows = rows_per_sample; y_row_off = 0; }
  cudaStream_t st = (cudaStream_t)stream;
  const int C = C1 + C2, CV = C / 8;
  const int threads = (512 / CV) * CV;
  const int RL = threads / CV;
  const long long min_rows = (long long)RL * GN_UNROLL;
  const long long max_by_rows = (rows_per_sample + min_rows - 1) / min_rows;
  // 2 CTAs per SM x 3 waves: a CTA lives ~4x longer than with the statistics kernels' grid, so its prologue (group statistics
  // -> mean / rstd -> 16 coefficient registers) is amortised; measured 120 -> see profiles/r02 launch lists
  long long slabs = (148 * 2 * 3 + n_samples - 1) / n_samples;
  if (slabs > max_by_rows) slabs = max_by_rows;
  if (slabs < 1) slabs = 1;
  long long rows_per_cta = (rows_per_sample + slabs - 1) / slabs;
  rows_per_cta = (rows_per_cta + RL - 1) / RL * RL;
  slabs = (rows_per_sample + rows_per_cta - 1) / rows_per_cta;
  if (slabs > 2147483647LL) { set_error("hi3d_groupnorm_apply: too many slabs"); return -2; }
  if (frame_rows > 0)
    gn_apply_kernel<true><<<dim3((unsigned)slabs, n_samples), threads, 0, st>>>(
        (const __half*)x1, C1, (const __half*)x2, C2, rows_per_sample, rows_per_cta, sums,
        (double)count_rows * (double)(C / GN_GROUPS), eps, gamma, beta, apply_silu, (__half*)y, y_sample_rows, y_row_off,
        (__half*)y_prev_rank, (__half*)y_next_rank, frame_rows, !y_prev_rank ? 1 : 0, !y_next_rank ? 1 : 0, g_apply_stats1,
        g_apply_stats2, g_apply_unit, g_apply_ips);
  else
    gn_apply_kernel<false><<<dim3((unsigned)slabs, n_samples), threads, 0, st>>>(
        (const __half*)x1, C1, (const __half*)x2, C2, rows_per_sample, rows_per_cta, sums,
        (double)count_rows * (double)(C / GN_GROUPS), eps, gamma, beta, apply_silu, (__half*)y, y_sample_rows, y_row_off,
        nullptr, nullptr, 0, 0, 0, g_apply_stats1, g_apply_stats2, g_apply_unit, g_apply_ips);
  return check_launch("hi3d_groupnorm_apply");
}

// ---- unit statistics of an existing tensor: (sum, sumsq) per image and per `unit` consecutive channels, accumulated -------
// grid (chunks, n_images); same streaming pattern as gn_stats_kernel, folding into units instead of the 32 groups.
// DET: no atomics -- the CTA's unit sums are formed in a fixed order (as in gn_stats_kernel<true>) and STORED into its own
// partials slot, stats = fp32 [n_images, chunks, units, 2]; gn_fold_kernel then sums the slots of an image in chunk order.
constexpr int GN_MAX_UNITS = 256;
template <bool DET>
__global__ void __launch_bounds__(512)
gn_unit_stats_kernel(const __half* __restrict__ x, int C, long long rows_per_image, long long rows_per_chunk, int unit,
                     float* __restrict__ stats) {
  __shared__ float su[GN_MAX_UNITS * 2];
  const int CV = C >> 3, nu = C / unit;
  const int tid = threadIdx.x;
  for (int i = tid; i < nu * 2; i += blockDim.x) su[i] = 0.f;
  __syncthreads();
  const int cv = tid % CV, rl = tid / CV, RL = blockDim.x / CV;
  const int n = blockIdx.y;
  const long long r0 = (long long)blockIdx.x * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > rows_per_image) r1 = rows_per_image;
  const int c0 = cv * 8;
  const __half* base = x + (long long)n * rows_per_image * C + c0;
  float s[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; e++) s[e] = q[e] = 0.f;
  // four independent 16-byte loads in flight per thread (a read-only stream: memory-level parallelism is the whole game)
  long long r = r0 + rl;
  for (; r + 3LL * RL < r1; r += 4LL * RL) {
    Half8 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = ld_stream(base + (r + (long long)u * RL) * C);
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float2 f = __half22float2(v[u].h[k]);
        s[2 * k] += f.x; q[2 * k] += f.x * f.x;
        s[2 * k + 1] += f.y; q[2 * k + 1] += f.y * f.y;
      }
  }
  for (; r < r1; r += RL) {
    const Half8 v = ld_stream(base + r * C);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const float2 f = __half22float2(v.h[k]);
      s[2 * k] += f.x; q[2 * k] += f.x * f.x;
      s[2 * k + 1] += f.y; q[2 * k + 1] += f.y * f.y;
    }
  }
  if constexpr (DET) {
    __shared__ float sch[2][512 * 8];           // [s | q][rl * C + channel]
#pragma unroll
    for (int e = 0; e < 8; e++) { sch[0][rl * C + c0 + e] = s[e]; sch[1][rl * C + c0 + e] = q[e]; }
    __syncthreads();
    float* slot = stats + ((long long)n * gridDim.x + blockIdx.x) * nu * 2;
    for (int i = tid; i < nu * 2; i += blockDim.x) {
      const int u = i >> 1, which = i & 1;
      float acc = 0.f;
      for (int c = u * unit; c < (u + 1) * unit; c++)
        for (int l = 0; l < RL; l++) acc += sch[which][l * C + c];
      slot[i] = acc;
    }
    return;
  }
  int ucur = c0 / unit;
  float as = 0.f, aq = 0.f;
#pragma unroll
  for (int e = 0; e < 8; e++) {
    const int ui = (c0 + e) / unit;
    if (ui != ucur) {
      atomicAdd(&su[2 * ucur], as); atomicAdd(&su[2 * ucur + 1], aq);
      as = aq = 0.f; ucur = ui;
    }
    as += s[e]; aq += q[e];
  }
  atomicAdd(&su[2 * ucur], as); atomicAdd(&su[2 * ucur + 1], aq);
  __syncthreads();
  for (int i = tid; i < nu * 2; i += blockDim.x) atomicAdd(&stats[(long long)n * nu * 2 + i], su[i]);
}

// unit tables -> (sum, sumsq) per (sample, group): sums[n][32][2]
// DET: one thread per (group, sum | sumsq) adds its table entries image-major, unit-minor (the order of the gn_apply prologue).
template <bool DET>
__global__ void __launch_bounds__(256)
gn_group_sums_kernel(const float* __restrict__ stats1, int C1, const float* __restrict__ stats2, int C2, int unit, int ips,
                     float* __restrict__ sums) {
  __shared__ float ssum[GN_GROUPS * 2];
  const int tid = threadIdx.x, n = blockIdx.x;
  if constexpr (DET) {
    if (tid < GN_GROUPS * 2) {
      const int g = tid >> 1, which = tid & 1;
      const int upg = (C1 + C2) / GN_GROUPS / unit, u1 = C1 / unit, u2 = C2 / unit;
      float acc = 0.f;
      for (int img = 0; img < ips; img++) {
        const long long im = (long long)n * ips + img;
        for (int uu = 0; uu < upg; uu++) {
          const int u = g * upg + uu;
          acc += (u < u1) ? stats1[(im * u1 + u) * 2 + which] : stats2[(im * u2 + (u - u1)) * 2 + which];
        }
      }
      sums[(long long)n * (GN_GROUPS * 2) + tid] = acc;
    }
    return;
  }
  if (tid < GN_GROUPS * 2) ssum[tid] = 0.f;
  __syncthreads();
  const int cpg = (C1 + C2) / GN_GROUPS, upg = cpg / unit, u1 = C1 / unit, u2 = C2 / unit;
  const int items = GN_GROUPS * ips * upg;
  for (int it = tid; it < items; it += blockDim.x) {
    const int g = it / (ips * upg), rem = it - g * (ips * upg);
    const int img = rem / upg, uu = rem - img * upg;
    const int u = g * upg + uu;
    const long long im = (long long)n * ips + img;
    const float* src = (u < u1) ? stats1 + (im * u1 + u) * 2 : stats2 + (im * u2 + (u - u1)) * 2;
    atomicAdd(&ssum[2 * g], src[0]);
    atomicAdd(&ssum[2 * g + 1], src[1]);
  }
  __syncthreads();
  if (tid < GN_GROUPS * 2) sums[(long long)n * (GN_GROUPS * 2) + tid] = ssum[tid];
}

// ---- fold: partials table -> unit table [n_images, units, 2], OVERWRITTEN --------------------------------------------------
// grid (units, n_images), GN_FOLD_THREADS threads.  Thread t adds the slots t, t + GN_FOLD_THREADS, ... in fp64, then a fixed
// shared-memory tree combines the threads: the order depends on the shapes only.  Two slot layouts:
//   octets = 0: [n_images][nblk][units][2]            (gn_unit_stats_kernel<true>: one slot per (image, chunk))
//   octets = 1: [n_images][nblk][C / 8][4]             (gemm_tc5 deterministic epilogue: one slot per (image, 32-row block,
//               8-channel octet) = (sum, sumsq) of the octet's first unit, then of the next unit it reaches into (unit >= 4))
constexpr int GN_FOLD_THREADS = 128;
__global__ void __launch_bounds__(GN_FOLD_THREADS)
gn_fold_kernel(const float* __restrict__ part, int nblk, int octets, int C, int unit, float* __restrict__ stats) {
  __shared__ double red[2][GN_FOLD_THREADS];
  const int u = blockIdx.x, n = blockIdx.y, nu = C / unit, tid = threadIdx.x;
  double as = 0.0, aq = 0.0;
  if (octets) {
    const int noct = C / 8, o0 = (u * unit) / 8, o1 = ((u + 1) * unit - 1) / 8;
    const float* base = part + (long long)n * nblk * noct * 4;
    for (int b = tid; b < nblk; b += GN_FOLD_THREADS)
      for (int o = o0; o <= o1; o++) {
        const int side = ((o * 8) / unit == u) ? 0 : 2;     // the octet's first unit, or the one after it
        const float2 v = *reinterpret_cast<const float2*>(base + ((long long)b * noct + o) * 4 + side);
        as += (double)v.x; aq += (double)v.y;
      }
  } else {
    const float* base = part + (long long)n * nblk * nu * 2 + u * 2;
    for (int b = tid; b < nblk; b += GN_FOLD_THREADS) {
      as += (double)base[(long long)b * nu * 2];
      aq += (double)base[(long long)b * nu * 2 + 1];
    }
  }
  red[0][tid] = as; red[1][tid] = aq;
  __syncthreads();
#pragma unroll
  for (int h = GN_FOLD_THREADS / 2; h > 0; h >>= 1) {
    if (tid < h) { red[0][tid] += red[0][tid + h]; red[1][tid] += red[1][tid + h]; }
    __syncthreads();
  }
  if (tid == 0) {
    stats[((long long)n * nu + u) * 2] = (float)red[0][0];
    stats[((long long)n * nu + u) * 2 + 1] = (float)red[1][0];
  }
}

static int unit_check(int C1, int C2, int unit, const char* who) {
  const int C = C1 + C2;
  if (unit <= 0 || (C % GN_GROUPS) || ((C / GN_GROUPS) % unit) || (C1 % unit) || (C2 % unit) || C1 / unit > GN_MAX_UNITS ||
      C2 / unit > GN_MAX_UNITS) {
    set_error("%s: unit %d must divide C1 = %d, C2 = %d and the channels per group %d (at most %d units per tensor)", who, unit,
              C1, C2, C / GN_GROUPS, GN_MAX_UNITS);
    return -2;
  }
  return 0;
}

// grid of gn_unit_stats_kernel: `chunks` CTAs of `threads` per image, rpc rows each
static long long unit_stats_grid(int C, int n_images, int64_t rows_per_image, int* threads_out, long long* rpc_out) {
  const int CV = C / 8;
  const int threads = (512 / CV) * CV;
  const int RL = threads / CV;
  long long chunks = (GN_TARGET_CTAS + n_images - 1) / n_images;
  const long long max_by_rows = (rows_per_image + RL * GN_UNROLL - 1) / ((long long)RL * GN_UNROLL);
  if (chunks > max_by_rows) chunks = max_by_rows;
  if (chunks < 1) chunks = 1;
  long long rpc = (rows_per_image + chunks - 1) / chunks;
  rpc = (rpc + RL - 1) / RL * RL;
  chunks = (rows_per_image + rpc - 1) / rpc;
  *threads_out = threads;
  *rpc_out = rpc;
  return chunks;
}

static int unit_stats_args(const void* x, int C, int n_images, int64_t rows_per_image, int unit, const float* stats,
                           const char* who) {
  if (!x || !stats || C <= 0 || (C % 8) || n_images <= 0 || n_images > 65535 || rows_per_image <= 0 || unit <= 0 ||
      (C % unit) || C / unit > GN_MAX_UNITS || ((uintptr_t)x & 15)) {
    set_error("%s: bad arguments (C=%d unit=%d n=%d rows=%lld)", who, C, unit, n_images, (long long)rows_per_image);
    return -2;
  }
  return 0;
}

extern "C" int hi3d_groupnorm_unit_stats(const void* x, int C, int n_images, int64_t rows_per_image, int unit, float* stats,
                                         void* stream) {
  int rc = unit_stats_args(x, C, n_images, rows_per_image, unit, stats, "hi3d_groupnorm_unit_stats");
  if (rc) return rc;
  int threads;
  long long rpc;
  const long long chunks = unit_stats_grid(C, n_images, rows_per_image, &threads, &rpc);
  gn_unit_stats_kernel<false><<<dim3((unsigned)chunks, n_images), threads, 0, (cudaStream_t)stream>>>((const __half*)x, C, rows_per_image,
                                                                                              rpc, unit, stats);
  return check_launch("hi3d_groupnorm_unit_stats");
}

extern "C" int64_t hi3d_groupnorm_partials_floats(int n_images, int64_t rows_per_image, int C, int unit) {
  if (n_images <= 0 || rows_per_image <= 0 || C <= 0 || (C % 8) || unit <= 0 || (C % unit)) return 0;
  int threads;
  long long rpc;
  const long long chunks = unit_stats_grid(C, n_images, rows_per_image, &threads, &rpc);
  const int64_t pass = (int64_t)n_images * chunks * (C / unit) * 2;                    // gn_unit_stats_kernel<true>
  const int64_t epi = (int64_t)n_images * ((rows_per_image + 31) / 32) * (C / 8) * 4;   // gemm_tc5 deterministic epilogue
  return pass > epi ? pass : epi;
}

extern "C" int hi3d_groupnorm_fold(const float* partials, int n_images, int blocks_per_image, int octets, int C, int unit,
                                   float* stats, void* stream) {
  if (!partials || !stats || n_images <= 0 || n_images > 65535 || blocks_per_image <= 0 || C <= 0 || (C % 8) || unit <= 0 ||
      (C % unit) || C / unit > GN_MAX_UNITS || (octets && unit < 4)) {
    set_error("hi3d_groupnorm_fold: bad arguments (n=%d blocks=%d C=%d unit=%d)", n_images, blocks_per_image, C, unit);
    return -2;
  }
  gn_fold_kernel<<<dim3((unsigned)(C / unit), n_images), GN_FOLD_THREADS, 0, (cudaStream_t)stream>>>(
      partials, blocks_per_image, octets ? 1 : 0, C, unit, stats);
  return check_launch("hi3d_groupnorm_fold");
}

extern "C" int hi3d_groupnorm_unit_stats_det(const void* x, int C, int n_images, int64_t rows_per_image, int unit, float* stats,
                                             float* partials, int64_t partials_floats, void* stream) {
  int rc = unit_stats_args(x, C, n_images, rows_per_image, unit, stats, "hi3d_groupnorm_unit_stats_det");
  if (rc) return rc;
  int threads;
  long long rpc;
  const long long chunks = unit_stats_grid(C, n_images, rows_per_image, &threads, &rpc);
  if (!partials || partials_floats < (int64_t)n_images * chunks * (C / unit) * 2) {
    set_error("hi3d_groupnorm_unit_stats_det: partials table of %lld floats, %lld needed", (long long)partials_floats,
              (long long)n_images * chunks * (C / unit) * 2);
    return -2;
  }
  gn_unit_stats_kernel<true><<<dim3((unsigned)chunks, n_images), threads, 0, (cudaStream_t)stream>>>((const __half*)x, C,
                                                                                             rows_per_image, rpc, unit, partials);
  rc = check_launch("hi3d_groupnorm_unit_stats_det");
  if (rc) return rc;
  return hi3d_groupnorm_fold(partials, n_images, (int)chunks, 0, C, unit, stats, stream);
}

template <bool DET>
static int group_sums(const float* stats1, int C1, const float* stats2, int C2, int unit, int n_samples, int imgs_per_sample,
                      float* sums, void* stream) {
  if (!stats2) C2 = 0;
  if (!stats1 || !sums || n_samples <= 0 || imgs_per_sample <= 0) { set_error("hi3d_groupnorm_group_sums: bad arguments"); return -2; }
  int rc = unit_check(C1, C2, unit, "hi3d_groupnorm_group_sums");
  if (rc) return rc;
  gn_group_sums_kernel<DET><<<n_samples, 256, 0, (cudaStream_t)stream>>>(stats1, C1, stats2, C2, unit, imgs_per_sample, sums);
  return check_launch("hi3d_groupnorm_group_sums");
}

extern "C" int hi3d_groupnorm_group_sums(const float* stats1, int C1, const float* stats2, int C2, int unit, int n_samples,
                                         int imgs_per_sample, float* sums, void* stream) {
  return group_sums<false>(stats1, C1, stats2, C2, unit, n_samples, imgs_per_sample, sums, stream);
}

extern "C" int hi3d_groupnorm_group_sums_det(const float* stats1, int C1, const float* stats2, int C2, int unit, int n_samples,
                                             int imgs_per_sample, float* sums, void* stream) {
  return group_sums<true>(stats1, C1, stats2, C2, unit, n_samples, imgs_per_sample, sums, stream);
}

extern "C" int hi3d_groupnorm_apply_stats(const void* x1, int C1, const float* stats1, const void* x2, int C2, const float* stats2,
                                          int unit, int n_samples, int64_t rows_per_sample, int imgs_per_sample,
                                          int64_t count_rows, const float* gamma, const float* beta, float eps, int apply_silu,
                                          void* y, int64_t y_sample_rows, int64_t y_row_off, void* y_prev_rank, void* y_next_rank,
                                          int64_t frame_rows, void* stream) {
  if (!x2) { C2 = 0; stats2 = nullptr; }
  if (!stats1 || (x2 && !stats2) || imgs_per_sample <= 0) { set_error("hi3d_groupnorm_apply_stats: null statistics table"); return -2; }
  int rc = unit_check(C1, C2, unit, "hi3d_groupnorm_apply_stats");
  if (rc) return rc;
  g_apply_stats1 = stats1; g_apply_stats2 = stats2; g_apply_unit = unit; g_apply_ips = imgs_per_sample;
  rc = hi3d_groupnorm_apply_halo(x1, C1, x2, C2, n_samples, rows_per_sample, nullptr, count_rows, gamma, beta, eps, apply_silu, y,
                                 y_sample_rows, y_row_off, y_prev_rank, y_next_rank, frame_rows, stream);
  g_apply_stats1 = g_apply_stats2 = nullptr; g_apply_unit = 0; g_apply_ips = 1;
  return rc;
}

template <bool DET>
static int groupnorm_silu(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                          const float* gamma, const float* beta, float eps, int apply_silu, void* y, float* ws, void* stream) {
  if (!ws) { set_error("hi3d_groupnorm_silu: null workspace"); return -2; }
  float* sums = ws + (long long)n_samples * GN_MAX_CHUNKS * GN_GROUPS * 2;
  int rc = groupnorm_sums<DET>(x1, C1, x2, C2, n_samples, rows_per_sample, sums, ws, stream);
  if (rc) return rc;
  return hi3d_groupnorm_apply(x1, C1, x2, C2, n_samples, rows_per_sample, sums, rows_per_sample, gamma, beta, eps, apply_silu,
                              y, 0, 0, stream);
}

extern "C" int hi3d_groupnorm_silu(const void* x1, int C1, const void* x2, int C2, int n_samples,
                                   int64_t rows_per_sample, const float* gamma, const float* beta, float eps,
                                   int apply_silu, void* y, float* ws, void* stream) {
  return groupnorm_silu<false>(x1, C1, x2, C2, n_samples, rows_per_sample, gamma, beta, eps, apply_silu, y, ws, stream);
}

extern "C" int hi3d_groupnorm_silu_det(const void* x1, int C1, const void* x2, int C2, int n_samples,
                                       int64_t rows_per_sample, const float* gamma, const float* beta, float eps,
                                       int apply_silu, void* y, float* ws, void* stream) {
  return groupnorm_silu<true>(x1, C1, x2, C2, n_samples, rows_per_sample, gamma, beta, eps, apply_silu, y, ws, stream);
}

extern "C" int hi3d_layernorm(const void* x, const void* addvec, int add_div, int add_mod, int64_t M, int C,
                              const float* gamma, const float* beta, float eps, void* y, void* stream) {
  if (!x || !y || !gamma || !beta || M <= 0 || C <= 0 || (C % 8) || C > 2560 || ((uintptr_t)x & 15) ||
      ((uintptr_t)y & 15) || ((uintptr_t)gamma & 7) || ((uintptr_t)beta & 7) ||
      (addvec && (add_div <= 0 || add_mod <= 0 || ((uintptr_t)addvec & 15)))) {
    set_error("hi3d_layernorm: bad arguments (M=%lld C=%d)", (long long)M, C);
    return -2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int CV = C / 8;
  const __half* xp = (const __half*)x;
  const __half* ap = (const __half*)addvec;
  __half* yp = (__half*)y;
#define HI3D_LN_LAUNCH(VPL, LPR)                                                                                        \
  do {                                                                                                                  \
    const long long rows_per_cta = 8 * (32 / LPR);                                                                      \
    const long long blocks = (M + rows_per_cta - 1) / rows_per_cta;                                                     \
    if (blocks > 2147483647LL) { set_error("hi3d_layernorm: M too large"); return -2; }                                 \
    layernorm_kernel<VPL, LPR><<<(unsigned)blocks, 256, 0, st>>>(xp, ap, add_div, add_mod, M, C, gamma, beta, eps, yp);  \
  } while (0)
#define HI3D_LN_GENERIC(VPL)                                                                                             \
  do {                                                                                                                  \
    const long long blocks = (M + 7) / 8;                                                                               \
    if (blocks > 2147483647LL) { set_error("hi3d_layernorm: M too large"); return -2; }                                 \
    layernorm_generic_kernel<VPL><<<(unsigned)blocks, 256, 0, st>>>(xp, ap, add_div, add_mod, M, C, gamma, beta, eps, yp); \
  } while (0)
  if (CV == 40) HI3D_LN_LAUNCH(5, 8);            // C = 320
  else if (CV == 80) HI3D_LN_LAUNCH(5, 16);      // C = 640
  else if (CV == 160) HI3D_LN_LAUNCH(5, 32);     // C = 1280
  else if (CV == 8) HI3D_LN_LAUNCH(1, 8);        // C = 64
  else if (CV == 16) HI3D_LN_LAUNCH(2, 8);       // C = 128
  else if (CV == 32) HI3D_LN_LAUNCH(2, 16);      // C = 256
  else if (CV == 64) HI3D_LN_LAUNCH(2, 32);      // C = 512
  else if (CV == 320) HI3D_LN_LAUNCH(10, 32);    // C = 2560
  else if (CV <= 64) HI3D_LN_GENERIC(2);
  else if (CV <= 160) HI3D_LN_GENERIC(5);
  else HI3D_LN_GENERIC(10);
#undef HI3D_LN_LAUNCH
#undef HI3D_LN_GENERIC
  return check_launch("hi3d_layernorm");
}
