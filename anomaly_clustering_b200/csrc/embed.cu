// Stage 1: hooked feature maps -> patch embeddings Z (fp32) + tensor-core operands (hi/lo).
//
// Replaces AnomalyClusteringCore._embed after the backbone
// (reference: Anomaly-Clustering/models/patchcore/patchcore.py:368-431, common.py:145-183).
//
// Closed form implemented here (SURVEY.md section 8c):
//   Z[b, y, x, t] = (1/|G_t|) sum_{g in G_t} (1/|F_g|) sum_{f in F_g} U_l(g)[b, f, y, x]
//   G_t = adaptive-pool window of t over the L*Dp concat (Aggregator),
//   F_g = adaptive-pool window of d = g % Dp over the C*k*k flat patch vector (MeanMapper),
//   U_l[b, f=(c,ki,kj), y', x'] = LN_l(b)[c, y'*s - pad + ki, x'*s - pad + kj] (0 outside the map),
//   layers whose patch grid differs from layer 0 are resampled plane-wise (bilinear,
//   align_corners=False) AFTER the unfold, as the reference does.
// Everything after the LayerNorm is a fixed sparse linear map, so one CTA stages the (LayerNorm'd,
// zero-padded) input rows it needs in shared memory once and every thread evaluates "its" output
// columns t for all positions of the row with per-thread tap tables held in registers.  HBM sees
// each feature map once and each Z element once; no im2col tensor exists.
#include "common.cuh"
#include <vector>
#include <algorithm>
#include <cstring>
#include <memory>
#include <type_traits>
#include <mutex>

namespace ac {

static constexpr int kMaxLayers = 8;
static constexpr int kThreads = 256;
static constexpr int kTPT = 2;            // output columns per thread
static constexpr int kStatSplit = 32;     // partial-sum blocks per (image, layer)

struct LayerDev {
  const float* ptr;
  int C, H, W;
  long long sb, sc, sh, sw;
  int gh, gw;     // unfold grid of this layer
  int CK;         // C*k*k
  int resample;   // grid differs from layer 0
};

struct ChunkDesc {
  int layer;
  int t0, t1;     // output columns [t0, t1)
  int c_lo, nch;  // staged channel range
  int maxtaps;
};

struct EmbedParams {
  LayerDev layers[kMaxLayers];
  int L, B, k, s, pad, Dp;
  int b0;                // first image of this sub-batch (kernels see b = b0 + blockIdx.z)
  int agg_in, agg_out;   // Aggregator pool: agg_in = L*Dp -> agg_out (== D when fused, else L*Dp)
  int h0, w0;
  int xseg_len, nxseg;
  int layernorm;
  float eps;
  float* Z;              // [B*P0, ldz] or null
  void* Zhi;
  void* Zlo;
  int op_dtype;
  long long ldz;
  const double* stats;   // [B][L][kStatSplit][2]
};

struct LaunchGeom {
  int chan_contig;       // smem tile is [row][col][chan] (token layout) else [chan][row][col]
  int SC, SR, SX;        // smem strides (elements)
  int nrows_max, ncols_max;
};

// ------------------------------------------------------------------------------------------------
// tap enumeration (host + device): output column t -> list of (f, weight) on layer `layer`
template <typename F>
__host__ __device__ inline void for_each_tap(int t, int agg_in, int agg_out, int Dp, int CK, F&& fn) {
  const int g0 = pool_start(t, agg_in, agg_out), g1 = pool_end(t, agg_in, agg_out);
  const float wg = 1.0f / (float)(g1 - g0);
  for (int g = g0; g < g1; ++g) {
    const int d = g % Dp;
    const int f0 = pool_start(d, CK, Dp), f1 = pool_end(d, CK, Dp);
    const float w = wg / (float)(f1 - f0);
    for (int f = f0; f < f1; ++f) fn(f, w);
  }
}

__host__ __device__ inline int tap_offset(int f, int k, int c_lo, int SC, int SR, int SX) {
  const int kk = k * k;
  const int c = f / kk, rem = f - c * kk;
  const int ki = rem / k, kj = rem - ki * k;
  return (c - c_lo) * SC + ki * SR + kj * SX;
}

// PyTorch upsample_bilinear2d source index, align_corners=False
__host__ __device__ inline void bilinear_src(int dst, int in_size, int out_size, int& i0, int& i1, float& l1) {
  const float scale = (float)in_size / (float)out_size;
#ifdef __CUDA_ARCH__
  float src = __fsub_rn(__fmul_rn(scale, (float)dst + 0.5f), 0.5f);  // no FMA contraction: same rounding as the host plan
#else
  volatile float prod = scale * ((float)dst + 0.5f);
  float src = prod - 0.5f;
#endif
  if (src < 0.f) src = 0.f;
  i0 = (int)src;
  if (i0 > in_size - 1) i0 = in_size - 1;
  i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  l1 = src - (float)i0;
}

// ------------------------------------------------------------------------------------------------
// per-(image, layer) sum / sum of squares partials for the whole-map LayerNorm (patchcore.py:384)
__global__ void __launch_bounds__(256) ln_stats_kernel(EmbedParams p, double* stats) {
  const int l = blockIdx.y, b = p.b0 + blockIdx.z;
  const LayerDev ly = p.layers[l];
  const long long n = (long long)ly.C * ly.H * ly.W;
  const float* base = ly.ptr + (long long)b * ly.sb;
  // dense images (any axis permutation) can be walked flat
  long long lo_e = n * blockIdx.x / gridDim.x, hi_e = n * (blockIdx.x + 1) / gridDim.x;
  float s = 0.f, q = 0.f;
  const bool tok = (ly.sc == 1 && ly.sw == ly.C && ly.sh == (long long)ly.W * ly.C);
  const bool cnn = (ly.sw == 1 && ly.sh == ly.W && ly.sc == (long long)ly.H * ly.W);
  if ((tok || cnn) && (n % (4LL * gridDim.x) == 0) && ((reinterpret_cast<uintptr_t>(base) & 15) == 0)) {
    // dense image, 16-byte aligned slices: 128-bit loads, 4 independent accumulator pairs
    const float4* b4 = reinterpret_cast<const float4*>(base);
    float s2 = 0.f, q2 = 0.f, s3 = 0.f, q3 = 0.f, s4 = 0.f, q4 = 0.f;
    for (long long e = lo_e / 4 + threadIdx.x; e < hi_e / 4; e += blockDim.x) {
      const float4 v = __ldg(b4 + e);
      s += v.x; q = fmaf(v.x, v.x, q);
      s2 += v.y; q2 = fmaf(v.y, v.y, q2);
      s3 += v.z; q3 = fmaf(v.z, v.z, q3);
      s4 += v.w; q4 = fmaf(v.w, v.w, q4);
    }
    s = (s + s2) + (s3 + s4);
    q = (q + q2) + (q3 + q4);
  } else if (tok || cnn) {
    for (long long e = lo_e + threadIdx.x; e < hi_e; e += blockDim.x) {
      const float v = __ldg(base + e);
      s += v;
      q = fmaf(v, v, q);
    }
  } else {
    const int HW = ly.H * ly.W;
    for (long long e = lo_e + threadIdx.x; e < hi_e; e += blockDim.x) {
      const int c = (int)(e / HW);
      const int r = (int)(e - (long long)c * HW);
      const int y = r / ly.W, x = r - y * ly.W;
      const float v = __ldg(base + c * ly.sc + y * ly.sh + x * ly.sw);
      s += v;
      q = fmaf(v, v, q);
    }
  }
  __shared__ double sh_s[8], sh_q[8];
  double ds = warp_sum((double)s), dq = warp_sum((double)q);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { sh_s[w] = ds; sh_q[w] = dq; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, c2 = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += sh_s[i]; c2 += sh_q[i]; }
    double* o = stats + (((long long)b * p.L + l) * kStatSplit + blockIdx.x) * 2;
    o[0] = a;
    o[1] = c2;
  }
}

// ------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ T to_op(float v);
template <> __device__ __forceinline__ __half to_op<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 to_op<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ float op_to_float(__half v) { return __half2float(v); }
__device__ __forceinline__ float op_to_float(__nv_bfloat16 v) { return __bfloat162float(v); }

__device__ __forceinline__ void store_out(const EmbedParams& p, long long row, int t, float v) {
  const long long idx = row * p.ldz + t;
  if (p.Z) p.Z[idx] = v;
  if (p.Zhi) {
    if (p.op_dtype == AC_DT_F16) {
      const __half h = __float2half_rn(v);
      reinterpret_cast<__half*>(p.Zhi)[idx] = h;
      if (p.Zlo) reinterpret_cast<__half*>(p.Zlo)[idx] = __float2half_rn(v - __half2float(h));
    } else {
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      reinterpret_cast<__nv_bfloat16*>(p.Zhi)[idx] = h;
      if (p.Zlo) reinterpret_cast<__nv_bfloat16*>(p.Zlo)[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
  }
}


// Warp-collective: mean / rstd of (image b, layer) from the statistics pre-pass partials
// (biased variance, eps inside the sqrt -- nn.LayerNorm semantics, patchcore.py:384-385).
__device__ __forceinline__ void warp_ln_params(const EmbedParams& p, const LayerDev& ly, int b, int layer, int lane, float& mu,
                                               float& rstd) {
  mu = 0.f;
  rstd = 1.f;
  if (!p.layernorm) return;
  const double* st = p.stats + (((long long)b * p.L + layer) * kStatSplit) * 2;
  double a = 0, q = 0;
  for (int i = lane; i < kStatSplit; i += 32) { a += st[2 * i]; q += st[2 * i + 1]; }
  a = warp_sum(a);
  q = warp_sum(q);
  const double n = (double)ly.C * ly.H * ly.W;
  const double m = a / n;
  double var = q / n - m * m;
  if (var < 0) var = 0;
  mu = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)p.eps));
}

// MAXTAPS > 0: per-thread tap tables in registers.  MAXTAPS == 0: taps re-enumerated on the fly
// (any pooling ratio / patch size; slow path).
template <int MAXTAPS, bool RESAMPLE>
__global__ void __launch_bounds__(kThreads) embed_kernel(EmbedParams p, const ChunkDesc* __restrict__ chunks,
                                                         int chunk_base, LaunchGeom g) {
  extern __shared__ float tile[];
  __shared__ float s_mu, s_rstd;
  __shared__ int s_xo0[RESAMPLE ? 256 : 1], s_xo1[RESAMPLE ? 256 : 1];
  __shared__ float s_lx[RESAMPLE ? 256 : 1];

  const ChunkDesc ck = chunks[chunk_base + blockIdx.x];
  const LayerDev ly = p.layers[ck.layer];
  const int y = blockIdx.y / p.nxseg, xseg = blockIdx.y - y * p.nxseg;
  const int b = p.b0 + blockIdx.z;
  const int xa = xseg * p.xseg_len, xb = min(p.w0, xa + p.xseg_len);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- LayerNorm statistics of (image b, layer) from the pre-pass partials
  if (warp == 0) {
    float mu, rstd;
    warp_ln_params(p, ly, b, ck.layer, lane, mu, rstd);
    if (lane == 0) { s_mu = mu; s_rstd = rstd; }
  }

  // ---- tile geometry (input rows / cols staged for this output row segment)
  int in_row0, nrows, in_col0, ncols, dyrow = 0;
  float wy1 = 0.f;
  if (!RESAMPLE) {
    in_row0 = y * p.s - p.pad;
    nrows = p.k;
    in_col0 = xa * p.s - p.pad;
    ncols = (xb - xa - 1) * p.s + p.k;
  } else {
    int y0, y1;
    bilinear_src(y, ly.gh, p.h0, y0, y1, wy1);
    in_row0 = y0 * p.s - p.pad;
    dyrow = (y1 - y0) * p.s;
    nrows = dyrow + p.k;
    int xl0, xl1, xh0, xh1;
    float tmp;
    bilinear_src(xa, ly.gw, p.w0, xl0, xl1, tmp);
    bilinear_src(xb - 1, ly.gw, p.w0, xh0, xh1, tmp);
    in_col0 = xl0 * p.s - p.pad;
    ncols = (xh1 - xl0) * p.s + p.k;
    for (int x = xa + tid; x < xb; x += kThreads) {
      int x0, x1;
      float l1;
      bilinear_src(x, ly.gw, p.w0, x0, x1, l1);
      s_xo0[x - xa] = (x0 - xl0) * p.s * g.SX;
      s_xo1[x - xa] = (x1 - xl0) * p.s * g.SX;
      s_lx[x - xa] = l1;
    }
  }
  __syncthreads();
  const float mu = s_mu, rstd = s_rstd;

  // ---- stage: (v - mu) * rstd inside the map, literal zeros outside (the reference pads AFTER LN)
  const float* src = ly.ptr + (long long)b * ly.sb + (long long)ck.c_lo * ly.sc;
  if (g.chan_contig) {
    const int npos = nrows * ncols;
    for (int pos = warp; pos < npos; pos += kThreads / 32) {
      const int r = pos / ncols, xx = pos - r * ncols;
      const int iy = in_row0 + r, ix = in_col0 + xx;
      const bool inside = (iy >= 0) && (iy < ly.H) && (ix >= 0) && (ix < ly.W);
      float* dst = tile + r * g.SR + xx * g.SX;
      const float* s0 = src + (long long)iy * ly.sh + (long long)ix * ly.sw;
      for (int c = lane; c < ck.nch; c += 32) dst[c] = inside ? (__ldg(s0 + c) - mu) * rstd : 0.f;
    }
  } else {
    const int ncr = ck.nch * nrows;
    for (int cr = warp; cr < ncr; cr += kThreads / 32) {
      const int c = cr / nrows, r = cr - c * nrows;
      const int iy = in_row0 + r;
      const bool rin = (iy >= 0) && (iy < ly.H);
      float* dst = tile + c * g.SC + r * g.SR;
      const float* s0 = src + (long long)c * ly.sc + (long long)iy * ly.sh;
      for (int xx = lane; xx < ncols; xx += 32) {
        const int ix = in_col0 + xx;
        const bool inside = rin && (ix >= 0) && (ix < ly.W);
        dst[xx * g.SX] = inside ? (__ldg(s0 + (long long)ix * ly.sw) - mu) * rstd : 0.f;
      }
    }
  }

  // ---- per-thread tap tables
  int tcol[kTPT];
  bool tvalid[kTPT];
  int off[kTPT][MAXTAPS > 0 ? MAXTAPS : 1];
  float wt[kTPT][MAXTAPS > 0 ? MAXTAPS : 1];
  int ntap[kTPT];
#pragma unroll
  for (int j = 0; j < kTPT; ++j) {
    tcol[j] = ck.t0 + tid + j * kThreads;
    tvalid[j] = tcol[j] < ck.t1;
    ntap[j] = 0;
    if (MAXTAPS > 0) {
#pragma unroll
      for (int q = 0; q < MAXTAPS; ++q) { off[j][q] = 0; wt[j][q] = 0.f; }
      if (tvalid[j]) {
        int n = 0;
        for_each_tap(tcol[j], p.agg_in, p.agg_out, p.Dp, ly.CK, [&](int f, float w) {
          const int o = tap_offset(f, p.k, ck.c_lo, g.SC, g.SR, g.SX);
#pragma unroll
          for (int q = 0; q < MAXTAPS; ++q)
            if (q == n) { off[j][q] = o; wt[j][q] = w; }
          ++n;
        });
        ntap[j] = n;
      }
    }
  }
  __syncthreads();

  // ---- evaluate every position of the row segment
  const long long row0 = ((long long)b * p.h0 + y) * p.w0;
#pragma unroll 2
  for (int x = xa; x < xb; ++x) {
    float acc[kTPT];
    if (!RESAMPLE) {
      const float* tb = tile + (x - xa) * p.s * g.SX;
#pragma unroll
      for (int j = 0; j < kTPT; ++j) {
        float a = 0.f;
        if (MAXTAPS > 0) {
#pragma unroll
          for (int q = 0; q < MAXTAPS; ++q) {
            const float v = tb[off[j][q]];
            a = (q < ntap[j]) ? fmaf(wt[j][q], v, a) : a;  // unused slots never touch the sum (NaN-safe)
          }
        } else if (tvalid[j]) {
          for_each_tap(tcol[j], p.agg_in, p.agg_out, p.Dp, ly.CK, [&](int f, float w) {
            a = fmaf(w, tb[tap_offset(f, p.k, ck.c_lo, g.SC, g.SR, g.SX)], a);
          });
        }
        acc[j] = a;
      }
    } else {
      const float lx1 = s_lx[x - xa], lx0 = 1.f - lx1, ly0 = 1.f - wy1;
      const float* t00 = tile + s_xo0[x - xa];
      const float* t01 = tile + s_xo1[x - xa];
      const float* t10 = t00 + dyrow * g.SR;
      const float* t11 = t01 + dyrow * g.SR;
#pragma unroll
      for (int j = 0; j < kTPT; ++j) {
        float a = 0.f;
        auto tap = [&](int o, float w, bool on) {
          const float v = ly0 * (lx0 * t00[o] + lx1 * t01[o]) + wy1 * (lx0 * t10[o] + lx1 * t11[o]);
          a = on ? fmaf(w, v, a) : a;
        };
        if (MAXTAPS > 0) {
#pragma unroll
          for (int q = 0; q < MAXTAPS; ++q) tap(off[j][q], wt[j][q], q < ntap[j]);
        } else if (tvalid[j]) {
          for_each_tap(tcol[j], p.agg_in, p.agg_out, p.Dp, ly.CK, [&](int f, float w) {
            tap(tap_offset(f, p.k, ck.c_lo, g.SC, g.SR, g.SX), w, true);
          });
        }
        acc[j] = a;
      }
    }
#pragma unroll
    for (int j = 0; j < kTPT; ++j)
      if (tvalid[j]) store_out(p, row0 + x, tcol[j], acc[j]);
  }
}



// Writes NOUT consecutive outputs of one patch row: fp32 Z (16-byte vectors when aligned) and the
// tensor-core operand copies hi = round(z), lo = round(z - hi).
template <typename T, int NOUT>
__device__ __forceinline__ void store_operand(void* Zhi, void* Zlo, long long idx, bool vec, const float (&out)[NOUT]) {
  __align__(16) T h[NOUT];
#pragma unroll
  for (int o = 0; o < NOUT; ++o) h[o] = to_op<T>(out[o]);
  T* ph = reinterpret_cast<T*>(Zhi) + idx;
  if (vec) {
#pragma unroll
    for (int o = 0; o + 8 <= NOUT; o += 8) *reinterpret_cast<uint4*>(ph + o) = *reinterpret_cast<const uint4*>(&h[o]);
  } else {
#pragma unroll
    for (int o = 0; o < NOUT; ++o) ph[o] = h[o];
  }
  if (Zlo) {
    __align__(16) T l[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) l[o] = to_op<T>(out[o] - op_to_float(h[o]));
    T* pl = reinterpret_cast<T*>(Zlo) + idx;
    if (vec) {
#pragma unroll
      for (int o = 0; o + 8 <= NOUT; o += 8) *reinterpret_cast<uint4*>(pl + o) = *reinterpret_cast<const uint4*>(&l[o]);
    } else {
#pragma unroll
      for (int o = 0; o < NOUT; ++o) pl[o] = l[o];
    }
  }
}

template <int NOUT>
__device__ __forceinline__ void store_outputs(const EmbedParams& p, long long idx, int t_base, const float (&out)[NOUT]) {
  if (p.Z) {
    if (NOUT % 4 == 0 && ((p.ldz | t_base) & 3) == 0) {
#pragma unroll
      for (int o = 0; o + 4 <= NOUT; o += 4)
        *reinterpret_cast<float4*>(p.Z + idx + o) = make_float4(out[o], out[o + 1], out[o + 2], out[o + 3]);
    } else {
#pragma unroll
      for (int o = 0; o < NOUT; ++o) p.Z[idx + o] = out[o];
    }
  }
  if (p.Zhi) {
    const bool vec = (NOUT % 8 == 0) && (((p.ldz | t_base) & 7) == 0);
    if (p.op_dtype == AC_DT_F16) store_operand<__half, NOUT>(p.Zhi, p.Zlo, idx, vec, out);
    else store_operand<__nv_bfloat16, NOUT>(p.Zhi, p.Zlo, idx, vec, out);
  }
}

// ------------------------------------------------------------------------------------------------
// Fast path for channel-contiguous layers (ViT tokens, channels_last maps) on the layer-0 grid,
// stride 1: "periodic sliding window".  With 9C/Dp = A/B in lowest terms (A a multiple of K*K),
// B consecutive pooled outputs depend on exactly A/(K*K) consecutive channels and the window
// pattern repeats every period, so one thread owns one period: it keeps the K x K neighbourhood of
// its channels in registers, slides it along x (K new values per channel per position instead of
// K*K) and emits its B (or B/R after an R:1 Aggregator) outputs per position as 16-byte vectors.
// Lanes own consecutive channel groups, so loads are fully coalesced straight from L2 (no shared
// memory, no barriers) and each warp writes B*128 contiguous bytes of Z per position.
template <int A, int B, int K, int R>
__global__ void __launch_bounds__(kThreads) embed_periodic_kernel(EmbedParams p, int layer, int t_base, int nperiods) {
  constexpr int CPP = A / (K * K);   // channels per period
  constexpr int NOUT = B / R;        // outputs per period after the aggregator
  static_assert(A % (K * K) == 0 && B % R == 0, "period must cover whole channels / aggregator windows");
  __shared__ float s_mu, s_rstd;
  const LayerDev ly = p.layers[layer];
  const int b = p.b0 + blockIdx.z;
  const int y = blockIdx.y / p.nxseg, xseg = blockIdx.y - y * p.nxseg;
  const int xa = xseg * p.xseg_len, xb = min(p.w0, xa + p.xseg_len);
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid < 32) {
    float mu, rstd;
    warp_ln_params(p, ly, b, layer, lane, mu, rstd);
    if (lane == 0) { s_mu = mu; s_rstd = rstd; }
  }
  __syncthreads();
  const float mu = s_mu, rstd = s_rstd;
  const int m = blockIdx.x * kThreads + tid;
  if (m >= nperiods) return;
  const float* src = ly.ptr + (long long)b * ly.sb + (long long)m * CPP;   // sc == 1
  bool rowok[K];
  const float* rowp[K];
#pragma unroll
  for (int ki = 0; ki < K; ++ki) {
    const int iy = y - p.pad + ki;
    rowok[ki] = (iy >= 0) && (iy < ly.H);
    rowp[ki] = src + (long long)iy * ly.sh;
  }
  auto load_col = [&](int ix, float (&dst)[CPP][K]) {
    const bool cin = (ix >= 0) && (ix < ly.W);
#pragma unroll
    for (int ki = 0; ki < K; ++ki) {
      const bool ok = cin && rowok[ki];
      const float* q = rowp[ki] + (long long)ix * ly.sw;
#pragma unroll
      for (int c = 0; c < CPP; ++c) dst[c][ki] = ok ? (__ldg(q + c) - mu) * rstd : 0.f;
    }
  };
  float v[CPP][K][K];   // [channel][ki][kj] window of the current position
  float nxt[CPP][K];    // prefetched right-most column of the next position
  // window of the fictitious position xa-1, so that the first shift lands on xa
#pragma unroll
  for (int kj = 1; kj < K; ++kj) {
    float col[CPP][K];
    load_col(xa - 1 - p.pad + kj, col);
#pragma unroll
    for (int c = 0; c < CPP; ++c)
#pragma unroll
      for (int ki = 0; ki < K; ++ki) v[c][ki][kj] = col[c][ki];
  }
  load_col(xa - p.pad + K - 1, nxt);
  const long long row0 = ((long long)b * p.h0 + y) * p.w0;
  const int t0 = t_base + m * NOUT;
  for (int x = xa; x < xb; ++x) {
#pragma unroll
    for (int c = 0; c < CPP; ++c)
#pragma unroll
      for (int ki = 0; ki < K; ++ki) {
#pragma unroll
        for (int kj = 0; kj + 1 < K; ++kj) v[c][ki][kj] = v[c][ki][kj + 1];
        v[c][ki][K - 1] = nxt[c][ki];
      }
    if (x + 1 < xb) load_col(x + 1 - p.pad + K - 1, nxt);   // prefetch while this position is reduced
    float out[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) {
      float acc_o = 0.f;
#pragma unroll
      for (int j = 0; j < R; ++j) {
        constexpr int dummy = 0; (void)dummy;
        const int r = o * R + j;
        const int f0 = (r * A) / B, f1 = ((r + 1) * A + B - 1) / B;
        float sacc = 0.f;
#pragma unroll
        for (int f = 0; f < A; ++f)
          if (f >= f0 && f < f1) sacc += v[f / (K * K)][(f % (K * K)) / K][f % K];
        acc_o += sacc * (1.0f / (float)(f1 - f0));
      }
      out[o] = (R == 1) ? acc_o : acc_o * (1.0f / (float)R);
    }
    store_outputs<NOUT>(p, (row0 + x) * p.ldz + t0, t_base, out);
  }
}


// ------------------------------------------------------------------------------------------------
// TMA-staged variant of the periodic kernel (the default when the 16-byte alignment rules of
// cp.async.bulk hold).  Same arithmetic, but the feature columns are streamed into a shared-memory
// ring by a dedicated producer warp with 1-D bulk copies (one 3 KB token row per (ki, column) for
// ViT-B) that run kRing columns ahead of the math, so HBM/L2 latency is hidden independently of
// occupancy and no registers are spent on prefetch.  Consumers read each staged column once
// (conflict-free: lane stride = channels per period), apply the LayerNorm affine in registers and
// slide the K x K window as above.
static constexpr int kRing = 6;

__device__ __forceinline__ uint32_t e_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void e_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void e_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void e_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool e_mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void e_mbar_wait(uint32_t bar, uint32_t parity) {
  if (e_mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!e_mbar_try(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();   // ~2 s: a broken pipeline must fail the launch, never hang the GPU
  }
}
__device__ __forceinline__ void e_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}

template <int A, int B, int K, int R>
__global__ void __launch_bounds__(kThreads + 32, 3) embed_tma_kernel(EmbedParams p, int layer, int t_base, int nperiods) {
  constexpr int CPP = A / (K * K);
  constexpr int NOUT = B / R;
  constexpr int NCH = kThreads * CPP;   // channels staged per column (all periods of this CTA)
  extern __shared__ __align__(128) float ring[];          // [kRing][K][NCH]
  __shared__ __align__(8) uint64_t s_full[kRing], s_empty[kRing];
  __shared__ float s_mu, s_rstd;
  const LayerDev ly = p.layers[layer];
  const int b = p.b0 + blockIdx.z;
  const int y = blockIdx.y / p.nxseg, xseg = blockIdx.y - y * p.nxseg;
  const int xa = xseg * p.xseg_len, xb = min(p.w0, xa + p.xseg_len);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m0 = blockIdx.x * kThreads;
  const int c_start = m0 * CPP;
  const int nch = min(NCH, ly.C - c_start);               // multiple of 4 (host guarantees C % 4 == 0)
  const int ncols = (xb - xa) + K - 1;                     // staged input columns xa-pad .. xb-1-pad+K-1
  if (tid == 0) {
    for (int i = 0; i < kRing; ++i) {
      e_mbar_init(e_smem_u32(&s_full[i]), 1);
      e_mbar_init(e_smem_u32(&s_empty[i]), kThreads / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    float mu, rstd;
    warp_ln_params(p, ly, b, layer, lane, mu, rstd);
    if (lane == 0) { s_mu = mu; s_rstd = rstd; }
  }
  __syncthreads();

  bool rowok[K];
#pragma unroll
  for (int ki = 0; ki < K; ++ki) {
    const int iy = y - p.pad + ki;
    rowok[ki] = (iy >= 0) && (iy < ly.H);
  }

  if (warp == kThreads / 32) {
    // ================================================================ producer warp
    if (lane == 0) {
      const float* src = ly.ptr + (long long)b * ly.sb + c_start;
      const uint32_t bytes_row = (uint32_t)nch * 4u;
      for (int j = 0; j < ncols; ++j) {
        const int slot = j % kRing;
        const uint32_t ph = (uint32_t)(j / kRing) & 1u;
        e_mbar_wait(e_smem_u32(&s_empty[slot]), ph ^ 1u);
        const int ix = xa - p.pad + j;
        const bool cin = (ix >= 0) && (ix < ly.W);
        uint32_t nrows = 0;
#pragma unroll
        for (int ki = 0; ki < K; ++ki) nrows += (cin && rowok[ki]) ? 1u : 0u;
        const uint32_t fb = e_smem_u32(&s_full[slot]);
        if (nrows == 0) {
          e_mbar_arrive(fb);
        } else {
          e_mbar_expect_tx(fb, nrows * bytes_row);
#pragma unroll
          for (int ki = 0; ki < K; ++ki)
            if (cin && rowok[ki])
              e_bulk_g2s(e_smem_u32(ring + ((size_t)slot * K + ki) * NCH),
                         src + (long long)(y - p.pad + ki) * ly.sh + (long long)ix * ly.sw, bytes_row, fb);
        }
      }
    }
    return;
  }

  // ================================================================== consumers (kThreads)
  static_assert(K == 3, "the rotating register window below is unrolled for 3x3 patches");
  const float mu = s_mu, rstd = s_rstd;
  const int m = m0 + tid;
  const bool active = m < nperiods;
  // LayerNorm affine folded into one FFMA per value; rows outside the map get scale = offset = 0
  // and read a valid staged row instead (finite * 0), so no per-value select is needed
  float sc[K], of[K];
  int krow[K];
  int kvalid = 0;
#pragma unroll
  for (int ki = 0; ki < K; ++ki)
    if (rowok[ki]) kvalid = ki;
#pragma unroll
  for (int ki = 0; ki < K; ++ki) {
    const bool ok = rowok[ki] && active;
    sc[ki] = ok ? rstd : 0.f;
    of[ki] = ok ? -mu * rstd : 0.f;
    krow[ki] = (rowok[ki] ? ki : kvalid) * NCH;
  }
  float v[CPP][K][K];   // [channel][ki][physical column slot]
#pragma unroll
  for (int c = 0; c < CPP; ++c)
#pragma unroll
    for (int ki = 0; ki < K; ++ki)
#pragma unroll
      for (int kj = 0; kj < K; ++kj) v[c][ki][kj] = 0.f;
  const long long row0 = ((long long)b * p.h0 + y) * p.w0;
  const int t0 = t_base + (active ? m : 0) * NOUT;

  // one step: append staged column j into physical slot j % K, then emit position xa + j - (K-1);
  // ROT = (j + 1) % K maps logical kj -> physical (kj + ROT) % K, all indices compile-time
  auto step = [&](auto rot_tag, int j) {
    constexpr int ROT = decltype(rot_tag)::value;
    constexpr int SLOT = (ROT + K - 1) % K;
    const int slot = j % kRing;
    const uint32_t ph = (uint32_t)(j / kRing) & 1u;
    const int ix = xa - p.pad + j;
    const bool cin = (ix >= 0) && (ix < ly.W);
    e_mbar_wait(e_smem_u32(&s_full[slot]), ph);
    if (cin) {
      const float* col = ring + (size_t)slot * K * NCH + tid * CPP;
#pragma unroll
      for (int c = 0; c < CPP; ++c)
#pragma unroll
        for (int ki = 0; ki < K; ++ki) v[c][ki][SLOT] = fmaf(col[krow[ki] + c], sc[ki], of[ki]);
    } else {
#pragma unroll
      for (int c = 0; c < CPP; ++c)
#pragma unroll
        for (int ki = 0; ki < K; ++ki) v[c][ki][SLOT] = 0.f;
    }
    __syncwarp();
    if (lane == 0) e_mbar_arrive(e_smem_u32(&s_empty[slot]));
    const int x = xa + j - (K - 1);
    if (x < xa || !active) return;
    float out[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) {
      float acc_o = 0.f;
#pragma unroll
      for (int jj = 0; jj < R; ++jj) {
        const int r = o * R + jj;
        const int f0 = (r * A) / B, f1 = ((r + 1) * A + B - 1) / B;
        float sacc = 0.f;
#pragma unroll
        for (int f = 0; f < A; ++f)
          if (f >= f0 && f < f1) sacc += v[f / (K * K)][(f % (K * K)) / K][((f % K) + ROT) % K];
        acc_o += sacc * (1.0f / (float)(f1 - f0));
      }
      out[o] = (R == 1) ? acc_o : acc_o * (1.0f / (float)R);
    }
    store_outputs<NOUT>(p, (row0 + x) * p.ldz + t0, t_base, out);
  };
  for (int j0 = 0; j0 < ncols; j0 += 3) {
    step(std::integral_constant<int, 1>{}, j0);
    if (j0 + 1 < ncols) step(std::integral_constant<int, 2>{}, j0 + 1);
    if (j0 + 2 < ncols) step(std::integral_constant<int, 0>{}, j0 + 2);
  }
}


// ------------------------------------------------------------------------------------------------
// Single-pass fused form: ONE persistent launch embeds every layer, folds the whole-map LayerNorm in without a second
// DRAM read of the feature maps, and emits the operands' squared norms as well (default whenever all layers are
// channel-contiguous, on one patch grid, of one width and 16-byte aligned: ViT tokens, channels_last maps).
//
// A work item = (image, row segment of <= kMaxSeg positions).  Items are claimed in order from a global counter; item
// q*S + s first reduces slice s of image q (its share of sum / sum of squares for the LayerNorm statistics, patchcore.py:384)
// and then embeds slice s of image q - LA.  An embed waits until all S slices of its image have been reduced; those
// belong to items claimed LA*S claims earlier, which are running on resident CTAs and never wait themselves, so the
// scheme cannot deadlock and the wait is short.  The maps of the LA + (resident items / S) images in flight (a few tens
// of MB) stay in L2 between their statistics read (DRAM) and their 3 x 3-neighbourhood reads by the embed phase (L2).
// Same producer-warp / mbarrier ring as embed_tma_kernel; the statistics slices travel through the same ring.
// The LayerNorm affine is folded into the pooling: out = rstd/n * sum(raw taps) - mu*rstd with out-of-map taps set to
// mu (the reference pads with zeros AFTER the LayerNorm), one FFMA per output instead of one per staged value.
static constexpr int kMaxSeg = 16;

struct FusedParams {
  EmbedParams e;
  float* n2;               // [B*P0] squared norms of the operand rows (hi [+ lo]) or null
  double* stats;           // [B][L][S][2] partial (sum, sum of squares)
  int* done;               // [B] slices reduced per image
  unsigned int* counter;   // item claims
  int S, LA, nperiods, gx, t_stride;
  long long n_items;       // (B + LA) * S
  const float* zero_row;   // >= 4 KB of zeros (lean kernel: stands in for taps outside the map)
  unsigned long long* murs;  // [B][L] (mean, 1/std) packed as two floats, all-ones until the last statistics warp of the image wrote it (lean kernel)
};

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory"); }

// stores NOUT consecutive operand values (hi [+ lo]) of one patch row, returns sum (hi + lo)^2
template <typename T, int NOUT>
__device__ __forceinline__ float store_operand_norm(void* Zhi, void* Zlo, long long idx, bool vec, const float (&out)[NOUT]) {
  __align__(16) T h[NOUT];
  float nv = 0.f;
#pragma unroll
  for (int o = 0; o < NOUT; ++o) h[o] = to_op<T>(out[o]);
  T* ph = reinterpret_cast<T*>(Zhi) + idx;
  if (vec) {
#pragma unroll
    for (int o = 0; o + 8 <= NOUT; o += 8) *reinterpret_cast<uint4*>(ph + o) = *reinterpret_cast<const uint4*>(&h[o]);
  } else {
#pragma unroll
    for (int o = 0; o < NOUT; ++o) ph[o] = h[o];
  }
  if (Zlo) {
    __align__(16) T l[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) {
      l[o] = to_op<T>(out[o] - op_to_float(h[o]));
      const float v = op_to_float(h[o]) + op_to_float(l[o]);
      nv = fmaf(v, v, nv);
    }
    T* pl = reinterpret_cast<T*>(Zlo) + idx;
    if (vec) {
#pragma unroll
      for (int o = 0; o + 8 <= NOUT; o += 8) *reinterpret_cast<uint4*>(pl + o) = *reinterpret_cast<const uint4*>(&l[o]);
    } else {
#pragma unroll
      for (int o = 0; o < NOUT; ++o) pl[o] = l[o];
    }
  } else {
#pragma unroll
    for (int o = 0; o < NOUT; ++o) { const float v = op_to_float(h[o]); nv = fmaf(v, v, nv); }
  }
  return nv;
}

// Consumer threads of the fused kernel.  One thread owns TWO consecutive periods and keeps their values as float2
// pairs, so that every add / fma of the pooling runs as ONE packed fp32x2 instruction (add.f32x2 / fma.rn.f32x2, new
// on sm_100) for both periods: the kernel is instruction-issue bound (ncu, round 2: issue slots 77 % busy at a DRAM
// throughput of 47 %), and this halves its arithmetic instructions.
static constexpr int kFT = 128;
static constexpr int kPP = 2;            // periods per thread

__device__ __forceinline__ void consumer_bar_f() { asm volatile("bar.sync 1, %0;" ::"n"(kFT) : "memory"); }

template <int A, int B, int R>
__global__ void __launch_bounds__(kFT + 32, 3) embed_fused_kernel(const __grid_constant__ FusedParams fp) {
  constexpr int K = 3;
  constexpr int CPP = A / (K * K);
  constexpr int NOUT = B / R;
  constexpr int TCH = kPP * CPP;                 // channels per thread
  constexpr int NCH = kFT * TCH;                 // channels per ring row
  const EmbedParams& p = fp.e;
  extern __shared__ __align__(128) float smem_f[];
  float* ring = smem_f;                                    // [kRing][K][NCH]
  float* s_nacc = smem_f + (size_t)kRing * K * NCH;        // [kMaxSeg][kFT] per-thread share of the row norms
  __shared__ __align__(8) uint64_t s_full[kRing], s_empty[kRing];
  __shared__ float s_red[2][kFT / 32];
  __shared__ float s_mu[kMaxLayers], s_rs[kMaxLayers];
  __shared__ long long s_item;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool producer = (warp == kFT / 32);
  if (tid == 0) {
    for (int i = 0; i < kRing; ++i) {
      e_mbar_init(e_smem_u32(&s_full[i]), 1);
      e_mbar_init(e_smem_u32(&s_empty[i]), kFT / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t slot = 0, ph = 0;                               // ring position: identical sequence in both roles
  const uint32_t full0 = e_smem_u32(&s_full[0]), empty0 = e_smem_u32(&s_empty[0]);
  const bool vec8 = (NOUT % 8 == 0) && (((p.ldz | fp.t_stride) & 7) == 0);
  const bool vec4 = (NOUT % 4 == 0) && (((p.ldz | fp.t_stride) & 3) == 0);
  const bool f16 = (p.op_dtype == AC_DT_F16);
  const float* ring_t = ring + tid * TCH;

  for (;;) {
    if (tid == 0) s_item = (long long)atomicAdd(fp.counter, 1u);
    __syncthreads();
    const long long item = s_item;
    if (item >= fp.n_items) break;
    const int q = (int)(item / fp.S), sg = (int)(item - (long long)q * fp.S);
    const int y = sg / p.nxseg, xs = sg - y * p.nxseg;
    const int xa = xs * p.xseg_len, xb = min(p.w0, xa + p.xseg_len), npos = xb - xa;
    const int bA = (q < p.B) ? q : -1;                     // image whose statistics slice is reduced
    const int bE = q - fp.LA;                              // image whose slice is embedded (< 0: prologue item)
    const int nA = (npos + K - 1) / K;                     // statistics slots: K tokens each
    const int ncols = npos + K - 1;                        // embed slots: input columns xa-1 .. xb

    if (producer) {
      // ================================================================ producer warp
      if (lane == 0) {
        if (bA >= 0 && p.layernorm) {
          for (int l = 0; l < p.L; ++l) {
            const LayerDev& ly = p.layers[l];
            for (int cx = 0; cx < fp.gx; ++cx) {
              const int c_start = cx * NCH;
              const uint32_t bytes = (uint32_t)min(NCH, ly.C - c_start) * 4u;
              const float* src = ly.ptr + (long long)(p.b0 + bA) * ly.sb + c_start + (long long)y * ly.sh + (long long)xa * ly.sw;
              for (int t = 0; t < nA; ++t) {
                e_mbar_wait(empty0 + slot * 8, ph ^ 1u);
                const int ntok = min(K, npos - K * t);
                const uint32_t fb = full0 + slot * 8;
                e_mbar_expect_tx(fb, (uint32_t)ntok * bytes);
                for (int ki = 0; ki < ntok; ++ki)
                  e_bulk_g2s(e_smem_u32(ring + ((size_t)slot * K + ki) * NCH), src + (long long)(K * t + ki) * ly.sw, bytes, fb);
                if (++slot == kRing) { slot = 0; ph ^= 1u; }
              }
            }
          }
        }
        if (bE >= 0) {
          for (int l = 0; l < p.L; ++l) {
            const LayerDev& ly = p.layers[l];
            for (int cx = 0; cx < fp.gx; ++cx) {
              const int c_start = cx * NCH;
              const uint32_t bytes = (uint32_t)min(NCH, ly.C - c_start) * 4u;
              const float* src = ly.ptr + (long long)(p.b0 + bE) * ly.sb + c_start;
              for (int j = 0; j < ncols; ++j) {
                e_mbar_wait(empty0 + slot * 8, ph ^ 1u);
                const int ix = xa - p.pad + j;
                const bool cin = (ix >= 0) && (ix < ly.W);
                uint32_t nrows = 0;
#pragma unroll
                for (int ki = 0; ki < K; ++ki) {
                  const int iy = y - p.pad + ki;
                  nrows += (cin && iy >= 0 && iy < ly.H) ? 1u : 0u;
                }
                const uint32_t fb = full0 + slot * 8;
                if (nrows == 0) {
                  e_mbar_arrive(fb);
                } else {
                  e_mbar_expect_tx(fb, nrows * bytes);
#pragma unroll
                  for (int ki = 0; ki < K; ++ki) {
                    const int iy = y - p.pad + ki;
                    if (cin && iy >= 0 && iy < ly.H)
                      e_bulk_g2s(e_smem_u32(ring + ((size_t)slot * K + ki) * NCH), src + (long long)iy * ly.sh + (long long)ix * ly.sw, bytes, fb);
                  }
                }
                if (++slot == kRing) { slot = 0; ph ^= 1u; }
              }
            }
          }
        }
      }
    } else {
      // ================================================================ consumers (kFT)
      // ---- phase A: this item's share of the LayerNorm statistics of image bA
      if (bA >= 0 && p.layernorm) {
        for (int l = 0; l < p.L; ++l) {
          float s = 0.f, qq = 0.f;
          for (int cx = 0; cx < fp.gx; ++cx) {
            const int m0 = (cx * kFT + tid) * kPP;            // first period of this thread
            for (int t = 0; t < nA; ++t) {
              e_mbar_wait(full0 + slot * 8, ph);
              const int ntok = min(K, npos - K * t);
              const float* col = ring_t + (size_t)slot * K * NCH;
#pragma unroll
              for (int ki = 0; ki < K; ++ki)
                if (ki < ntok) {
#pragma unroll
                  for (int c = 0; c < TCH; ++c)
                    if (m0 + c / CPP < fp.nperiods) { const float v = col[ki * NCH + c]; s += v; qq = fmaf(v, v, qq); }
                }
              __syncwarp();
              if (lane == 0) e_mbar_arrive(empty0 + slot * 8);
              if (++slot == kRing) { slot = 0; ph ^= 1u; }
            }
          }
          s = warp_sum(s);
          qq = warp_sum(qq);
          if (lane == 0) { s_red[0][warp] = s; s_red[1][warp] = qq; }
          consumer_bar_f();
          if (tid == 0) {
            double a = 0, c2 = 0;
            for (int w = 0; w < kFT / 32; ++w) { a += (double)s_red[0][w]; c2 += (double)s_red[1][w]; }
            double* o = fp.stats + (((long long)bA * p.L + l) * fp.S + sg) * 2;
            o[0] = a;
            o[1] = c2;
          }
          consumer_bar_f();
        }
        if (tid == 0) {
          __threadfence();
          atomicAdd(fp.done + bA, 1);
        }
      }
      // ---- phase B: embed slice sg of image bE
      if (bE >= 0) {
        if (p.layernorm) {
          if (tid == 0) {
            const long long t0 = clock64();
            while (ld_acquire_gpu(fp.done + bE) < fp.S) {
              __nanosleep(100);
              if (clock64() - t0 > 4000000000LL) __trap();     // a broken schedule must fail the launch, never hang the GPU
            }
          }
          consumer_bar_f();
          if (warp == 0) {
            for (int l = 0; l < p.L; ++l) {
              const double* st = fp.stats + (((long long)bE * p.L + l) * fp.S) * 2;
              double a = 0, c2 = 0;
              for (int i = lane; i < fp.S; i += 32) { a += __ldcg(st + 2 * i); c2 += __ldcg(st + 2 * i + 1); }
              a = warp_sum(a);
              c2 = warp_sum(c2);
              const double n = (double)p.layers[l].C * p.layers[l].H * p.layers[l].W;
              const double m = a / n;
              double var = c2 / n - m * m;
              if (var < 0) var = 0;
              if (lane == 0) { s_mu[l] = (float)m; s_rs[l] = (float)(1.0 / sqrt(var + (double)p.eps)); }
            }
          }
          consumer_bar_f();
        }
        const long long row0 = ((long long)(p.b0 + bE) * p.h0 + y) * p.w0;
        bool first = true;
        for (int l = 0; l < p.L; ++l) {
          const LayerDev& ly = p.layers[l];
          const float mu = p.layernorm ? s_mu[l] : 0.f, rs = p.layernorm ? s_rs[l] : 1.f;
          const float2 mu2 = make_float2(mu, mu), nmr2 = make_float2(-mu * rs, -mu * rs);
          bool rowok[K];
#pragma unroll
          for (int ki = 0; ki < K; ++ki) {
            const int iy = y - p.pad + ki;
            rowok[ki] = (iy >= 0) && (iy < ly.H);
          }
          for (int cx = 0; cx < fp.gx; ++cx, first = false) {
            const int m0 = (cx * kFT + tid) * kPP;
            const bool actA = m0 < fp.nperiods, actB = m0 + 1 < fp.nperiods;
            // the two periods' outputs are adjacent: [t0, t0 + NOUT) and [t0 + NOUT, t0 + 2 NOUT)
            long long idx = (row0 + xa) * p.ldz + (long long)l * fp.t_stride + (long long)(actA ? m0 : 0) * NOUT;
            float2 v[CPP][K][K];   // [channel][ki][physical column slot], .x = first period, .y = second; out-of-map taps hold mu
#pragma unroll
            for (int c = 0; c < CPP; ++c)
#pragma unroll
              for (int ki = 0; ki < K; ++ki)
#pragma unroll
                for (int kj = 0; kj < K; ++kj) v[c][ki][kj] = mu2;
            float* na = s_nacc + tid;
            auto step = [&](auto rot_tag, int j) {
              constexpr int ROT = decltype(rot_tag)::value;
              constexpr int SLOT = (ROT + K - 1) % K;
              const int ix = xa - p.pad + j;
              const bool cin = (ix >= 0) && (ix < ly.W);
              e_mbar_wait(full0 + slot * 8, ph);
              const float* col = ring_t + (size_t)slot * K * NCH;
#pragma unroll
              for (int ki = 0; ki < K; ++ki) {
                if (cin && rowok[ki]) {                      // warp-uniform
#pragma unroll
                  for (int c = 0; c < CPP; ++c) v[c][ki][SLOT] = make_float2(col[ki * NCH + c], col[ki * NCH + CPP + c]);
                } else {
#pragma unroll
                  for (int c = 0; c < CPP; ++c) v[c][ki][SLOT] = mu2;
                }
              }
              __syncwarp();
              if (lane == 0) e_mbar_arrive(empty0 + slot * 8);
              if (++slot == kRing) { slot = 0; ph ^= 1u; }
              if (j < K - 1) return;                         // the window is not full yet
              float nv = 0.f;
              if (actA) {
                float2 out[NOUT];
#pragma unroll
                for (int o = 0; o < NOUT; ++o) {
                  float2 acc_o = nmr2;
#pragma unroll
                  for (int jj = 0; jj < R; ++jj) {
                    const int r = o * R + jj;
                    const int f0 = (r * A) / B, f1 = ((r + 1) * A + B - 1) / B;
                    float2 sacc = v[f0 / (K * K)][(f0 % (K * K)) / K][((f0 % K) + ROT) % K];
#pragma unroll
                    for (int f = 0; f < A; ++f)
                      if (f > f0 && f < f1) sacc = __fadd2_rn(sacc, v[f / (K * K)][(f % (K * K)) / K][((f % K) + ROT) % K]);
                    const float cf = rs * (1.0f / (float)(R * (f1 - f0)));
                    acc_o = __ffma2_rn(sacc, make_float2(cf, cf), acc_o);
                  }
                  out[o] = acc_o;
                }
                float oa[NOUT], ob[NOUT];
#pragma unroll
                for (int o = 0; o < NOUT; ++o) { oa[o] = out[o].x; ob[o] = out[o].y; }
                if (p.Z) {
                  if (vec4) {
#pragma unroll
                    for (int o = 0; o + 4 <= NOUT; o += 4)
                      *reinterpret_cast<float4*>(p.Z + idx + o) = make_float4(oa[o], oa[o + 1], oa[o + 2], oa[o + 3]);
                    if (actB) {
#pragma unroll
                      for (int o = 0; o + 4 <= NOUT; o += 4)
                        *reinterpret_cast<float4*>(p.Z + idx + NOUT + o) = make_float4(ob[o], ob[o + 1], ob[o + 2], ob[o + 3]);
                    }
                  } else {
#pragma unroll
                    for (int o = 0; o < NOUT; ++o) p.Z[idx + o] = oa[o];
                    if (actB) {
#pragma unroll
                      for (int o = 0; o < NOUT; ++o) p.Z[idx + NOUT + o] = ob[o];
                    }
                  }
                }
                if (p.Zhi) {
                  if (f16) {
                    nv = store_operand_norm<__half, NOUT>(p.Zhi, p.Zlo, idx, vec8, oa);
                    if (actB) nv += store_operand_norm<__half, NOUT>(p.Zhi, p.Zlo, idx + NOUT, vec8, ob);
                  } else {
                    nv = store_operand_norm<__nv_bfloat16, NOUT>(p.Zhi, p.Zlo, idx, vec8, oa);
                    if (actB) nv += store_operand_norm<__nv_bfloat16, NOUT>(p.Zhi, p.Zlo, idx + NOUT, vec8, ob);
                  }
                }
              }
              if (fp.n2) {
                *na = first ? nv : (*na + nv);
                na += kFT;
              }
              idx += p.ldz;
            };
            for (int j0 = 0; j0 < ncols; j0 += 3) {
              step(std::integral_constant<int, 1>{}, j0);
              if (j0 + 1 < ncols) step(std::integral_constant<int, 2>{}, j0 + 1);
              if (j0 + 2 < ncols) step(std::integral_constant<int, 0>{}, j0 + 2);
            }
          }
        }
        if (fp.n2) {
          // squared norms of the operand rows of this segment: fixed summation order (bit-reproducible)
          consumer_bar_f();
          for (int pos = warp; pos < npos; pos += kFT / 32) {
            float a = 0.f;
#pragma unroll
            for (int k2 = 0; k2 < kFT / 32; ++k2) a += s_nacc[pos * kFT + lane + 32 * k2];
            a = warp_sum(a);
            if (lane == 0) fp.n2[row0 + xa + pos] = a;
          }
        }
      }
    }
    __syncthreads();      // s_item / s_nacc / s_red are reused by the next item
  }
}

// ------------------------------------------------------------------------------------------------
// Lean form of the fused kernel for the shapes the headline workloads use (fp16 operands + norms, optionally fp32 Z,
// every consumer thread active).  Same schedule, ring and arithmetic as embed_fused_kernel; what changes is the cost of a
// step.  ncu of the general kernel (profiles/r02_ncu_full.md): 355 warp instructions per staged column of which ~100 do
// the work -- the rest were per-value selects for taps outside the map, register moves that re-pair LDS.64 results for
// the packed adds, run-time switches on the output set and generic-pointer shared-memory addressing.  Here
//   * taps outside the map are staged as ZEROS by the producer (bulk copies from a zero row in the workspace), so the
//     consumers load unconditionally; the zero-padding of the reference (pad AFTER the LayerNorm, patchcore.py:384-385 then
//     :447) is restored on the few edge positions by adding mu * rstd * (missing taps / window) per output,
//   * staged values are read with 32-bit ld.shared straight into the halves of the packed registers (immediate offsets
//     from one base register per step),
//   * the output set is a template parameter.
__device__ __forceinline__ float2 e_lds64(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
template <int OFF>
__device__ __forceinline__ float e_lds32(uint32_t base) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(base), "n"(OFF));
  return v;
}
__device__ __forceinline__ void e_mbar_wait_spin(uint32_t bar, uint32_t parity) {
  while (!e_mbar_try(bar, parity)) {}
}
// producer side of the lean kernel: a full ring means the consumers are several slots behind, so the single producer
// thread sleeps between polls instead of burning issue slots of the scheduler it shares with three consumer warps
// (round-2 capture: 25 % of all issued instructions were the producer's, most of them this loop)
__device__ __forceinline__ bool e_mbar_try_suspend(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void e_mbar_wait_sleep(uint32_t bar, uint32_t parity) {
  if (e_mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!e_mbar_try_suspend(bar, parity, 2000u)) {   // suspended by the hardware until the phase flips (or the hint elapses)
    if (clock64() - t0 > 4000000000LL) __trap();   // ~2 s: a broken pipeline must fail the launch, never hang the GPU
  }
}
// acc + h * h with the product and the sum in fp32 (one FHFMA; the half is read straight from its half2 register)
__device__ __forceinline__ float e_sq_acc(__half h, float acc) {
  const unsigned short x = __half_as_ushort(h);
  asm("fma.rn.f32.f16 %0, %1, %1, %0;" : "+f"(acc) : "h"(x));
  return acc;
}

// one staged row of this thread: .x = channel c of its first period, .y = channel c of its second period, which lies
// HALF floats further (periods tid and tid + FT): far enough apart that ptxas keeps the 32-bit loads apart and lets each
// land in its half of the packed register pair (adjacent periods became LDS.64 + two moves per pair)
template <int KI, int NCH_, int HALF>
__device__ __forceinline__ void e_load_row3(uint32_t base, float2& a, float2& b, float2& c) {
  a = make_float2(e_lds32<(KI * NCH_ + 0) * 4>(base), e_lds32<(KI * NCH_ + HALF + 0) * 4>(base));
  b = make_float2(e_lds32<(KI * NCH_ + 1) * 4>(base), e_lds32<(KI * NCH_ + HALF + 1) * 4>(base));
  c = make_float2(e_lds32<(KI * NCH_ + 2) * 4>(base), e_lds32<(KI * NCH_ + HALF + 2) * 4>(base));
}

// "The data is the flag": a partial statistic (sum, sum of squares) and a final (mean, 1/std) travel as ONE 64-bit relaxed
// store into a slot that holds all-ones until then (no arithmetic produces that pattern: NaNs come out canonical,
// 0x7fffffff), and readers poll the slot itself.  No release / acquire fences: a gpu-scope release made every consumer
// warp wait for all its outstanding operand stores (MEMBAR + ERRBAR: 6 % of the samples in the round-2 capture), an
// acquire invalidates L1 on every poll.
static constexpr unsigned long long kUnset = ~0ull;
__device__ __forceinline__ int e_atom_add_relaxed(int* p, int v) {
  int old;
  asm volatile("atom.add.relaxed.gpu.global.s32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void e_st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long e_ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long e_pack2(float a, float b) {
  return (unsigned long long)__float_as_uint(a) | ((unsigned long long)__float_as_uint(b) << 32);
}
// polls a slot until it is set; a broken schedule must fail the launch, never hang the GPU
__device__ __forceinline__ unsigned long long e_wait_set(const unsigned long long* p, unsigned long long v) {
  if (v != kUnset) return v;
  const long long t0 = clock64();
  while ((v = e_ld_relaxed_u64(p)) == kUnset) {
    __nanosleep(64);
    if (clock64() - t0 > 4000000000LL) __trap();
  }
  return v;
}
__device__ __forceinline__ void e_bulk_g2s_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void e_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

static constexpr int kRingL = 7;         // ring depth of the lean kernel (72 KB of shared memory per CTA at 768 channels, 3 CTAs per SM; a 5-slot ring
                                         // at 4 CTAs per SM and 96 registers was measured 20 % slower: more images in flight than L2 holds)
static constexpr int kItemQ = 2;         // items the producer may be ahead of the consumers

template <int A, int B, int R, int FT, bool WZ, int RING, int MINB>
__global__ void __launch_bounds__(FT + 32, MINB) embed_fused_fast_kernel(const __grid_constant__ FusedParams fp) {
  constexpr int K = 3;
  constexpr int CPP = A / (K * K);
  constexpr int NOUT = B / R;
  constexpr int TCH = kPP * CPP;                 // channels per thread (two periods)
  constexpr int NCH = FT * TCH;                  // channels per ring row == C of every layer (host checks)
  static_assert(NOUT % 8 == 0 || NOUT == 4, "operand rows are written in 16-byte pieces");
  static_assert(TCH % 2 == 0, "the statistics phase reads channel pairs");
  static_assert(CPP == 3, "three channels per period (9C : Dp = 27 : B)");
  const EmbedParams& p = fp.e;
  extern __shared__ __align__(128) float smem_f[];
  float* ring = smem_f;                                    // [RING][K][NCH]
  float* s_nacc = smem_f + (size_t)RING * K * NCH;       // [kMaxSeg][FT] per-thread share of the row norms
  __shared__ __align__(8) uint64_t s_full[RING], s_empty[RING];
  __shared__ __align__(8) uint64_t s_qfull[kItemQ], s_qempty[kItemQ];
  __shared__ long long s_items[kItemQ];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool producer = (warp == FT / 32);
  if (tid == 0) {
    for (int i = 0; i < RING; ++i) {
      e_mbar_init(e_smem_u32(&s_full[i]), 1);
      e_mbar_init(e_smem_u32(&s_empty[i]), FT / 32);
    }
    for (int i = 0; i < kItemQ; ++i) {
      e_mbar_init(e_smem_u32(&s_qfull[i]), 1);
      e_mbar_init(e_smem_u32(&s_qempty[i]), FT / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t slot = 0, ph = 0;                               // ring position: identical sequence in both roles
  const uint32_t full0 = e_smem_u32(&s_full[0]), empty0 = e_smem_u32(&s_empty[0]);
  const uint32_t ring_a = e_smem_u32(ring) + (uint32_t)tid * TCH * 4u;      // statistics phase: TCH consecutive channels of a ring row
  const uint32_t ring_t = e_smem_u32(ring) + (uint32_t)tid * CPP * 4u;      // embed phase: periods tid and tid + FT
  constexpr uint32_t kSlotBytes = (uint32_t)K * NCH * 4u;
  constexpr uint32_t kRowBytes = (uint32_t)NCH * 4u;

  // Items are claimed by the PRODUCER, which publishes them through a kItemQ-deep queue and keeps staging: the copies of
  // the next item (its statistics slots come from DRAM) are in flight while the consumers still work on this one.  (With
  // one CTA-wide claim per item the ring ran dry at every item boundary: 28 % of the consumers' cycles waited for data.)
  // The earliest unfinished item is always at the head of its CTA's queue, so the wait of an embed phase for the
  // statistics of its image cannot deadlock.
  uint32_t qs = 0, qph = 0;
  if (producer && lane != 0) return;
  // L2 policies of the map loads: the maps must survive in L2 from their statistics read to their last embed read while
  // 1.3x their volume of operand rows streams out through the same cache
  uint64_t pol_keep = 0;
  if (producer) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
  for (;;) {
    long long item;
    if (producer) {
      e_mbar_wait_sleep(e_smem_u32(&s_qempty[qs]), qph ^ 1u);
      item = (long long)atomicAdd(fp.counter, 1u);
      s_items[qs] = item;
      asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(e_smem_u32(&s_qfull[qs])) : "memory");
    } else {
      long long it = 0;
      if (lane == 0) {
        e_mbar_wait(e_smem_u32(&s_qfull[qs]), qph);
        it = *reinterpret_cast<volatile long long*>(&s_items[qs]);
        e_mbar_arrive(e_smem_u32(&s_qempty[qs]));
      }
      item = __shfl_sync(0xffffffffu, it, 0);
    }
    if (++qs == kItemQ) { qs = 0; qph ^= 1u; }
    if (item >= fp.n_items) break;
    // Slice sg of an image (square patch grid, the host checks): for the STATISTICS it is a run of <= xseg_len tokens of one
    // map row (yA, xaA ..), for the EMBEDDING it is one patch column x and the rows ya .. yb - 1.  The embed window slides
    // DOWN a column because the K tokens (x-1, x, x+1) of a map row are contiguous in memory: a ring slot is ONE bulk copy
    // of K tokens instead of K copies (the single producer thread pays ~30 instructions per copy).
    const int q = (int)(item / fp.S), sg = (int)(item - (long long)q * fp.S);
    const int s_hi = sg / p.nxseg, s_lo = sg - s_hi * p.nxseg;
    const int yA = s_hi, xaA = s_lo * p.xseg_len, nposA = min(p.w0, xaA + p.xseg_len) - xaA;
    const int x = s_hi, ya = s_lo * p.xseg_len, yb = min(p.h0, ya + p.xseg_len), npos = yb - ya;
    const int bA = (q < p.B) ? q : -1;                     // image whose statistics slice is reduced
    const int bE = q - fp.LA;                              // image whose slice is embedded (< 0: prologue item)
    const int nA = (nposA + K - 1) / K;                    // statistics slots: K tokens each (missing ones staged as zeros)
    const int nrows = npos + K - 1;                        // embed slots: input rows ya-1 .. yb

    if (producer) {
      // ================================================================ producer thread: every slot is K full rows
      // statistics slots of image bA first (they never wait for anything), then the embed slots of image bE.  (Spreading the
      // statistics slots through the embed loop hides their DRAM latency but delays done[bA] to the end of an item that
      // itself waits for done[bE]: the images then advance LA per item time -- measured 2.5 / 1.3 / 0.65 ms at LA 1 / 2 / 4.)
      // The producer is ONE thread and every slot costs it a serial chain (ncu, round 2: 188 instructions per slot with the
      // addresses recomputed per row -- 1 250 cycles per slot and CTA, the consumers waited for data 23 % of their time), so
      // everything that does not change inside an item is hoisted: per row one running pointer, per slot one add and one
      // select per row.
      const bool hasA = (bA >= 0) && p.layernorm, hasB = (bE >= 0);
      const uint32_t ring_u = e_smem_u32(ring);
      if (hasA) {
        // statistics rows of the item just claimed (its first copies wait behind the ring slots of the previous item):
        // DRAM -> L2 ahead of time, so that the statistics slots at the head of the item's in-order ring are L2 hits like
        // its embed slots
        for (int l = 0; l < p.L; ++l) {
          const LayerDev& ly = p.layers[l];
          if (ly.sw == NCH)      // the tokens of a row are contiguous
            e_prefetch_l2(ly.ptr + (long long)bA * ly.sb + (long long)yA * ly.sh + (long long)xaA * ly.sw, (uint32_t)nposA * kRowBytes);
        }
        for (int l = 0; l < p.L; ++l) {
          const LayerDev& ly = p.layers[l];
          const long long sw = ly.sw;
          const bool contig = (sw == NCH);                   // K tokens = one copy
          const float* cur = ly.ptr + (long long)bA * ly.sb + (long long)yA * ly.sh + (long long)xaA * sw;
          int rem = nposA;                                   // tokens left (>= 1 at every slot)
          for (int t = 0; t < nA; ++t, rem -= K, cur += K * sw) {
            e_mbar_wait_sleep(empty0 + slot * 8, ph ^ 1u);
            const uint32_t fb = full0 + slot * 8, dst = ring_u + slot * kSlotBytes;
            e_mbar_expect_tx(fb, kSlotBytes);
            if (contig && rem >= K) {
              e_bulk_g2s_hint(dst, cur, kSlotBytes, fb, pol_keep);
            } else {
#pragma unroll
              for (int ki = 0; ki < K; ++ki) e_bulk_g2s_hint(dst + ki * kRowBytes, (ki < rem) ? cur + ki * sw : fp.zero_row, kRowBytes, fb, pol_keep);
            }
            if (++slot == RING) { slot = 0; ph ^= 1u; }
          }
        }
      }
      if (hasB) {
        // map row ya - 1 + j lies outside the map only at j == 0 of the first segment and at the last j of the last segment
        const int jlo = (ya == 0) ? 0 : -1, jhi = (yb == p.h0) ? nrows - 1 : -1;
        const bool ok0 = (x >= 1), ok2 = (x + 1 < p.w0);
        for (int l = 0; l < p.L; ++l) {
          const LayerDev& ly = p.layers[l];
          const long long sw = ly.sw;
          const bool one = ok0 && ok2 && (sw == NCH);        // the K tokens x-1 .. x+1 of a row: one copy
          const float* r0 = ly.ptr + (long long)bE * ly.sb + (long long)(ya - 1) * ly.sh + (long long)(x - 1) * sw;
          for (int j = 0; j < nrows; ++j, r0 += ly.sh) {
            e_mbar_wait_sleep(empty0 + slot * 8, ph ^ 1u);
            const bool rin = (j != jlo) && (j != jhi);
            const uint32_t fb = full0 + slot * 8, dst = ring_u + slot * kSlotBytes;
            e_mbar_expect_tx(fb, kSlotBytes);
            if (!rin) {
              e_bulk_g2s_hint(dst, fp.zero_row, kSlotBytes, fb, pol_keep);
            } else if (one) {
              e_bulk_g2s_hint(dst, r0, kSlotBytes, fb, pol_keep);
            } else {
              e_bulk_g2s_hint(dst, ok0 ? r0 : fp.zero_row, kRowBytes, fb, pol_keep);
              e_bulk_g2s_hint(dst + kRowBytes, r0 + sw, kRowBytes, fb, pol_keep);
              e_bulk_g2s_hint(dst + 2 * kRowBytes, ok2 ? r0 + 2 * sw : fp.zero_row, kRowBytes, fb, pol_keep);
            }
            if (++slot == RING) { slot = 0; ph ^= 1u; }
          }
        }
      }
    } else {
      // ================================================================ consumers (FT)
      const bool hasA = (bA >= 0) && p.layernorm, hasB = (bE >= 0);
      constexpr int NW = FT / 32;
      float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
      // one statistics slot: K tokens of image bA (all channels of this thread's share), sum and sum of squares
      auto stats_slot = [&]() {
        e_mbar_wait_spin(full0 + slot * 8, ph);
        const uint32_t base = ring_a + slot * kSlotBytes;
#pragma unroll
        for (int ki = 0; ki < K; ++ki)
#pragma unroll
          for (int c = 0; c < TCH; c += 2) {
            const float2 v = e_lds64(base + (uint32_t)(ki * NCH + c) * 4u);
            s2 = __fadd2_rn(s2, v);
            q2 = __ffma2_rn(v, v, q2);
          }
        __syncwarp();
        if (lane == 0) e_mbar_arrive(empty0 + slot * 8);
        if (++slot == RING) { slot = 0; ph ^= 1u; }
      };
      // per-warp partial of layer l -> its slot in global memory (one 64-bit relaxed store, see kUnset)
      unsigned long long* part = reinterpret_cast<unsigned long long*>(fp.stats);
      auto stats_flush = [&](int l) {
        const float s = warp_sum(s2.x + s2.y), qq = warp_sum(q2.x + q2.y);
        if (lane == 0) e_st_relaxed_u64(part + (((long long)bA * p.L + l) * fp.S + sg) * NW + warp, e_pack2(s, qq));
        s2 = make_float2(0.f, 0.f);
        q2 = make_float2(0.f, 0.f);
      };
      // ---- phase A: this item's share of the LayerNorm statistics of image bA, published per warp (no CTA barrier).
      // The warp that publishes the LAST partial of an image folds all of them (fixed order, fp64) into mean and 1/std
      // once; the embed phases of that image then read two floats per layer.  (Every embed item used to re-reduce the
      // S * NW partials behind two CTA barriers: 11 % of the consumers' samples in the round-2 ncu capture.)
      if (hasA) {
        for (int l = 0; l < p.L; ++l) {
          for (int t = 0; t < nA; ++t) stats_slot();
          stats_flush(l);
        }
        int old = 0;
        if (lane == 0) old = e_atom_add_relaxed(fp.done + bA, 1);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old == fp.S * NW - 1) {
          // every partial of the image has been stored (the counter says so) but not necessarily become visible: wait per slot
          const int n = fp.S * NW;
          for (int l = 0; l < p.L; ++l) {
            const unsigned long long* st = part + (((long long)bA * p.L + l) * fp.S) * NW;
            double a = 0, c2 = 0;
            for (int i0 = 0; i0 < n; i0 += 32 * 8) {
              unsigned long long v[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * 32 + lane;
                v[u] = (i < n) ? e_ld_relaxed_u64(st + i) : 0ull;
              }
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * 32 + lane;
                if (i < n) {
                  const unsigned long long pk = e_wait_set(st + i, v[u]);
                  a += (double)__uint_as_float((unsigned int)pk);
                  c2 += (double)__uint_as_float((unsigned int)(pk >> 32));
                }
              }
            }
            a = warp_sum(a);
            c2 = warp_sum(c2);
            const double nn = (double)p.layers[l].C * p.layers[l].H * p.layers[l].W;
            const double m = a / nn;
            double var = c2 / nn - m * m;
            if (var < 0) var = 0;
            if (lane == 0) e_st_relaxed_u64(fp.murs + (long long)bA * p.L + l, e_pack2((float)m, (float)(1.0 / sqrt(var + (double)p.eps))));
          }
        }
      }
      // ---- phase B: embed slice sg of image bE
      if (hasB) {
        const long long row0 = ((long long)bE * p.h0 + ya) * p.w0 + x;      // first output row of the slice; the next is w0 further
        const bool xedge = (x == 0) || (x == p.w0 - 1);
        for (int l = 0; l < p.L; ++l) {
          const LayerDev& ly = p.layers[l];
          float mu = 0.f, rs = 1.f;
          if (p.layernorm) {
            const unsigned long long* mr = fp.murs + (long long)bE * p.L + l;
            unsigned long long pk = 0ull;
            if (lane == 0) pk = e_wait_set(mr, e_ld_relaxed_u64(mr));
            pk = __shfl_sync(0xffffffffu, pk, 0);
            mu = __uint_as_float((unsigned int)pk);
            rs = __uint_as_float((unsigned int)(pk >> 32));
          }
          const float nmr = -mu * rs;
          const float2 nmr2 = make_float2(nmr, nmr);
          // outputs of period tid at [tid * NOUT, + NOUT), of period tid + FT at FT * NOUT further
          long long idx = row0 * p.ldz + (long long)l * fp.t_stride + (long long)tid * NOUT;
          const long long idx_step = (long long)p.w0 * p.ldz;
          float2 v[CPP][K][K];   // [channel][physical row slot][kj]; .x = first period, .y = second
          float* na = s_nacc + tid;
          auto step = [&](auto rot_tag, int j) {
            constexpr int ROT = decltype(rot_tag)::value;
            constexpr int SLOT = (ROT + K - 1) % K;
            e_mbar_wait_spin(full0 + slot * 8, ph);
            const uint32_t base = ring_t + slot * kSlotBytes;
            // the slot holds map row ya - 1 + j: tokens x-1, x, x+1 (kj = 0, 1, 2), NCH channels each
            e_load_row3<0, NCH, FT * CPP>(base, v[0][SLOT][0], v[1][SLOT][0], v[2][SLOT][0]);
            e_load_row3<1, NCH, FT * CPP>(base, v[0][SLOT][1], v[1][SLOT][1], v[2][SLOT][1]);
            e_load_row3<2, NCH, FT * CPP>(base, v[0][SLOT][2], v[1][SLOT][2], v[2][SLOT][2]);
            __syncwarp();
            if (lane == 0) e_mbar_arrive(empty0 + slot * 8);
            if (++slot == RING) { slot = 0; ph ^= 1u; }
            if (j < K - 1) return;                         // the window is not full yet
            float2 out[NOUT];
#pragma unroll
            for (int o = 0; o < NOUT; ++o) {
              float2 acc_o = nmr2;
#pragma unroll
              for (int jj = 0; jj < R; ++jj) {
                const int r = o * R + jj;
                const int f0 = (r * A) / B, f1 = ((r + 1) * A + B - 1) / B;
                float2 sacc = v[f0 / (K * K)][((f0 % (K * K)) / K + ROT) % K][f0 % K];
#pragma unroll
                for (int f = 0; f < A; ++f)
                  if (f > f0 && f < f1) sacc = __fadd2_rn(sacc, v[f / (K * K)][((f % (K * K)) / K + ROT) % K][f % K]);
                const float cf = rs * (1.0f / (float)(R * (f1 - f0)));
                acc_o = __ffma2_rn(sacc, make_float2(cf, cf), acc_o);
              }
              out[o] = acc_o;
            }
            const int y = ya + j - (K - 1);
            if (xedge || y == 0 || y == p.h0 - 1) {          // warp-uniform, a few percent of the positions
              // taps outside the map were staged as zeros; the reference pads after the LayerNorm, i.e. they must count as
              // mu before the affine: add mu * rstd * (missing taps of the window) / (window size)
              float bad[K][K];
#pragma unroll
              for (int ki = 0; ki < K; ++ki)
#pragma unroll
                for (int kj = 0; kj < K; ++kj) {
                  const int iy = y - 1 + ki, ix = x - 1 + kj;
                  bad[ki][kj] = (iy >= 0 && iy < ly.H && ix >= 0 && ix < ly.W) ? 0.f : 1.f;
                }
#pragma unroll
              for (int o = 0; o < NOUT; ++o) {
                float corr = 0.f;
#pragma unroll
                for (int jj = 0; jj < R; ++jj) {
                  const int r = o * R + jj;
                  const int f0 = (r * A) / B, f1 = ((r + 1) * A + B - 1) / B;
                  float cnt = 0.f;
#pragma unroll
                  for (int f = 0; f < A; ++f)
                    if (f >= f0 && f < f1) cnt += bad[(f % (K * K)) / K][f % K];
                  corr = fmaf(cnt, 1.0f / (float)(R * (f1 - f0)), corr);
                }
                const float add = -nmr * corr;
                out[o] = __fadd2_rn(out[o], make_float2(add, add));
              }
            }
            if constexpr (WZ) {
#pragma unroll
              for (int o = 0; o + 4 <= NOUT; o += 4) {
                *reinterpret_cast<float4*>(p.Z + idx + o) = make_float4(out[o].x, out[o + 1].x, out[o + 2].x, out[o + 3].x);
                *reinterpret_cast<float4*>(p.Z + idx + FT * NOUT + o) = make_float4(out[o].y, out[o + 1].y, out[o + 2].y, out[o + 3].y);
              }
            }
            // fp16 operand rows (16-byte stores) and the squared norm of the ROUNDED values
            float2 nv2 = make_float2(0.f, 0.f);
            __half* ph_ = reinterpret_cast<__half*>(p.Zhi) + idx;
#pragma unroll
            for (int half_ = 0; half_ < 2; ++half_) {
#pragma unroll
              for (int o = 0; o + 8 <= NOUT; o += 8) {
                __align__(16) __half2 h[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  h[i] = half_ == 0 ? __floats2half2_rn(out[o + 2 * i].x, out[o + 2 * i + 1].x)
                                    : __floats2half2_rn(out[o + 2 * i].y, out[o + 2 * i + 1].y);
                  nv2.x = e_sq_acc(__low2half(h[i]), nv2.x);
                  nv2.y = e_sq_acc(__high2half(h[i]), nv2.y);
                }
                // streaming (evict-first) store: the operand rows must not push the maps out of L2
                __stcs(reinterpret_cast<uint4*>(ph_ + half_ * (FT * NOUT) + o), *reinterpret_cast<const uint4*>(h));
              }
              if constexpr (NOUT == 4) {
                __align__(8) __half2 h[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                  h[i] = half_ == 0 ? __floats2half2_rn(out[2 * i].x, out[2 * i + 1].x) : __floats2half2_rn(out[2 * i].y, out[2 * i + 1].y);
                  nv2.x = e_sq_acc(__low2half(h[i]), nv2.x);
                  nv2.y = e_sq_acc(__high2half(h[i]), nv2.y);
                }
                *reinterpret_cast<uint2*>(ph_ + half_ * (FT * NOUT)) = *reinterpret_cast<const uint2*>(h);
              }
            }
            const float nv = nv2.x + nv2.y;
            *na = (l == 0) ? nv : (*na + nv);
            na += FT;
            idx += idx_step;
          };
          for (int j0 = 0; j0 < nrows; j0 += 3) {
            step(std::integral_constant<int, 1>{}, j0);
            if (j0 + 1 < nrows) step(std::integral_constant<int, 2>{}, j0 + 1);
            if (j0 + 2 < nrows) step(std::integral_constant<int, 0>{}, j0 + 2);
          }
        }
        // squared norms of the operand rows of this segment: fixed summation order (bit-reproducible)
        asm volatile("bar.sync 1, %0;" ::"n"(FT) : "memory");
        for (int pos = warp; pos < npos; pos += FT / 32) {
          float a = 0.f;
#pragma unroll
          for (int k2 = 0; k2 < FT / 32; ++k2) a += s_nacc[pos * FT + lane + 32 * k2];
          a = warp_sum(a);
          if (lane == 0) fp.n2[row0 + (long long)pos * p.w0] = a;
        }
      }
    }
    if (!producer) asm volatile("bar.sync 1, %0;" ::"n"(FT) : "memory");      // s_nacc is reused by the next item
  }
}

__global__ void init_words_kernel(unsigned int* __restrict__ ones, long long n_ones, unsigned int* __restrict__ zeros, long long n_zeros) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_ones + n_zeros; i += (long long)gridDim.x * blockDim.x) {
    if (i < n_ones) ones[i] = 0xffffffffu;
    else zeros[i - n_ones] = 0u;
  }
}

// ------------------------------------------------------------------------------------------------
// Layout / grid adapters that let every layer take the periodic fast path:
//  * nchw_to_nhwc_kernel: CNN maps [B,C,H,W] -> channel-contiguous scratch (32x32 smem tile transpose).
//  * upsample_store_kernel: a layer whose patch grid differs from layer 0 is pooled at ITS OWN grid into a
//    small scratch and then resampled; the reference resamples the unfolded planes and pools afterwards
//    (patchcore.py:398-421), but both maps are linear and act on different axes (positions vs. the flat
//    patch vector), so they commute -- same bilinear weights (align_corners=False), 1/9 of the gathers.
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(LayerDev ly, int b0, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int HW = ly.H * ly.W;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  const float* src = ly.ptr + (long long)(b0 + b) * ly.sb;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, pos = p0 + tx;
    float v = 0.f;
    if (c < ly.C && pos < HW) {
      const int y = pos / ly.W, x = pos - y * ly.W;
      v = __ldg(src + (long long)c * ly.sc + (long long)y * ly.sh + (long long)x * ly.sw);
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  float* dst = out + (long long)b * HW * ly.C;
  for (int r = ty; r < 32; r += 8) {
    const int pos = p0 + r, c = c0 + tx;
    if (c < ly.C && pos < HW) dst[(long long)pos * ly.C + c] = tile[tx][r];
  }
}

// coarse [B, gh*gw, ncols] fp32 -> Z / Zhi / Zlo columns [t_base, t_base + ncols) on the layer-0 grid
__global__ void __launch_bounds__(256) upsample_store_kernel(EmbedParams p, const float* __restrict__ coarse, int gh, int gw, int ncols,
                                                             int t_base) {
  const int cpr = (ncols + 3) / 4;                       // 4-column groups per row
  const long long rows = (long long)p.B * p.h0 * p.w0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < rows * cpr; e += (long long)gridDim.x * blockDim.x) {
    const long long row = e / cpr;
    const int c4 = (int)(e - row * cpr) * 4;
    const int x = (int)(row % p.w0);
    const int y = (int)((row / p.w0) % p.h0);
    const int b = (int)(row / ((long long)p.w0 * p.h0));
    int y0, y1, x0, x1;
    float ly1, lx1;
    bilinear_src(y, gh, p.h0, y0, y1, ly1);
    bilinear_src(x, gw, p.w0, x0, x1, lx1);
    const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    const float* base = coarse + (long long)b * gh * gw * ncols;
    const float* r00 = base + ((long long)y0 * gw + x0) * ncols;
    const float* r01 = base + ((long long)y0 * gw + x1) * ncols;
    const float* r10 = base + ((long long)y1 * gw + x0) * ncols;
    const float* r11 = base + ((long long)y1 * gw + x1) * ncols;
    float out[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = min(c4 + i, ncols - 1);
      out[i] = ly0 * (lx0 * __ldg(r00 + c) + lx1 * __ldg(r01 + c)) + ly1 * (lx0 * __ldg(r10 + c) + lx1 * __ldg(r11 + c));
    }
    const long long grow = (long long)p.b0 * p.h0 * p.w0 + row;
    if (c4 + 4 <= ncols) {
      store_outputs<4>(p, grow * p.ldz + t_base + c4, t_base | c4, out);
    } else {
      for (int i = 0; c4 + i < ncols; ++i) {
        const float o1[1] = {out[i]};
        store_outputs<1>(p, grow * p.ldz + t_base + c4 + i, 1, o1);
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------
// X straight from the feature maps (SURVEY.md section 8f row 4).  Z is a fixed linear map of the LayerNorm'd
// maps, so  X_i = sum_p alpha_ip Z_ip = Pool( A_i ),  A_i[c,ki,kj] = sum_p alpha_ip * LN_i[c, y_p+ki-pad, x_p+kj-pad]
// (zero outside the map): a k x k correlation of the alpha map with every channel, then the SAME two pooling
// windows applied once per image instead of once per patch.  fp32 Z never has to exist.
//   xcorr_kernel : partial A over a slice of rows; thread = channel (coalesced), alpha map with a zero halo in smem
//   xpool_kernel : X[i,t] = sum over taps of wt * (sum of partials)
static constexpr int kXSplit = 4;

template <int K>
__global__ void __launch_bounds__(256) xcorr_kernel(EmbedParams p, int layer, const float* __restrict__ alpha /*[B, P0]*/,
                                                    float* __restrict__ part /*[B, kXSplit, K*K, C]*/) {
  extern __shared__ float s_alpha[];   // (h0 + 2*pad) x (w0 + 2*pad), zero halo
  __shared__ float s_mu, s_rstd;
  const LayerDev ly = p.layers[layer];
  const int b = blockIdx.z, split = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int aw = p.w0 + 2 * p.pad, ah = p.h0 + 2 * p.pad;
  for (int e = threadIdx.x; e < aw * ah; e += blockDim.x) {
    const int y = e / aw - p.pad, x = e % aw - p.pad;
    s_alpha[e] = (y >= 0 && y < p.h0 && x >= 0 && x < p.w0) ? alpha[(long long)b * p.h0 * p.w0 + y * p.w0 + x] : 0.f;
  }
  if (threadIdx.x < 32) {
    float mu, rstd;
    warp_ln_params(p, ly, p.b0 + b, layer, lane, mu, rstd);
    if (lane == 0) { s_mu = mu; s_rstd = rstd; }
  }
  __syncthreads();
  if (c >= ly.C) return;
  const float mu = s_mu, rstd = s_rstd;
  float acc[K][K];
#pragma unroll
  for (int ki = 0; ki < K; ++ki)
#pragma unroll
    for (int kj = 0; kj < K; ++kj) acc[ki][kj] = 0.f;
  const int y0 = (int)((long long)ly.H * split / kXSplit), y1 = (int)((long long)ly.H * (split + 1) / kXSplit);
  const float* src = ly.ptr + (long long)(p.b0 + b) * ly.sb + (long long)c * ly.sc;
  for (int iy = y0; iy < y1; ++iy)
    for (int ix = 0; ix < ly.W; ++ix) {
      const float v = (__ldg(src + (long long)iy * ly.sh + (long long)ix * ly.sw) - mu) * rstd;
      // input (iy, ix) is tap (ki, kj) of output position (iy - ki + pad, ix - kj + pad); s_alpha is offset by pad
      const float* a = s_alpha + (iy + 2 * p.pad) * aw + (ix + 2 * p.pad);
#pragma unroll
      for (int ki = 0; ki < K; ++ki)
#pragma unroll
        for (int kj = 0; kj < K; ++kj) acc[ki][kj] = fmaf(a[-ki * aw - kj], v, acc[ki][kj]);
    }
  float* out = part + (((long long)b * kXSplit + split) * K * K) * ly.C + c;
#pragma unroll
  for (int ki = 0; ki < K; ++ki)
#pragma unroll
    for (int kj = 0; kj < K; ++kj) out[(long long)(ki * K + kj) * ly.C] = acc[ki][kj];
}

__global__ void __launch_bounds__(256) xpool_kernel(EmbedParams p, int layer, int t_begin, int t_end, const float* __restrict__ part,
                                                    float* __restrict__ X /*[B, D]*/) {
  const LayerDev ly = p.layers[layer];
  const int b = blockIdx.y;
  const int t = t_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= t_end) return;
  const int kk = p.k * p.k;
  float acc = 0.f;
  for_each_tap(t, p.agg_in, p.agg_out, p.Dp, ly.CK, [&](int f, float w) {
    const int c = f / kk, tap = f - c * kk;
    float sacc = 0.f;
    for (int sp = 0; sp < kXSplit; ++sp) sacc += __ldg(part + (((long long)b * kXSplit + sp) * kk + tap) * ly.C + c);
    acc = fmaf(w, sacc, acc);
  });
  X[(long long)(p.b0 + b) * p.agg_out + t] = acc;
}

// ------------------------------------------------------------------------------------------------
// standalone compat kernels
__global__ void patchify_kernel(const float* __restrict__ x, int B, int C, int H, int W, int k, int s, int pad,
                                int gh, int gw, float* __restrict__ out) {
  // out [B, gh*gw, C, k, k]
  const long long total = (long long)B * gh * gw * C * k * k;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    long long r = e;
    const int kj = (int)(r % k); r /= k;
    const int ki = (int)(r % k); r /= k;
    const int c = (int)(r % C); r /= C;
    const int px = (int)(r % gw); r /= gw;
    const int py = (int)(r % gh); r /= gh;
    const int b = (int)r;
    const int iy = py * s - pad + ki, ix = px * s - pad + kj;
    float v = 0.f;
    if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(x + (((long long)b * C + c) * H + iy) * W + ix);
    out[e] = v;
  }
}

__global__ void pool1d_kernel(const float* __restrict__ in, long long rows, int Lin, int Lout, float* __restrict__ out) {
  const long long total = rows * Lout;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / Lout;
    const int d = (int)(e - r * Lout);
    const int f0 = pool_start(d, Lin, Lout), f1 = pool_end(d, Lin, Lout);
    const float* src = in + r * Lin;
    float a = 0.f;
    for (int f = f0; f < f1; ++f) a += __ldg(src + f);
    out[e] = a / (float)(f1 - f0);
  }
}

template <typename T>
__global__ void split_kernel(const float* __restrict__ x, long long n, T* __restrict__ hi, T* __restrict__ lo) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const float v = x[e];
    const T h = to_op<T>(v);
    hi[e] = h;
    if (lo) lo[e] = to_op<T>(v - op_to_float(h));
  }
}

__device__ __forceinline__ float ld_as_float(const float* p, long long i) { return __ldg(p + i); }
__device__ __forceinline__ float ld_as_float(const __half* p, long long i) { return __half2float(p[i]); }
__device__ __forceinline__ float ld_as_float(const __nv_bfloat16* p, long long i) { return __bfloat162float(p[i]); }

// one warp per row
template <typename T>
__global__ void __launch_bounds__(256) row_norms_kernel(const T* __restrict__ A, const T* __restrict__ A2, long long rows, int D,
                                                        float* __restrict__ n2) {
  const long long r = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) {
    float v = ld_as_float(A, r * D + d);
    if (A2) v += ld_as_float(A2, r * D + d);
    s = fmaf(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) n2[r] = s;
}

// ------------------------------------------------------------------------------------------------
// host plan
struct Plan {
  EmbedParams p;
  std::vector<ChunkDesc> chunks;
  struct PerLayer { int chunk_base, nchunks, maxtaps, nch_max; LaunchGeom g; size_t smem; } pl[kMaxLayers];
  bool fused;
};

static int conflict_score(const EmbedParams& p, const ChunkDesc& ck, const LayerDev& ly, int SC, int SR, int SX) {
  // sum over (warp, tap slot) of the worst bank multiplicity for the first column of each thread
  int score = 0;
  std::vector<int> offs;
  for (int w = 0; w < kThreads / 32; ++w) {
    std::vector<std::vector<int>> per_lane(32);
    size_t mx = 0;
    for (int l = 0; l < 32; ++l) {
      const int t = ck.t0 + w * 32 + l;
      if (t >= ck.t1) continue;
      for_each_tap(t, p.agg_in, p.agg_out, p.Dp, ly.CK,
                   [&](int f, float) { per_lane[l].push_back(tap_offset(f, p.k, ck.c_lo, SC, SR, SX)); });
      mx = std::max(mx, per_lane[l].size());
    }
    for (size_t q = 0; q < mx; ++q) {
      int cnt[32] = {0};
      // distinct addresses in the same bank conflict; identical addresses broadcast
      std::vector<int> seen;
      for (int l = 0; l < 32; ++l)
        if (q < per_lane[l].size()) {
          const int a = per_lane[l][q];
          if (std::find(seen.begin(), seen.end(), a) == seen.end()) { seen.push_back(a); cnt[((a % 32) + 32) % 32]++; }
        }
      score += *std::max_element(cnt, cnt + 32);
    }
  }
  return score;
}

static int build_plan(const ac_layer_t* layers, int L, int B, int k, int s, int Dp, int D, int layernorm, float eps,
                      Plan& plan) {
  if (L < 1 || L > kMaxLayers || B < 1 || k < 1 || s < 1 || Dp < 1 || D < 1) return AC_ERR_INVALID;
  EmbedParams& p = plan.p;
  memset(&p, 0, sizeof(p));
  p.L = L; p.B = B; p.k = k; p.s = s; p.pad = (k - 1) / 2; p.Dp = Dp;
  p.layernorm = layernorm; p.eps = eps;
  for (int l = 0; l < L; ++l) {
    const ac_layer_t& a = layers[l];
    if (!a.ptr || a.C < 1 || a.H < 1 || a.W < 1) return AC_ERR_INVALID;
    LayerDev& d = p.layers[l];
    d.ptr = a.ptr; d.C = a.C; d.H = a.H; d.W = a.W;
    d.sb = a.sb; d.sc = a.sc; d.sh = a.sh; d.sw = a.sw;
    d.gh = (a.H + 2 * p.pad - (k - 1) - 1) / s + 1;
    d.gw = (a.W + 2 * p.pad - (k - 1) - 1) / s + 1;
    if (d.gh < 1 || d.gw < 1) return AC_ERR_INVALID;
    d.CK = a.C * k * k;
  }
  p.h0 = p.layers[0].gh; p.w0 = p.layers[0].gw;
  for (int l = 0; l < L; ++l) p.layers[l].resample = (p.layers[l].gh != p.h0 || p.layers[l].gw != p.w0);
  p.agg_in = L * Dp;
  // fused aggregator iff no Aggregator window straddles two layers
  bool fused = true;
  for (int t = 0; t < D && fused; ++t) {
    const int g0 = pool_start(t, p.agg_in, D), g1 = pool_end(t, p.agg_in, D);
    if (g0 / Dp != (g1 - 1) / Dp) fused = false;
  }
  plan.fused = fused;
  p.agg_out = fused ? D : p.agg_in;
  p.ldz = p.agg_out;

  // ---- choose chunking so that the staged tile fits shared memory
  const size_t kSoft = 72 * 1024, kHard = 200 * 1024;
  int tchunk = kThreads * kTPT;
  p.xseg_len = p.w0;
  for (int l = 0; l < L; ++l)
    if (p.layers[l].resample) p.xseg_len = std::min(p.xseg_len, 256);  // s_xo tables hold 256 positions
  for (;;) {
    plan.chunks.clear();
    size_t worst = 0;
    p.nxseg = ceil_div(p.w0, p.xseg_len);
    for (int l = 0; l < L; ++l) {
      const LayerDev& ly = p.layers[l];
      Plan::PerLayer& pl = plan.pl[l];
      pl.chunk_base = (int)plan.chunks.size();
      pl.maxtaps = 0; pl.nch_max = 0;
      // columns owned by this layer
      int ta = -1, tb = -1;
      for (int t = 0; t < p.agg_out; ++t) {
        const int lay = pool_start(t, p.agg_in, p.agg_out) / Dp;
        if (lay == l) { if (ta < 0) ta = t; tb = t + 1; }
      }
      if (ta < 0) { pl.nchunks = 0; continue; }
      for (int t0 = ta; t0 < tb; t0 += tchunk) {
        ChunkDesc ck;
        ck.layer = l; ck.t0 = t0; ck.t1 = std::min(tb, t0 + tchunk);
        int fmin = 1 << 30, fmax = -1, mt = 0;
        for (int t = ck.t0; t < ck.t1; ++t) {
          int n = 0;
          for_each_tap(t, p.agg_in, p.agg_out, Dp, ly.CK, [&](int f, float) { fmin = std::min(fmin, f); fmax = std::max(fmax, f); ++n; });
          mt = std::max(mt, n);
        }
        ck.c_lo = fmin / (k * k);
        ck.nch = fmax / (k * k) - ck.c_lo + 1;
        ck.maxtaps = mt;
        pl.maxtaps = std::max(pl.maxtaps, mt);
        pl.nch_max = std::max(pl.nch_max, ck.nch);
        plan.chunks.push_back(ck);
      }
      pl.nchunks = (int)plan.chunks.size() - pl.chunk_base;
      // tile extents
      LaunchGeom& g = pl.g;
      if (!ly.resample) {
        g.nrows_max = k;
        g.ncols_max = (std::min(p.xseg_len, p.w0) - 1) * s + k;
      } else {
        g.nrows_max = s + k;
        // widest coarse span over all segments
        int span = 1;
        for (int xs = 0; xs < p.nxseg; ++xs) {
          const int xa = xs * p.xseg_len, xb = std::min(p.w0, xa + p.xseg_len);
          int a0, a1, b0, b1; float tmp;
          bilinear_src(xa, ly.gw, p.w0, a0, a1, tmp);
          bilinear_src(xb - 1, ly.gw, p.w0, b0, b1, tmp);
          span = std::max(span, b1 - a0);
        }
        g.ncols_max = span * s + k;
      }
      g.chan_contig = (ly.sc == 1);
      if (g.chan_contig) { g.SC = 1; g.SX = pl.nch_max; g.SR = g.ncols_max * g.SX; }
      else { g.SX = 1; g.SR = g.ncols_max; g.SC = g.nrows_max * g.SR; }
      pl.smem = (size_t)g.nrows_max * g.ncols_max * (pl.nch_max + 32) * sizeof(float);  // incl. padding headroom
      worst = std::max(worst, pl.smem);
    }
    if (worst <= kSoft) break;
    if (tchunk > 32) { tchunk /= 2; continue; }
    if (worst <= kHard) break;
    if (p.xseg_len > 1) { p.xseg_len = (p.xseg_len + 1) / 2; continue; }
    return AC_ERR_UNSUPPORTED;
  }
  // ---- bank-conflict-aware padding of the channel / position pitch
  for (int l = 0; l < L; ++l) {
    Plan::PerLayer& pl = plan.pl[l];
    if (pl.nchunks == 0) continue;
    LaunchGeom& g = pl.g;
    const ChunkDesc& ck = plan.chunks[pl.chunk_base];
    int best = 1 << 30, best_pad = 0;
    for (int padv = 0; padv < 32; ++padv) {
      int SC, SR, SX;
      if (g.chan_contig) { SC = 1; SX = pl.nch_max + padv; SR = g.ncols_max * SX; }
      else { SX = 1; SR = g.ncols_max; SC = g.nrows_max * SR + padv; }
      const int sc = conflict_score(p, ck, p.layers[l], SC, SR, SX);
      if (sc < best) { best = sc; best_pad = padv; }
    }
    if (g.chan_contig) { g.SX = pl.nch_max + best_pad; g.SR = g.ncols_max * g.SX; pl.smem = (size_t)g.nrows_max * g.SR * sizeof(float); }
    else { g.SC = g.nrows_max * g.SR + best_pad; pl.smem = (size_t)pl.nch_max * g.SC * sizeof(float); }
  }
  return AC_OK;
}

template <int MAXTAPS, bool RESAMPLE>
static int launch_embed(const EmbedParams& p, const Plan& plan, int l, const ChunkDesc* dchunks, cudaStream_t st) {
  const Plan::PerLayer& pl = plan.pl[l];
  auto kern = embed_kernel<MAXTAPS, RESAMPLE>;
  AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  dim3 grid(pl.nchunks, p.h0 * p.nxseg, p.B);
  kern<<<grid, kThreads, pl.smem, st>>>(p, dchunks, pl.chunk_base, pl.g);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

template <bool RESAMPLE>
static int dispatch_taps(const EmbedParams& p, const Plan& plan, int l, const ChunkDesc* dchunks, cudaStream_t st) {
  const int mt = plan.pl[l].maxtaps;
  if (mt <= 5) return launch_embed<5, RESAMPLE>(p, plan, l, dchunks, st);
  if (mt <= 10) return launch_embed<10, RESAMPLE>(p, plan, l, dchunks, st);
  if (mt <= 18) return launch_embed<18, RESAMPLE>(p, plan, l, dchunks, st);
  if (mt <= 32) return launch_embed<32, RESAMPLE>(p, plan, l, dchunks, st);
  return launch_embed<0, RESAMPLE>(p, plan, l, dchunks, st);
}

// ---- periodic fast path: eligibility and dispatch
struct Periodic { int ok, A, B, R, nperiods, t_base, transpose, upsample, ncols; };

static int gcd_i(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

static Periodic periodic_of(const Plan& plan, int l) {
  Periodic pr = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  const EmbedParams& p = plan.p;
  const LayerDev& ly = p.layers[l];
  if (!plan.fused || p.s != 1 || p.k != 3) return pr;
  if (p.agg_in % p.agg_out != 0) return pr;
  const int R = p.agg_in / p.agg_out;
  if (p.Dp % R != 0) return pr;
  const int g = gcd_i(ly.CK, p.Dp);
  int a = ly.CK / g, b = p.Dp / g;
  if (a % (p.k * p.k) != 0) return pr;
  if (b % R != 0) {
    const int f = R / gcd_i(b, R);
    if (g % f != 0) return pr;
    a *= f; b *= f;
  }
  pr.A = a; pr.B = b; pr.R = R; pr.nperiods = p.Dp / b; pr.t_base = l * (p.Dp / R);
  pr.transpose = (ly.sc != 1);      // CNN layout: go through a channel-contiguous scratch copy
  pr.upsample = ly.resample;        // pool at the layer's own grid, then resample
  pr.ncols = p.Dp / R;
  pr.ok = 1;
  return pr;
}

#define AC_PERIODIC_CASES(X) \
  X(27, 4, 1) X(27, 8, 1) X(27, 16, 1) X(9, 1, 1) X(9, 2, 1) X(9, 4, 1) X(18, 1, 1) \
  X(9, 2, 2) X(18, 2, 2) X(9, 4, 2) X(27, 8, 2) X(27, 16, 2)

static bool periodic_instantiated(const Periodic& pr) {
#define X(a, b, r) if (pr.A == a && pr.B == b && pr.R == r) return true;
  AC_PERIODIC_CASES(X)
#undef X
  return false;
}

static int g_embed_variant = 0;   // test hook (ac_debug_set key 2): 0 = auto, 1 = force LDG periodic, 2 = force generic tap kernel, 3 = per-layer TMA launches

static bool tma_aligned(const EmbedParams& p, int l) {
  const LayerDev& ly = p.layers[l];
  if (ly.C % 4 != 0) return false;
  if ((reinterpret_cast<uintptr_t>(ly.ptr) & 15) != 0) return false;
  return (ly.sb % 4 == 0) && (ly.sh % 4 == 0) && (ly.sw % 4 == 0);
}

static int launch_periodic(EmbedParams p, const Periodic& pr, int l, int num_sms, cudaStream_t st) {
  // split rows into x segments until the launch has a few waves of CTAs
  const int gx = ceil_div(pr.nperiods, kThreads);
  const long long base_blocks = (long long)gx * p.h0 * p.B;
  int nxseg = (int)std::min<long long>(std::max<long long>(1, (num_sms * 16LL + base_blocks - 1) / base_blocks), std::max(1, p.w0 / 4));
  p.xseg_len = ceil_div(p.w0, nxseg);
  p.nxseg = ceil_div(p.w0, p.xseg_len);
  dim3 grid(gx, p.h0 * p.nxseg, p.B);
  const bool use_tma = (g_embed_variant == 0 || g_embed_variant == 3) && tma_aligned(p, l);
#define X(a, b, r)                                                                                         \
  if (pr.A == a && pr.B == b && pr.R == r) {                                                               \
    if (use_tma) {                                                                                         \
      auto kern = embed_tma_kernel<a, b, 3, r>;                                                            \
      const size_t smem = (size_t)kRing * 3 * kThreads * (a / 9) * sizeof(float);                          \
      AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));         \
      kern<<<grid, kThreads + 32, smem, st>>>(p, l, pr.t_base, pr.nperiods);                               \
    } else {                                                                                               \
      embed_periodic_kernel<a, b, 3, r><<<grid, kThreads, 0, st>>>(p, l, pr.t_base, pr.nperiods);          \
    }                                                                                                      \
    AC_LAUNCH_CHECK();                                                                                     \
    return AC_OK;                                                                                          \
  }
  AC_PERIODIC_CASES(X)
#undef X
  return AC_ERR_UNSUPPORTED;
}

// ---- single-pass fused form: eligibility and launch
static constexpr int kLookAhead = 2;   // images the statistics run ahead of the embedding
static constexpr int kCtasPerSm = 3;   // persistent CTAs per SM (the lean kernel: at most its MINB)

static bool fused_eligible(const Plan& plan, const EmbedParams& p, const Periodic* pr, int L) {
  if (g_embed_variant != 0 || !plan.fused || p.k != 3 || p.s != 1) return false;
  for (int l = 0; l < L; ++l) {
    if (plan.pl[l].nchunks == 0 || !tma_aligned(p, l)) return false;
    if (!pr[l].ok || !periodic_instantiated(pr[l]) || pr[l].transpose || pr[l].upsample) return false;
    if (pr[l].A != pr[0].A || pr[l].B != pr[0].B || pr[l].R != pr[0].R) return false;
    if (p.layers[l].C != p.layers[0].C || p.layers[l].H != p.layers[0].H || p.layers[l].W != p.layers[0].W) return false;
    if (pr[l].t_base != l * pr[0].ncols) return false;
  }
  return true;
}

static constexpr size_t kZeroRowBytes = 12288;  // lean kernel: zeros that stand in for taps outside the map (one ring slot: 3 tokens x <= 768 channels)

static constexpr int kMinSeg = 4;   // the workspace sizes the lean kernel's statistics slots for x segments this short

// workspace of the fused kernels: [mean / rstd per (image, layer)] [statistics partials] [done[B], claim counter] [zero row]
static size_t fused_murs_bytes(int L, int B) { return ((size_t)B * L * sizeof(unsigned long long) + 255) & ~(size_t)255; }
static size_t fused_stats_bytes(int L, int B, int h0, int w0) {
  // general kernel: one (sum, sum of squares) pair of doubles per slice; lean kernel: one packed 64-bit slot per slice and
  // consumer warp (<= 4), slices as short as kMinSeg
  const size_t S_gen = (size_t)h0 * ceil_div(w0, kMaxSeg), S_lean = (size_t)h0 * ceil_div(w0, kMinSeg);
  return (std::max(S_gen * 2 * sizeof(double), S_lean * 4 * sizeof(unsigned long long)) * B * L + 255) & ~(size_t)255;
}
static size_t fused_ctr_bytes(int B) { return (((size_t)B + 64) * sizeof(int) + 255) & ~(size_t)255; }
static size_t fused_ws_bytes(int L, int B, int h0, int w0) {
  return fused_murs_bytes(L, B) + fused_stats_bytes(L, B, h0, w0) + fused_ctr_bytes(B) + kZeroRowBytes;
}

static int g_fused_lean = 1;      // test hook (ac_debug_set key 9): 0 = always the general fused kernel

static int launch_fused(EmbedParams p, const Periodic& pr, float* n2, void* ws, int num_sms, cudaStream_t st) {
  FusedParams fp;
  memset(&fp, 0, sizeof(fp));
  // lean kernel: fp16 operands + norms (+ fp32 Z), every consumer thread owns two periods of every layer
  const bool lean_out = g_fused_lean && p.Zhi && !p.Zlo && p.op_dtype == AC_DT_F16 && n2 && pr.R == 1 && pr.A == 27 &&
                        (p.ldz % 8 == 0) && (pr.ncols % 8 == 0) && (reinterpret_cast<uintptr_t>(p.Zhi) % 16 == 0) &&
                        (!p.Z || reinterpret_cast<uintptr_t>(p.Z) % 16 == 0) && p.h0 == p.w0;   // slices: row runs / column runs
  p.nxseg = ceil_div(p.w0, kMaxSeg);
  p.xseg_len = ceil_div(p.w0, p.nxseg);
  p.nxseg = ceil_div(p.w0, p.xseg_len);
  p.b0 = 0;
  fp.n2 = n2;
  fp.S = p.h0 * p.nxseg;
  fp.LA = std::max(1, std::min(kLookAhead, p.B));
  fp.nperiods = pr.nperiods;
  fp.gx = ceil_div(pr.nperiods, kFT * kPP);
  fp.t_stride = pr.ncols;
  fp.n_items = (long long)(p.B + fp.LA) * fp.S;
  const size_t murs_b = fused_murs_bytes(p.L, p.B), stats_b = fused_stats_bytes(p.L, p.B, p.h0, p.w0), ctr_b = fused_ctr_bytes(p.B);
  fp.murs = (unsigned long long*)ws;
  fp.stats = (double*)((char*)ws + murs_b);
  fp.done = (int*)((char*)ws + murs_b + stats_b);
  fp.counter = (unsigned int*)(fp.done + p.B);
  fp.zero_row = (const float*)((char*)fp.done + ctr_b);
  fp.e = p;
  // one launch: mean / rstd and the lean kernel's statistics slots = all-ones ("unset", see kUnset); done[B], the claim counter
  // and the zero row = 0
  const long long ones = (long long)((murs_b + (lean_out ? (size_t)p.B * p.L * fp.S * 4 * sizeof(unsigned long long) : 0)) / 4);
  const long long zeros = (long long)((ctr_b + kZeroRowBytes) / 4);
  init_words_kernel<<<(unsigned)std::min<long long>((ones + zeros + 255) / 256, 296), 256, 0, st>>>((unsigned int*)ws, ones, (unsigned int*)fp.done,
                                                                                                   zeros);
  AC_LAUNCH_CHECK();
#define XLK(b, ft, wz, ring, minb)                                                                                    \
  {                                                                                                                   \
    const size_t smem = ((size_t)ring * 3 * ft * kPP * 3 + (size_t)kMaxSeg * ft) * sizeof(float);                     \
    const int grid_l = (int)std::min<long long>(fp.n_items, (long long)num_sms * std::min(kCtasPerSm, minb));         \
    auto kern = embed_fused_fast_kernel<27, b, 1, ft, wz, ring, minb>;                                                \
    AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                      \
    kern<<<grid_l, ft + 32, smem, st>>>(fp);                                                                          \
    AC_LAUNCH_CHECK();                                                                                                \
    return AC_OK;                                                                                                     \
  }
#define XL(b, ft)                                                                                                     \
  if (lean_out && pr.B == b && pr.nperiods == ft * kPP && p.layers[0].C == ft * kPP * 3) {                            \
    if (p.Z) XLK(b, ft, true, kRingL, (ft == 128 ? 3 : 5)) else XLK(b, ft, false, kRingL, (ft == 128 ? 3 : 5))        \
  }
  XL(8, 128) XL(4, 128) XL(16, 64)
#undef XL
#undef XLK
  const int grid = (int)std::min<long long>(fp.n_items, (long long)num_sms * kCtasPerSm);
#define X(a, b, r)                                                                                                   \
  if (pr.A == a && pr.B == b && pr.R == r) {                                                                         \
    auto kern = embed_fused_kernel<a, b, r>;                                                                         \
    const size_t smem = ((size_t)kRing * 3 * kFT * kPP * (a / 9) + (size_t)kMaxSeg * kFT) * sizeof(float);           \
    AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                     \
    kern<<<grid, kFT + 32, smem, st>>>(fp);                                                                          \
    AC_LAUNCH_CHECK();                                                                                               \
    return AC_OK;                                                                                                    \
  }
  AC_PERIODIC_CASES(X)
#undef X
  return AC_ERR_UNSUPPORTED;
}

// ---- plan cache: building a plan walks every output column; reuse it across calls of one shape
struct PlanKey {
  int L, k, s, Dp, D, layernorm;
  int C[kMaxLayers], H[kMaxLayers], W[kMaxLayers];
  long long sc[kMaxLayers], sh[kMaxLayers], sw[kMaxLayers];
  bool operator==(const PlanKey& o) const { return memcmp(this, &o, sizeof(PlanKey)) == 0; }
};

static std::mutex g_plan_mu;
static std::vector<std::pair<PlanKey, std::shared_ptr<Plan>>> g_plans;

static int get_plan(const ac_layer_t* layers, int L, int k, int s, int Dp, int D, int layernorm, float eps,
                    std::shared_ptr<Plan>& out) {
  if (L < 1 || L > kMaxLayers) return AC_ERR_INVALID;
  PlanKey key;
  memset(&key, 0, sizeof(key));
  key.L = L; key.k = k; key.s = s; key.Dp = Dp; key.D = D; key.layernorm = layernorm;
  for (int l = 0; l < L; ++l) {
    key.C[l] = layers[l].C; key.H[l] = layers[l].H; key.W[l] = layers[l].W;
    key.sc[l] = layers[l].sc; key.sh[l] = layers[l].sh; key.sw[l] = layers[l].sw;
  }
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto& e : g_plans)
      if (e.first == key) { out = e.second; return AC_OK; }
  }
  auto plan = std::make_shared<Plan>();
  int rc = build_plan(layers, L, 1, k, s, Dp, D, layernorm, eps, *plan);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g_plan_mu);
  if (g_plans.size() >= 16) g_plans.erase(g_plans.begin());
  g_plans.emplace_back(key, plan);
  out = plan;
  return AC_OK;
}

}  // namespace ac

using namespace ac;

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static bool aggregator_fusable(int L, int Dp, int D) {
  const int agg_in = L * Dp;
  for (int t = 0; t < D; ++t) {
    const int g0 = pool_start(t, agg_in, D), g1 = pool_end(t, agg_in, D);
    if (g0 / Dp != (g1 - 1) / Dp) return false;
  }
  return true;
}

// scratch needed by the layout / grid adapters of the fast path (upper bound: assumes every layer uses them)
static size_t adapter_bytes(const ac_layer_t* layers, int L, int B, int k, int s, int Dp, int D, size_t* per_layer_t, size_t* per_layer_c) {
  size_t total = 0;
  const int pad = (k - 1) / 2;
  const int R = std::max(1, (L * Dp) / std::max(1, D));
  for (int l = 0; l < L; ++l) {
    const size_t tb = align256((size_t)B * layers[l].C * layers[l].H * layers[l].W * sizeof(float));
    const int gh = (layers[l].H + 2 * pad - (k - 1) - 1) / s + 1, gw = (layers[l].W + 2 * pad - (k - 1) - 1) / s + 1;
    const size_t cb = align256((size_t)B * std::max(1, gh) * std::max(1, gw) * (size_t)(Dp / R + 4) * sizeof(float));
    if (per_layer_t) per_layer_t[l] = tb;
    if (per_layer_c) per_layer_c[l] = cb;
    total += tb + cb;
  }
  return total;
}

extern "C" size_t ac_embed_workspace_bytes(const ac_layer_t* layers, int L, int B, int patchsize, int stride, int Dp, int D) {
  if (!layers || L < 1 || L > kMaxLayers || B < 1 || patchsize < 1 || stride < 1 || Dp < 1 || D < 1) return 0;
  const int pad = (patchsize - 1) / 2;
  const long long P = (long long)((layers[0].H + 2 * pad - (patchsize - 1) - 1) / stride + 1) *
                      ((layers[0].W + 2 * pad - (patchsize - 1) - 1) / stride + 1);
  if (P < 1) return 0;
  size_t stats = align256((size_t)B * L * kStatSplit * 2 * sizeof(double));
  size_t chunks = align256(((size_t)L * Dp / 32 + (size_t)D / 32 + 2 * L + 16) * sizeof(ChunkDesc));
  // the [B*P, L*Dp] concat scratch exists only when an Aggregator window straddles two layers
  size_t concat = aggregator_fusable(L, Dp, D) ? 0 : align256((size_t)B * P * (size_t)L * Dp * sizeof(float));
  // channel-contiguous copies of CNN-layout maps + coarse pooled tiles of resampled layers (fast path)
  bool any_adapter = false;
  for (int l = 0; l < L; ++l) {
    const int gh = (layers[l].H + 2 * pad - (patchsize - 1) - 1) / stride + 1, gw = (layers[l].W + 2 * pad - (patchsize - 1) - 1) / stride + 1;
    if (layers[l].sc != 1 || (long long)gh * gw != P) any_adapter = true;
  }
  size_t adapters = any_adapter ? adapter_bytes(layers, L, B, patchsize, stride, Dp, D, nullptr, nullptr) : 0;
  // statistics slices + image counters of the single-pass fused form (at the end of the workspace)
  const int gh0 = (layers[0].H + 2 * pad - (patchsize - 1) - 1) / stride + 1, gw0 = (layers[0].W + 2 * pad - (patchsize - 1) - 1) / stride + 1;
  return stats + chunks + concat + adapters + fused_ws_bytes(L, B, gh0, gw0) + 256;
}

extern "C" int ac_embed_ex(const ac_layer_t* layers, int L, int B, int patchsize, int stride, int Dp, int D, int layernorm,
                           float eps, float* Z, void* Zhi, void* Zlo, int op_dtype, float* n2, void* ws, size_t ws_bytes,
                           ac_stream_t stream) {
  if (!layers || !ws) return AC_ERR_INVALID;
  if (!Z && !Zhi) return AC_ERR_INVALID;
  if (n2 && !Zhi) return AC_ERR_INVALID;
  if (Zhi && op_dtype != AC_DT_F16 && op_dtype != AC_DT_BF16) return AC_ERR_INVALID;
  if (Zlo && !Zhi) return AC_ERR_INVALID;
  if (B < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  std::shared_ptr<Plan> plan_sp;
  rc = get_plan(layers, L, patchsize, stride, Dp, D, layernorm, eps, plan_sp);
  if (rc) return rc;
  const Plan& plan = *plan_sp;
  // operand-only output needs the fused aggregator (no Aggregator window straddling two layers): refuse BEFORE anything is
  // enqueued -- callers ask for Z as well in that case (pipeline.embed_images does)
  if (!plan.fused && !Z) return AC_ERR_UNSUPPORTED;
  EmbedParams p = plan.p;   // cached geometry; pointers and batch are per call
  p.eps = eps;
  for (int l = 0; l < L; ++l) {
    if (!layers[l].ptr) return AC_ERR_INVALID;
    p.layers[l].ptr = layers[l].ptr;
    p.layers[l].sb = layers[l].sb;
  }
  const long long P0 = (long long)p.h0 * p.w0;

  const size_t stats_b = align256((size_t)B * L * kStatSplit * 2 * sizeof(double));
  const size_t chunks_b = align256(plan.chunks.size() * sizeof(ChunkDesc));
  const size_t concat_b = plan.fused ? 0 : align256((size_t)B * P0 * p.agg_in * sizeof(float));
  if (stats_b + chunks_b + concat_b > ws_bytes) return AC_ERR_WORKSPACE;
  char* w8 = (char*)ws;
  double* dstats = (double*)w8;
  ChunkDesc* dchunks = (ChunkDesc*)(w8 + stats_b);
  float* dconcat = (float*)(w8 + stats_b + chunks_b);

  Periodic pr[kMaxLayers];
  bool need_chunks = false, any_adapter = false;
  for (int l = 0; l < L; ++l) {
    pr[l] = periodic_of(plan, l);
    if (pr[l].ok && (!periodic_instantiated(pr[l]) || g_embed_variant == 2)) pr[l].ok = 0;
    if (!pr[l].ok && plan.pl[l].nchunks > 0) need_chunks = true;
    if (pr[l].ok && (pr[l].transpose || pr[l].upsample)) any_adapter = true;
  }
  // scratch of the layout / grid adapters (only carved when a fast-path layer needs one)
  size_t tb[kMaxLayers], cb[kMaxLayers];
  float* tbuf[kMaxLayers] = {nullptr};
  float* cbuf[kMaxLayers] = {nullptr};
  if (any_adapter) {
    const size_t ad = adapter_bytes(layers, L, B, patchsize, stride, Dp, D, tb, cb);
    if (stats_b + chunks_b + concat_b + ad > ws_bytes) return AC_ERR_WORKSPACE;
    char* cur = w8 + stats_b + chunks_b + concat_b;
    for (int l = 0; l < L; ++l) {
      tbuf[l] = (float*)cur; cur += tb[l];
      cbuf[l] = (float*)cur; cur += cb[l];
    }
  }
  if (need_chunks)
    AC_CUDA(cudaMemcpyAsync(dchunks, plan.chunks.data(), plan.chunks.size() * sizeof(ChunkDesc), cudaMemcpyHostToDevice, st));

  p.stats = dstats;
  if (plan.fused) {
    p.Z = Z; p.Zhi = Zhi; p.Zlo = Zlo; p.op_dtype = op_dtype;
  } else {
    p.Z = dconcat; p.Zhi = nullptr; p.Zlo = nullptr; p.op_dtype = 0;
  }
  int dev = 0, num_sms = 148;
  AC_CUDA(cudaGetDevice(&dev));
  AC_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));

  // Single-pass fused form (one persistent launch: statistics, every layer, operand norms) when the shape allows it
  if (fused_eligible(plan, p, pr, L)) {
    const size_t fb = fused_ws_bytes(L, B, p.h0, p.w0) + 256;
    if (fb > ws_bytes || (reinterpret_cast<uintptr_t>(ws) & 15) != 0) return AC_ERR_WORKSPACE;
    p.B = B;
    return launch_fused(p, pr[0], n2, w8 + ((ws_bytes - fb) & ~(size_t)255), num_sms, st);
  }

  // One statistics launch and one embed launch per layer for the whole batch.  Measured on B200:
  // L2-sized sub-batches (statistics + embed sharing the maps in L2) cost more in launch tails than
  // the second HBM read of the feature maps (20 % of the traffic) saves.  grid.z is limited to 65535.
  const int nb = std::min(B, 65535);
  for (int b0 = 0; b0 < B; b0 += nb) {
    p.b0 = b0;
    p.B = std::min(nb, B - b0);
    if (layernorm) {
      ln_stats_kernel<<<dim3(kStatSplit, L, p.B), 256, 0, st>>>(p, dstats);
      AC_LAUNCH_CHECK();
    }
    for (int l = 0; l < L; ++l) {
      if (plan.pl[l].nchunks == 0) continue;
      if (!pr[l].ok) {
        rc = p.layers[l].resample ? dispatch_taps<true>(p, plan, l, dchunks, st) : dispatch_taps<false>(p, plan, l, dchunks, st);
        if (rc) return rc;
        continue;
      }
      EmbedParams q = p;
      Periodic prl = pr[l];
      LayerDev& ly = q.layers[l];
      if (prl.transpose) {
        // CNN layout -> channel-contiguous scratch [B, H*W, C]
        dim3 tg(ceil_div(ly.H * ly.W, 32), ceil_div(ly.C, 32), q.B);
        nchw_to_nhwc_kernel<<<tg, 256, 0, st>>>(p.layers[l], q.b0, tbuf[l]);
        AC_LAUNCH_CHECK();
        ly.ptr = tbuf[l] - (long long)q.b0 * ly.C * ly.H * ly.W;   // kernels index images as b0 + blockIdx.z
        ly.sb = (long long)ly.C * ly.H * ly.W; ly.sc = 1; ly.sh = (long long)ly.W * ly.C; ly.sw = ly.C;
      }
      if (prl.upsample) {
        // pool at the layer's own patch grid into scratch [B, gh*gw, ncols], resample afterwards
        q.h0 = ly.gh; q.w0 = ly.gw;
        q.Z = cbuf[l] - (long long)q.b0 * ly.gh * ly.gw * prl.ncols;
        q.Zhi = nullptr; q.Zlo = nullptr; q.op_dtype = 0; q.ldz = prl.ncols;
        prl.t_base = 0;
      }
      rc = launch_periodic(q, prl, l, num_sms, st);
      if (rc) return rc;
      if (prl.upsample) {
        const long long groups = (long long)p.B * p.h0 * p.w0 * ((prl.ncols + 3) / 4);
        const int blocks = (int)std::min<long long>((groups + 255) / 256, (long long)num_sms * 32);
        upsample_store_kernel<<<blocks, 256, 0, st>>>(p, cbuf[l], ly.gh, ly.gw, prl.ncols, pr[l].t_base);
        AC_LAUNCH_CHECK();
      }
    }
  }
  if (!plan.fused) {
    // Aggregator windows straddle layers: pool the concat [B*P, L*Dp] -> [B*P, D] in a second pass
    const long long rows = (long long)B * P0;
    float* zout = Z;
    if (!zout) return AC_ERR_UNSUPPORTED;  // operand-only output needs the fused aggregator
    const long long total = rows * D;
    int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    pool1d_kernel<<<blocks, 256, 0, st>>>(dconcat, rows, p.agg_in, D, zout);
    AC_LAUNCH_CHECK();
    if (Zhi) {
      rc = ac_split_operand(zout, total, Zhi, Zlo, op_dtype, stream);
      if (rc) return rc;
    }
  }
  if (n2) return ac_row_norms(Zhi, Zlo, op_dtype, (long long)B * P0, D, n2, stream);
  return AC_OK;
}

extern "C" int ac_embed(const ac_layer_t* layers, int L, int B, int patchsize, int stride, int Dp, int D, int layernorm,
                        float eps, float* Z, void* Zhi, void* Zlo, int op_dtype, void* ws, size_t ws_bytes,
                        ac_stream_t stream) {
  return ac_embed_ex(layers, L, B, patchsize, stride, Dp, D, layernorm, eps, Z, Zhi, Zlo, op_dtype, nullptr, ws, ws_bytes, stream);
}

// test hook (not part of the public header): forces the embedding paths the library otherwise picks from the input.
//   key 2 = kernel variant: 0 auto, 1 LDG periodic, 2 generic tap kernel, 3 per-layer launches (TMA kernel where it applies)
//   key 9 = lean fused kernel: 1 when eligible, 0 always the general fused kernel
extern "C" int ac_debug_set(int key, int value) {
  if (key == 2 && value >= 0 && value <= 3) { g_embed_variant = value; return AC_OK; }
  if (key == 9 && (value == 0 || value == 1)) { g_fused_lean = value; return AC_OK; }
  return AC_ERR_INVALID;
}

extern "C" size_t ac_weighted_embed_from_features_workspace_bytes(const ac_layer_t* layers, int L, int B, int patchsize) {
  if (!layers || L < 1 || L > kMaxLayers || B < 1 || patchsize < 1) return 0;
  size_t stats = align256((size_t)B * L * kStatSplit * 2 * sizeof(double));
  size_t part = 0;
  for (int l = 0; l < L; ++l) part = std::max(part, align256((size_t)B * kXSplit * patchsize * patchsize * layers[l].C * sizeof(float)));
  return stats + part;
}

extern "C" int ac_weighted_embed_from_features(const ac_layer_t* layers, int L, int B, int patchsize, int stride, int Dp, int D,
                                               int layernorm, float eps, const float* alpha, float* X, void* ws, size_t ws_bytes,
                                               ac_stream_t stream) {
  if (!layers || !alpha || !X || !ws || B < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  std::shared_ptr<Plan> plan_sp;
  rc = get_plan(layers, L, patchsize, stride, Dp, D, layernorm, eps, plan_sp);
  if (rc) return rc;
  const Plan& plan = *plan_sp;
  if (!plan.fused || patchsize != 3 || stride != 1) return AC_ERR_UNSUPPORTED;   // Aggregator windows inside one layer, 3x3 patches
  EmbedParams p = plan.p;
  p.eps = eps;
  for (int l = 0; l < L; ++l) {
    if (!layers[l].ptr) return AC_ERR_INVALID;
    if (p.layers[l].resample) return AC_ERR_UNSUPPORTED;                          // all layers on the layer-0 grid
    p.layers[l].ptr = layers[l].ptr;
    p.layers[l].sb = layers[l].sb;
  }
  const size_t need = ac_weighted_embed_from_features_workspace_bytes(layers, L, B, patchsize);
  if (ws_bytes < need) return AC_ERR_WORKSPACE;
  const size_t stats_b = align256((size_t)B * L * kStatSplit * 2 * sizeof(double));
  double* dstats = (double*)ws;
  float* part = (float*)((char*)ws + stats_b);
  p.stats = dstats;
  const int nb = std::min(B, 65535);
  const size_t smem = (size_t)(p.h0 + 2 * p.pad) * (p.w0 + 2 * p.pad) * sizeof(float);
  if (smem > 200 * 1024) return AC_ERR_UNSUPPORTED;
  if (smem > 48 * 1024) AC_CUDA(cudaFuncSetAttribute(xcorr_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int b0 = 0; b0 < B; b0 += nb) {
    p.b0 = b0;
    p.B = std::min(nb, B - b0);
    if (layernorm) {
      ln_stats_kernel<<<dim3(kStatSplit, L, p.B), 256, 0, st>>>(p, dstats);
      AC_LAUNCH_CHECK();
    }
    for (int l = 0; l < L; ++l) {
      // output columns owned by layer l (fused Aggregator: contiguous range)
      int ta = -1, tb = -1;
      for (int t = 0; t < p.agg_out; ++t)
        if (pool_start(t, p.agg_in, p.agg_out) / Dp == l) { if (ta < 0) ta = t; tb = t + 1; }
      if (ta < 0) continue;
      xcorr_kernel<3><<<dim3(ceil_div(p.layers[l].C, 256), kXSplit, p.B), 256, smem, st>>>(p, l, alpha + (long long)b0 * p.h0 * p.w0, part);
      AC_LAUNCH_CHECK();
      xpool_kernel<<<dim3(ceil_div(tb - ta, 256), p.B), 256, 0, st>>>(p, l, ta, tb, part, X);
      AC_LAUNCH_CHECK();
    }
  }
  return AC_OK;
}

extern "C" int ac_patchify(const float* x, int B, int C, int H, int W, int patchsize, int stride, float* out,
                           int* grid_host, ac_stream_t stream) {
  if (!x || !out || B < 1 || C < 1 || H < 1 || W < 1 || patchsize < 1 || stride < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  const int pad = (patchsize - 1) / 2;
  const int gh = (H + 2 * pad - (patchsize - 1) - 1) / stride + 1;
  const int gw = (W + 2 * pad - (patchsize - 1) - 1) / stride + 1;
  if (gh < 1 || gw < 1) return AC_ERR_INVALID;
  if (grid_host) { grid_host[0] = gh; grid_host[1] = gw; }
  const long long total = (long long)B * gh * gw * C * patchsize * patchsize;
  int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 32);
  patchify_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, B, C, H, W, patchsize, stride, pad, gh, gw, out);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_adaptive_pool1d(const float* in, int64_t rows, int Lin, int Lout, float* out, ac_stream_t stream) {
  if (!in || !out || rows < 0 || Lin < 1 || Lout < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (rows == 0) return AC_OK;
  const long long total = (long long)rows * Lout;
  int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 32);
  pool1d_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(in, rows, Lin, Lout, out);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_split_operand(const float* x, int64_t n, void* hi, void* lo, int dtype, ac_stream_t stream) {
  if (!x || !hi || n < 0) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (n == 0) return AC_OK;
  int blocks = (int)std::min<long long>((n + 255) / 256, 148 * 32);
  if (dtype == AC_DT_F16)
    split_kernel<__half><<<blocks, 256, 0, (cudaStream_t)stream>>>(x, n, (__half*)hi, (__half*)lo);
  else if (dtype == AC_DT_BF16)
    split_kernel<__nv_bfloat16><<<blocks, 256, 0, (cudaStream_t)stream>>>(x, n, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo);
  else
    return AC_ERR_INVALID;
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_row_norms(const void* A, const void* A2, int dtype, int64_t rows, int D, float* n2, ac_stream_t stream) {
  if (!A || !n2 || rows < 0 || D < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (rows == 0) return AC_OK;
  const int wpb = 8;
  const unsigned blocks = (unsigned)((rows + wpb - 1) / wpb);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == AC_DT_F32)
    row_norms_kernel<float><<<blocks, 256, 0, st>>>((const float*)A, (const float*)A2, rows, D, n2);
  else if (dtype == AC_DT_F16)
    row_norms_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)A, (const __half*)A2, rows, D, n2);
  else if (dtype == AC_DT_BF16)
    row_norms_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)A, (const __nv_bfloat16*)A2, rows, D, n2);
  else
    return AC_ERR_INVALID;
  AC_LAUNCH_CHECK();
  return AC_OK;
}
