// Exact re-evaluation of the nearest-neighbour distances the tensor-core pass SELECTED (precision mode "f16r").
//
// The tcgen05 pass (mindist_tc.cu) finds, per (query row r, bank image j), the nearest bank row -- torch.cdist +
// torch.min(dim=1) of Weight_Distance_* (reference: Anomaly-Clustering/models/patchcore/utils.py:226, :233-234) -- but
// its distance carries the tensor core's fp32 accumulation error over K = D products of magnitude |q||b| (systematic,
// ~3e-3 absolute at config 2: too much for softmax(w / tau) once tau < 1).  The arg-min is far more robust than the
// value, so that pass also records WHICH row won (ac_min_dist_arg / ac_min_dist_sym_arg) and this kernel recomputes
//      d(r, j) = || q_r - b_(j,c) ||,   c = arg-min row of image j for query row r,
// with IEEE fp32 FMAs (round to nearest, 128 short partial sums per pair): one gathered bank row (fp16/bf16 operand, + its
// lo part if present) per pair against the query row held in shared memory as fp32 (from fp32 Z when the caller has
// it -- measured: the query row must NOT be the rounded operand, its rounding error is common to all bank images and
// does not average out).  When the caller passes the bank rows' squared norms the pair costs one FFMA per element
// (|q|^2 + |b|^2 - 2 q.b, |q|^2 summed in the kernel; the cancellation costs ~1e-6 absolute in d), else sum (q-b)^2.
// Cost: one 2*D-byte row per pair from L2 -- 64 GB at config 2.
//
// Blocking: grid = (query chunks of kRQ rows, groups of Jb bank images); blocks are dispatched x-fastest, so all
// resident blocks gather from the same Jb bank images (they stay in L2) while the query chunks stream past once per group.
#include "common.cuh"
#include <algorithm>

namespace ac {

static constexpr int kRQ = 4;            // query rows per block (fp32 in shared memory)
static constexpr int kWPR = 4;           // warps per query row: they take every kWPR-th bank image of the group
static constexpr int kRefThreads = kRQ * kWPR * 32;
static constexpr int kRefineL2MB = 128;  // MB of bank operand rows one group keeps L2-resident (evict_last; measured at config 2
                                         // with the policy hints: 32 / 64 / 96 / 128 / 192 / 256 MB -> 14.7 / 11.6 / 11.8 / 10.3 / 10.8 / 10.8 ms)

// L2 policies: the gathered bank rows of a group (<= 96 MB) are re-read by every query chunk and must stay L2-resident while
// the 16 KB fp32 query rows, the arg-min tables and the results stream through once per group (round-2 capture before the
// hints: 28 GB of DRAM reads for 12.5 GB compulsory, L2 hit rate 47 %)
__device__ __forceinline__ uint64_t l2_policy_keep() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint4 ld_hint(const uint4* p, uint64_t pol) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
// (no L1::no_allocate here: a thread reads the two 16-byte halves of a 32-byte sector with two loads, and without L1 each
// of them fetched the sector from L2 again -- measured +12 GB of L2 -> SM traffic)
__device__ __forceinline__ float4 ld_hint(const float4* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p), "l"(pol));
  return v;
}

struct RefineParams {
  const float* Zq;                    // [Mq, D] fp32 or null
  const void* Qhi; const void* Qlo;   // [Mq, D] operand copies (used when Zq is null)
  const void* Bhi; const void* Blo;   // [nb_img*P, D]
  long long Mq;
  int nb_img, P, D, Pq;
  const int* rowarg;                  // [nb_img, Mq]
  const unsigned long long* colkey;   // [nb_img, Mq] (sym) or null
  int sym, q_img0;
  const int* q_self;                  // non-sym: bank index of each query image (its pair is skipped) or null
  const int* groups;                  // sym: (first image, count) of the category of every bank image, or null
  const float* Bn2;                   // [nb_img*P] squared norms of the bank rows as gathered (hi, or hi + lo), or null
  float* dex;                         // [nb_img, Mq]
  int Jb;
  // growth (ac_refine_min_dist_grow): query row r is row r0 + r of the whole category (its fp32 Z row: Zq + r*D), partners are
  // images [jbase, nb_img); rowarg / dex [nb_img, Mn] over the Mn = (nb_img - n_old) * P new rows, colkey / dcol [nb_img - n_old,
  // nb_img * P] over every row of the category
  int n_old, jbase;
  long long r0, Mn;
  float* dcol;
};

template <typename T> __device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]);
template <> __device__ __forceinline__ void unpack8<__half>(const uint4& u, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 v = __half22float2(h[i]); f[2 * i] = v.x; f[2 * i + 1] = v.y; }
}
template <> __device__ __forceinline__ void unpack8<__nv_bfloat16>(const uint4& u, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 v = __bfloat1622float2(h[i]); f[2 * i] = v.x; f[2 * i + 1] = v.y; }
}

// sum_k (q[k] - b[k])^2 over one row: lane owns the 16-byte groups g = lane, lane + 32, ...  NIT > 0: trip count known
// at compile time (D = 256 * NIT), fully unrolled -- all NIT loads of the gathered row are in flight before the first use.
// DOT: accumulate q.b (one FFMA per element) instead of (q-b)^2.
template <typename T, int NIT, bool LO, bool DOT>
__device__ __forceinline__ float row_dist2(const uint4* __restrict__ bh, const uint4* __restrict__ bl, const float4* qlo4,
                                           const float4* qhi4, int G8, int lane, uint64_t pol_keep) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  float2 A = make_float2(0.f, 0.f), B = make_float2(0.f, 0.f);   // DOT: (a0, a1) and (a2, a3) as packed accumulators
  auto body = [&](const uint4& ub, int g) {
    float b[8];
    unpack8<T>(ub, b);
    if (LO) {
      float l[8];
      unpack8<T>(__ldg(bl + g), l);
#pragma unroll
      for (int t = 0; t < 8; ++t) b[t] += l[t];
    }
    const float4 ql = qlo4[g], qh = qhi4[g];
    if (DOT) {
      // same four accumulation chains as the scalar form (bit-identical), two per packed fma.rn.f32x2
      A = __ffma2_rn(make_float2(ql.x, ql.y), make_float2(b[0], b[1]), A);
      B = __ffma2_rn(make_float2(ql.z, ql.w), make_float2(b[2], b[3]), B);
      A = __ffma2_rn(make_float2(qh.x, qh.y), make_float2(b[4], b[5]), A);
      B = __ffma2_rn(make_float2(qh.z, qh.w), make_float2(b[6], b[7]), B);
    } else {
      float d;
      d = ql.x - b[0]; a0 = fmaf(d, d, a0);
      d = ql.y - b[1]; a1 = fmaf(d, d, a1);
      d = ql.z - b[2]; a2 = fmaf(d, d, a2);
      d = ql.w - b[3]; a3 = fmaf(d, d, a3);
      d = qh.x - b[4]; a0 = fmaf(d, d, a0);
      d = qh.y - b[5]; a1 = fmaf(d, d, a1);
      d = qh.z - b[6]; a2 = fmaf(d, d, a2);
      d = qh.w - b[7]; a3 = fmaf(d, d, a3);
    }
  };
  if (NIT > 0) {
    // batches of up to 8 independent 16-byte loads in flight per lane (the compiler barrier keeps ptxas from
    // re-serialising them to save registers -- measured in SASS: 3 in flight without it)
    constexpr int kBatch = NIT > 8 ? 8 : (NIT > 0 ? NIT : 1);
#pragma unroll
    for (int it0 = 0; it0 < NIT; it0 += kBatch) {
      uint4 u[kBatch];
#pragma unroll
      for (int it = 0; it < kBatch; ++it) u[it] = ld_hint(bh + lane + 32 * (it0 + it), pol_keep);
      asm volatile("" ::: "memory");
#pragma unroll
      for (int it = 0; it < kBatch; ++it) body(u[it], lane + 32 * (it0 + it));
    }
  } else {
#pragma unroll 4
    for (int g = lane; g < G8; g += 32) body(ld_hint(bh + g, pol_keep), g);
  }
  if (DOT) return (A.x + A.y) + (B.x + B.y);
  return (a0 + a1) + (a2 + a3);
}

template <typename T, int NIT, bool LO, bool DOT, bool GROW>
__global__ void __launch_bounds__(kRefThreads, 2) refine_kernel(const RefineParams p) {
  // query rows as fp32, split so that a lane's 8 values are two conflict-free 16-byte reads:
  // element 8g+t lives in lo4[g] (t < 4) or hi4[g] (t >= 4)
  extern __shared__ __align__(16) float4 s_q[];          // [kRQ][2][D/8]
  __shared__ float s_part[kRQ][kRefThreads / 32];
  __shared__ float s_qn2[kRQ];
  const int G8 = p.D >> 3;
  const long long m0 = (long long)blockIdx.x * kRQ;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t pol_keep = l2_policy_keep(), pol_stream = l2_policy_stream();
  float qacc[kRQ];                                       // DOT: this lane's share of |q|^2 per staged row
#pragma unroll
  for (int t = 0; t < kRQ; ++t) qacc[t] = 0.f;
  for (int e0 = 0; e0 < kRQ * G8; e0 += kRefThreads) {
    const int e = e0 + tid;
    const bool on = e < kRQ * G8;
    if (!on) break;
    const int rr = on ? e / G8 : 0, g = e - rr * G8;
    const long long r = m0 + rr;
    float f[8];
    if (!on || r >= p.Mq) {
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = 0.f;
    } else if (p.Zq) {
      const float4* z = reinterpret_cast<const float4*>(p.Zq + r * p.D) + 2 * g;
      const float4 a = ld_hint(z, pol_stream), b = ld_hint(z + 1, pol_stream);
      f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
    } else {
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.Qhi) + r * p.D) + g), f);
      if (p.Qlo) {
        float l[8];
        unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.Qlo) + r * p.D) + g), l);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] += l[i];
      }
    }
    if (on) {
      s_q[(rr * 2 + 0) * G8 + g] = make_float4(f[0], f[1], f[2], f[3]);
      s_q[(rr * 2 + 1) * G8 + g] = make_float4(f[4], f[5], f[6], f[7]);
    }
    if (DOT) {
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < 8; ++t) s = fmaf(f[t], f[t], s);
#pragma unroll
      for (int t = 0; t < kRQ; ++t) qacc[t] += (t == rr) ? s : 0.f;
    }
  }
  if (DOT) {
    // fixed summation order (lane tree, then warps 0..15): results are bit-reproducible
#pragma unroll
    for (int t = 0; t < kRQ; ++t) {
      const float v = warp_sum(qacc[t]);
      if (lane == 0) s_part[t][warp] = v;
    }
    __syncthreads();
    if (tid < kRQ) {
      float v = 0.f;
      for (int w = 0; w < kRefThreads / 32; ++w) v += s_part[tid][w];
      s_qn2[tid] = v;
    }
  }
  __syncthreads();

  const int rr = warp / kWPR, par = warp % kWPR;
  const long long r = m0 + rr;
  if (r >= p.Mq) return;
  const int qi = (int)(r / p.Pq);
  const long long R = p.r0 + r;                            // GROW: row of the whole category
  const int i = GROW ? (int)(R / p.P) : (p.sym ? p.q_img0 + qi : (p.q_self ? __ldg(p.q_self + qi) : -1));
  const float4* qlo4 = s_q + (rr * 2 + 0) * G8;
  const float4* qhi4 = s_q + (rr * 2 + 1) * G8;
  const int j0 = (GROW ? p.jbase : 0) + blockIdx.y * p.Jb, j1 = min(p.nb_img, j0 + p.Jb);
  // categories: only the images of the query image's own category are its bank (the rest is never read by the reduction)
  int g0 = 0, gn = p.nb_img;
  if (p.sym && p.groups) { g0 = __ldg(p.groups + 2 * i); gn = __ldg(p.groups + 2 * i + 1); }
  for (int j = j0 + par; j < j1; j += kWPR) {
    bool col;          // arg-min from the column minima (the partner image owns the pair)
    long long e;
    if (GROW) {
      // only the pairs the growth launch computed: never two old images
      if (j == i || (i < p.n_old && j < p.n_old)) continue;
      col = !pair_owned_grow(p.n_old, i, j, p.nb_img);
      e = col ? (long long)(j - p.n_old) * ((long long)p.nb_img * p.P) + R : (long long)j * p.Mn + (R - (long long)p.n_old * p.P);
    } else {
      if (j < g0 || j >= g0 + gn) continue;
      if (j == i) {
        if (lane == 0) p.dex[(long long)j * p.Mq + r] = 0.f;     // own image: excluded by the reduction
        continue;
      }
      col = p.sym && !pair_owned(i - g0, j - g0, gn);
      e = (long long)j * p.Mq + r;
    }
    int c = 0;
    if (lane == 0) {
      if (col) c = (int)(unsigned int)(__ldg(p.colkey + e) & 0xffffffffull);
      else c = __ldg(p.rowarg + e);
      c = min(max(c, 0), p.P - 1);
    }
    c = __shfl_sync(0xffffffffu, c, 0);
    const uint4* bh = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.Bhi) + ((long long)j * p.P + c) * p.D);
    const uint4* bl = LO ? reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.Blo) + ((long long)j * p.P + c) * p.D) : nullptr;
    float s = warp_sum(row_dist2<T, NIT, LO, DOT>(bh, bl, qlo4, qhi4, G8, lane, pol_keep));
    if (DOT) s = fmaxf(fmaf(-2.f, s, s_qn2[rr] + __ldg(p.Bn2 + (long long)j * p.P + c)), 0.f);
    if (lane == 0) (GROW && col ? p.dcol : p.dex)[e] = sqrtf(s);
  }
}

template <typename T, int NIT, bool LO, bool DOT, bool GROW>
static int launch_refine(const RefineParams& p, dim3 grid, size_t smem, cudaStream_t st) {
  AC_CUDA(cudaFuncSetAttribute(refine_kernel<T, NIT, LO, DOT, GROW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  refine_kernel<T, NIT, LO, DOT, GROW><<<grid, kRefThreads, smem, st>>>(p);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

template <typename T, bool GROW>
static int dispatch_refine(const RefineParams& p, dim3 grid, size_t smem, cudaStream_t st) {
  if (p.Blo) return launch_refine<T, 0, true, false, GROW>(p, grid, smem, st);      // bank given as hi + lo: generic loop
  if (p.Bn2) {                                                                        // |q|^2 + |b|^2 - 2 q.b
    if (p.D == 4096) return launch_refine<T, 16, false, true, GROW>(p, grid, smem, st);
    if (p.D == 1024) return launch_refine<T, 4, false, true, GROW>(p, grid, smem, st);
    return launch_refine<T, 0, false, true, GROW>(p, grid, smem, st);
  }
  if (p.D == 4096) return launch_refine<T, 16, false, false, GROW>(p, grid, smem, st);
  return launch_refine<T, 0, false, false, GROW>(p, grid, smem, st);
}

// grid = (query chunks of kRQ rows, groups of p.Jb of the n_part partner images); p.Jb is set here
template <bool GROW>
static int run_refine(RefineParams& p, int op_dtype, int n_part, cudaStream_t st) {
  const size_t smem = (size_t)kRQ * p.D * sizeof(float);
  // bank images per group: their operand rows (kRefineL2MB, measured best on B200) stay L2-resident while every query chunk passes
  const double img_bytes = (double)p.P * p.D * 2.0 * (p.Blo ? 2 : 1);
  p.Jb = (int)std::max((double)kWPR, std::min(256.0, kRefineL2MB * 1.0e6 / img_bytes));
  p.Jb -= p.Jb % kWPR;                                             // the kWPR warps of a row take every kWPR-th image
  const long long chunks = (p.Mq + kRQ - 1) / kRQ;
  const int nbg = (n_part + p.Jb - 1) / p.Jb;
  if (chunks > 0x7fffffffLL || nbg > 65535) return AC_ERR_UNSUPPORTED;
  if (chunks == 0 || nbg == 0) return AC_OK;
  dim3 grid((unsigned)chunks, (unsigned)nbg);
  return op_dtype == AC_DT_F16 ? dispatch_refine<__half, GROW>(p, grid, smem, st) : dispatch_refine<__nv_bfloat16, GROW>(p, grid, smem, st);
}

}  // namespace ac

using namespace ac;

extern "C" int ac_refine_min_dist(const float* Zq, const void* Qhi, const void* Qlo, int64_t Mq, const void* Bhi, const void* Blo,
                                  int op_dtype, int nb_img, int P, int D, const int32_t* rowarg, const uint64_t* colkey, int sym,
                                  int q_img0, const int32_t* q_self, int Pq, const int32_t* groups, const float* Bn2, float* dmin,
                                  ac_stream_t stream) {
  if ((!Zq && !Qhi) || !Bhi || !rowarg || !dmin || Mq < 0 || nb_img < 1 || P < 1 || D < 1 || Pq < 1 || q_img0 < 0) return AC_ERR_INVALID;
  if (op_dtype != AC_DT_F16 && op_dtype != AC_DT_BF16) return AC_ERR_INVALID;
  if (sym && (!colkey || Pq != P)) return AC_ERR_INVALID;
  if (D % 8 != 0) return AC_ERR_UNSUPPORTED;                       // 16-byte operand vectors
  for (const void* v : {(const void*)Zq, Qhi, Qlo, Bhi, Blo})      // ... read from 16-byte aligned rows
    if (reinterpret_cast<uintptr_t>(v) % 16 != 0) return AC_ERR_INVALID;
  const size_t smem = (size_t)kRQ * D * sizeof(float);
  if (smem > 200 * 1024) return AC_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc) return rc;
  if (Mq == 0) return AC_OK;
  RefineParams p = {};
  p.Zq = Zq; p.Qhi = Qhi; p.Qlo = Qlo; p.Bhi = Bhi; p.Blo = Blo;
  p.Mq = Mq; p.nb_img = nb_img; p.P = P; p.D = D; p.Pq = Pq;
  p.rowarg = rowarg; p.colkey = (const unsigned long long*)colkey; p.sym = sym; p.q_img0 = q_img0; p.q_self = q_self; p.dex = dmin;
  p.groups = sym ? groups : nullptr;
  p.Bn2 = Bn2;
  return run_refine<false>(p, op_dtype, nb_img, (cudaStream_t)stream);
}

extern "C" int ac_refine_min_dist_grow(const float* Z, const void* Bhi, const void* Blo, int op_dtype, int n_old, int nb_img, int P,
                                       int D, const int32_t* rowarg, const uint64_t* colkey, const float* Bn2, float* drow, float* dcol,
                                       ac_stream_t stream) {
  if (!Z || !Bhi || !rowarg || !colkey || !drow || !dcol || n_old < 0 || nb_img <= n_old || P < 1 || D < 1) return AC_ERR_INVALID;
  if (op_dtype != AC_DT_F16 && op_dtype != AC_DT_BF16) return AC_ERR_INVALID;
  if (D % 8 != 0) return AC_ERR_UNSUPPORTED;
  for (const void* v : {(const void*)Z, Bhi, Blo})
    if (reinterpret_cast<uintptr_t>(v) % 16 != 0) return AC_ERR_INVALID;
  if ((size_t)kRQ * D * sizeof(float) > 200 * 1024) return AC_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  RefineParams p = {};
  p.Bhi = Bhi; p.Blo = Blo; p.Bn2 = Bn2;
  p.nb_img = nb_img; p.P = P; p.D = D; p.Pq = P;
  p.rowarg = rowarg; p.colkey = (const unsigned long long*)colkey; p.sym = 1; p.dex = drow; p.dcol = dcol;
  p.n_old = n_old;
  p.Mn = (long long)(nb_img - n_old) * P;
  // the new rows against every other image ...
  p.r0 = (long long)n_old * P; p.Zq = Z + p.r0 * D; p.Mq = p.Mn; p.jbase = 0;
  if ((rc = run_refine<true>(p, op_dtype, nb_img, st))) return rc;
  // ... and the old rows against the new images only: the cost follows the number of new pairs
  p.r0 = 0; p.Zq = Z; p.Mq = (long long)n_old * P; p.jbase = n_old;
  return run_refine<true>(p, op_dtype, nb_img - n_old, st);
}
