// Stage 2 tail + stage 3: per-image-min reduction -> w, tau-softmax alpha, weighted embedding X,
// image-to-image Euclidean matrix.  All HBM-bound and tiny next to the distance GEMM.
//
// Reference lines replaced:
//   ac_reduce_weights  models/patchcore/utils.py:227 (mean over j != i) / :236 (min over j; MIN_UPDATE lowers a running min)
//   ac_alpha           models/patchcore/utils.py:246-255, 266-275
//   ac_weighted_embed  examples/main.py:294-296
//   ac_pairwise_l2     examples/test.py:193-195 (Ward's internal pdist)
#include "common.cuh"
#include <math.h>
#include <vector>

namespace ac {

thread_local int g_last_cuda_error = 0;
unsigned long long g_kernel_launches = 0;

int check_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e);
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e);
  return major == 10 ? AC_OK : AC_ERR_DEVICE;
}

// one thread per query row; dmin is [nb_img, Mq] so consecutive threads read consecutive addresses
__global__ void __launch_bounds__(256) reduce_weights_kernel(const float* __restrict__ dmin, long long Mq, int nb_img, int Pq,
                                                             const int* __restrict__ q_self, const int* __restrict__ groups, int mode,
                                                             float* __restrict__ w) {
  const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (r >= Mq) return;
  const int self = q_self ? q_self[r / Pq] : -1;
  // categories (groups != null, needs q_self): the bank of a query image is its own category only
  int j0 = 0, j1 = nb_img;
  if (groups && self >= 0) { j0 = groups[2 * self]; j1 = j0 + groups[2 * self + 1]; }
  if (mode == AC_REDUCE_MEAN) {
    float s = 0.f;
    int cnt = 0;
    for (int j = j0; j < j1; ++j) {
      if (j == self) continue;
      s += __ldg(dmin + (long long)j * Mq + r);  // same left-to-right order as torch.mean over the cat'ed columns
      ++cnt;
    }
    w[r] = cnt > 0 ? s / (float)cnt : nanf("");
  } else {
    // AC_REDUCE_MIN_UPDATE lowers the running minimum w holds; a min of fp32 values does not depend on the order it is taken in
    float m = mode == AC_REDUCE_MIN_UPDATE ? w[r] : INFINITY;
    for (int j = j0; j < j1; ++j) {
      if (j == self) continue;
      m = fminf(m, __ldg(dmin + (long long)j * Mq + r));
    }
    w[r] = m;
  }
}

// one CTA per image, all taus in one pass; float64 like the reference
struct TauTable { double v[64]; };

__global__ void __launch_bounds__(256) alpha_kernel(const float* __restrict__ w, int N, int P, TauTable taus, int T,
                                                    double* __restrict__ a64, float* __restrict__ a32) {
  const int i = blockIdx.x;
  const float* wi = w + (long long)i * P;
  __shared__ double red[8];
  __shared__ double s_bcast;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;

  // row max (shared by every tau)
  float m = -INFINITY;
  for (int p = threadIdx.x; p < P; p += blockDim.x) m = fmaxf(m, wi[p]);
  m = warp_max(m);
  if (lane == 0) red[warp] = (double)m;
  __syncthreads();
  if (threadIdx.x == 0) {
    double mm = red[0];
    for (int k = 1; k < nw; ++k) mm = fmax(mm, red[k]);
    s_bcast = mm;
  }
  __syncthreads();
  const double wmax = s_bcast;

  for (int t = 0; t < T; ++t) {
    const double tau = taus.v[t];
    const bool onehot = (tau == 0.0);  // math.isclose(tau, 0) with the default rel_tol is true only for tau == 0
    const double inv = onehot ? 0.0 : 1.0 / tau;
    double s = 0.0;
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
      const double x = (double)wi[p];
      s += onehot ? (x == wmax ? 1.0 : 0.0) : exp(inv * (x - wmax));
    }
    s = warp_sum(s);
    __syncthreads();
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double tot = 0;
      for (int k = 0; k < nw; ++k) tot += red[k];
      s_bcast = tot;
    }
    __syncthreads();
    const double tot = s_bcast;
    const long long base = ((long long)t * N + i) * P;
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
      const double x = (double)wi[p];
      const double e = onehot ? (x == wmax ? 1.0 : 0.0) : exp(inv * (x - wmax));
      const double a = e / tot;
      if (a64) a64[base + p] = a;
      if (a32) a32[base + p] = (float)a;
    }
    __syncthreads();
  }
}

// X[i, d] = sum_p alpha[i,p] * Z[i,p,d]; grid (ceil(D / (128*4)), N); each thread owns 4 columns.
// vec (decided on the host): D % 4 == 0 and Z, X 16-byte aligned -- float4 loads and stores; else the scalar loop, which
// sums in the same order (bit-identical results).
__global__ void __launch_bounds__(128) weighted_embed_kernel(const float* __restrict__ alpha, const float* __restrict__ Z, int N, int P,
                                                             int D, float* __restrict__ X, bool vec) {
  extern __shared__ float s_alpha[];
  const int i = blockIdx.y;
  for (int p = threadIdx.x; p < P; p += blockDim.x) s_alpha[p] = alpha[(long long)i * P + p];
  __syncthreads();
  const int d0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (d0 >= D) return;
  const float* zi = Z + (long long)i * P * D;
  if (vec) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int p = 0; p < P; ++p) {
      const float a = s_alpha[p];
      const float4 z = __ldg(reinterpret_cast<const float4*>(zi + (long long)p * D + d0));
      acc.x = fmaf(a, z.x, acc.x);
      acc.y = fmaf(a, z.y, acc.y);
      acc.z = fmaf(a, z.z, acc.z);
      acc.w = fmaf(a, z.w, acc.w);
    }
    *reinterpret_cast<float4*>(X + (long long)i * D + d0) = acc;
  } else {
    for (int d = d0; d < min(D, d0 + 4); ++d) {
      float acc = 0.f;
      for (int p = 0; p < P; ++p) acc = fmaf(s_alpha[p], __ldg(zi + (long long)p * D + d), acc);
      X[(long long)i * D + d] = acc;
    }
  }
}

// The same for T temperatures from ONE pass over Z (a tau sweep re-read the whole Z once per tau: 6 x 0.57 ms at config 5, 17 x
// 0.19 ms for the reference's tau list at config 2): X[t,i,d] = sum_p alpha[t,i,p] * Z[i,p,d], T <= 8 accumulators per thread,
// the same summation order per tau as weighted_embed_kernel (bit-identical results).
template <int T>
__global__ void __launch_bounds__(128) weighted_embed_multi_kernel(const float* __restrict__ alpha, const float* __restrict__ Z, int N,
                                                                   int P, int D, float* __restrict__ X) {
  extern __shared__ float s_alpha[];    // [T][P]
  const int i = blockIdx.y;
  for (int e = threadIdx.x; e < T * P; e += blockDim.x) {
    const int t = e / P, p = e - t * P;
    s_alpha[e] = alpha[((long long)t * N + i) * P + p];
  }
  __syncthreads();
  const int d0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (d0 >= D) return;
  const float* zi = Z + (long long)i * P * D;
  float4 acc[T];
#pragma unroll
  for (int t = 0; t < T; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
  for (int p = 0; p < P; ++p) {
    const float4 z = __ldg(reinterpret_cast<const float4*>(zi + (long long)p * D + d0));
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float a = s_alpha[t * P + p];
      acc[t].x = fmaf(a, z.x, acc[t].x);
      acc[t].y = fmaf(a, z.y, acc[t].y);
      acc[t].z = fmaf(a, z.z, acc[t].z);
      acc[t].w = fmaf(a, z.w, acc[t].w);
    }
  }
#pragma unroll
  for (int t = 0; t < T; ++t) *reinterpret_cast<float4*>(X + ((long long)t * N + i) * D + d0) = acc[t];
}

// Dmat[i,j] = sqrt(sum_d (X[i,d]-X[j,d])^2): 32x32 output tile per CTA, 2x2 per thread... kept simple:
// 16x16 threads, each computes a 2x2 micro-tile, D walked in chunks of 32 through shared memory.
__global__ void __launch_bounds__(256) pairwise_l2_kernel(const float* __restrict__ X, int N, int D, float* __restrict__ Dm) {
  __shared__ float sa[32][33], sb[32][33];
  const int bi = blockIdx.y * 32, bj = blockIdx.x * 32;
  if (bj < bi) return;  // upper triangle only; mirrored on store
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  for (int d0 = 0; d0 < D; d0 += 32) {
    for (int e = threadIdx.x; e < 32 * 32; e += 256) {
      const int r = e >> 5, c = e & 31;
      const int d = d0 + c;
      sa[r][c] = (bi + r < N && d < D) ? __ldg(X + (long long)(bi + r) * D + d) : 0.f;
      sb[r][c] = (bj + r < N && d < D) ? __ldg(X + (long long)(bj + r) * D + d) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < 32; ++c) {
      const float a0 = sa[ty][c], a1 = sa[ty + 16][c];
      const float b0 = sb[tx][c], b1 = sb[tx + 16][c];
      float t;
      t = a0 - b0; acc[0][0] = fmaf(t, t, acc[0][0]);
      t = a0 - b1; acc[0][1] = fmaf(t, t, acc[0][1]);
      t = a1 - b0; acc[1][0] = fmaf(t, t, acc[1][0]);
      t = a1 - b1; acc[1][1] = fmaf(t, t, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int i = bi + ty + 16 * u, j = bj + tx + 16 * v;
      if (i < N && j < N) {
        const float d = (i == j) ? 0.f : sqrtf(acc[u][v]);
        if (j >= i) {
          Dm[(long long)i * N + j] = d;
          Dm[(long long)j * N + i] = d;
        }
      }
    }
}

// small N (one category: N ~ 100): one warp per (i, j >= i) pair, X stays L2-resident; the tiled
// kernel above would run only ~N^2/2048 CTAs.  vec (decided on the host: X 16-byte aligned) picks float4 loads; without it
// the same four elements are loaded one by one and summed in the same order (bit-identical results).
__device__ __forceinline__ float4 ld4(const float* p, bool vec) {
  if (vec) return __ldg(reinterpret_cast<const float4*>(p));
  return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}

__global__ void __launch_bounds__(256) pairwise_l2_warp_kernel(const float* __restrict__ X, int N, int D, float* __restrict__ Dm,
                                                               bool vec) {
  const long long w = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= (long long)N * N) return;
  const int i = (int)(w / N), j = (int)(w - (long long)i * N);
  if (j < i) return;
  const int lane = threadIdx.x & 31;
  const float* xi = X + (long long)i * D;
  const float* xj = X + (long long)j * D;
  float acc = 0.f;
  if ((D & 3) == 0) {
    for (int d = lane * 4; d < D; d += 128) {
      const float4 a = ld4(xi + d, vec);
      const float4 b = ld4(xj + d, vec);
      float t;
      t = a.x - b.x; acc = fmaf(t, t, acc);
      t = a.y - b.y; acc = fmaf(t, t, acc);
      t = a.z - b.z; acc = fmaf(t, t, acc);
      t = a.w - b.w; acc = fmaf(t, t, acc);
    }
  } else {
    for (int d = lane; d < D; d += 32) {
      const float t = __ldg(xi + d) - __ldg(xj + d);
      acc = fmaf(t, t, acc);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    const float dd = (i == j) ? 0.f : sqrtf(acc);
    Dm[(long long)i * N + j] = dd;
    Dm[(long long)j * N + i] = dd;
  }
}

}  // namespace ac

using namespace ac;

extern "C" int ac_version(void) { return 100; }

extern "C" const char* ac_strerror(int code) {
  switch (code) {
    case AC_OK: return "ok";
    case AC_ERR_INVALID: return "invalid argument";
    case AC_ERR_UNSUPPORTED: return "unsupported shape for this kernel";
    case AC_ERR_DEVICE: return "device is not sm_100 (B200); libac_b200 has no other code path";
    case AC_ERR_CUDA: return "CUDA call failed (see ac_last_cuda_error)";
    case AC_ERR_WORKSPACE: return "workspace too small";
    default: return "unknown error";
  }
}

extern "C" int ac_last_cuda_error(void) { return g_last_cuda_error; }

// test / bench hook (not in the public header): kernels launched by the library so far
extern "C" unsigned long long ac_debug_launches(void) { return __atomic_load_n(&g_kernel_launches, __ATOMIC_RELAXED); }

extern "C" int ac_device_ok(int dev) {
  int major = 0;
  cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e);
  return major == 10 ? AC_OK : AC_ERR_DEVICE;
}

extern "C" int ac_reduce_weights_ex(const float* dmin, int64_t Mq, int nb_img, int Pq, const int32_t* q_self, const int32_t* groups,
                                    int mode, float* w, ac_stream_t stream) {
  if (!dmin || !w || Mq < 0 || nb_img < 1 || Pq < 1) return AC_ERR_INVALID;
  if (mode != AC_REDUCE_MEAN && mode != AC_REDUCE_MIN && mode != AC_REDUCE_MIN_UPDATE) return AC_ERR_INVALID;
  if (groups && !q_self) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (Mq == 0) return AC_OK;
  reduce_weights_kernel<<<(unsigned)((Mq + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dmin, Mq, nb_img, Pq, q_self, groups, mode, w);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_reduce_weights(const float* dmin, int64_t Mq, int nb_img, int Pq, const int32_t* q_self, int mode, float* w,
                                 ac_stream_t stream) {
  return ac_reduce_weights_ex(dmin, Mq, nb_img, Pq, q_self, nullptr, mode, w, stream);
}

extern "C" int ac_alpha(const float* w, int N, int P, const double* taus_host, int T, double* alpha64, float* alpha32,
                        ac_stream_t stream) {
  if (!w || !taus_host || N < 0 || P < 1 || T < 1 || T > 64) return AC_ERR_INVALID;
  if (!alpha64 && !alpha32) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (N == 0) return AC_OK;
  TauTable tt;  // <= 64 taus travel by value as a kernel parameter: re-entrant, no allocation, no sync
  for (int t = 0; t < T; ++t) tt.v[t] = taus_host[t];
  for (int t = T; t < 64; ++t) tt.v[t] = 1.0;
  alpha_kernel<<<N, 256, 0, (cudaStream_t)stream>>>(w, N, P, tt, T, alpha64, alpha32);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_weighted_embed(const float* alpha, const float* Z, int N, int P, int D, float* X, ac_stream_t stream) {
  if (!alpha || !Z || !X || N < 0 || P < 1 || D < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (N == 0) return AC_OK;
  if ((size_t)P * sizeof(float) > 200 * 1024) return AC_ERR_UNSUPPORTED;
  auto kern = weighted_embed_kernel;
  const size_t smem = (size_t)P * sizeof(float);
  if (smem > 48 * 1024) AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // float4 path only when every vector access is 16-byte aligned (a contiguous view may start anywhere)
  const bool vec = (D % 4 == 0) && (reinterpret_cast<uintptr_t>(Z) % 16 == 0) && (reinterpret_cast<uintptr_t>(X) % 16 == 0);
  dim3 grid(ceil_div(D, 128 * 4), N);
  kern<<<grid, 128, smem, (cudaStream_t)stream>>>(alpha, Z, N, P, D, X, vec);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

template <int T>
static int launch_weighted_multi(const float* alpha, const float* Z, int N, int P, int D, float* X, cudaStream_t st) {
  auto kern = weighted_embed_multi_kernel<T>;
  const size_t smem = (size_t)T * P * sizeof(float);
  if (smem > 48 * 1024) AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(ceil_div(D, 128 * 4), N);
  kern<<<grid, 128, smem, st>>>(alpha, Z, N, P, D, X);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_weighted_embed_multi(const float* alpha, const float* Z, int T, int N, int P, int D, float* X, ac_stream_t stream) {
  if (!alpha || !Z || !X || T < 1 || N < 0 || P < 1 || D < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (N == 0) return AC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // taus in groups of up to 8 (accumulators in registers); shapes the vector kernel does not take go through the single-tau one
  const bool vec = (D % 4 == 0) && (reinterpret_cast<uintptr_t>(Z) % 16 == 0) && (reinterpret_cast<uintptr_t>(X) % 16 == 0);
  for (int t0 = 0; t0 < T;) {
    int g = std::min(8, T - t0);
    while (g > 1 && (size_t)g * P * sizeof(float) > 200 * 1024) --g;
    const float* a = alpha + (long long)t0 * N * P;
    float* x = X + (long long)t0 * N * D;
    if (!vec || g == 1) {
      g = 1;
      rc = ac_weighted_embed(a, Z, N, P, D, x, stream);
    } else {
      // groups are launched with a compile-time size; a tail of 3 runs as 2 + 1
      int gg = g >= 8 ? 8 : g >= 4 ? 4 : g >= 2 ? 2 : 1;
      g = gg;
      rc = gg == 8 ? launch_weighted_multi<8>(a, Z, N, P, D, x, st) : gg == 4 ? launch_weighted_multi<4>(a, Z, N, P, D, x, st)
                                                                              : launch_weighted_multi<2>(a, Z, N, P, D, x, st);
    }
    if (rc) return rc;
    t0 += g;
  }
  return AC_OK;
}

extern "C" int ac_pairwise_l2(const float* X, int N, int D, float* Dmat, ac_stream_t stream) {
  if (!X || !Dmat || N < 0 || D < 1) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (N == 0) return AC_OK;
  if (N <= 384) {
    const long long warps = (long long)N * N;
    const bool vec = reinterpret_cast<uintptr_t>(X) % 16 == 0;   // float4 loads (rows are 16-byte aligned when D % 4 == 0)
    pairwise_l2_warp_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(X, N, D, Dmat, vec);
  } else {
    dim3 grid(ceil_div(N, 32), ceil_div(N, 32));
    pairwise_l2_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X, N, D, Dmat);
  }
  AC_LAUNCH_CHECK();
  return AC_OK;
}

// ------------------------------------------------------------------------------------------------
// Batched strided 2-D copy (multi-GPU plumbing, no counterpart in the reference): up to 16 blocks of `rows` x `row_bytes` with
// their own row strides in ONE launch.  The sharded path reads the column-minimum blocks of its query rows out of every
// peer's symmetric-memory buffer with it (the sources are NVLink peer mappings; eight separate copy launches cost 64 us of
// a 2.7 ms step at 8 GPUs).
namespace ac {
static constexpr int kMaxCopyBlocks = 16;
struct CopyBlocks {
  const char* src[kMaxCopyBlocks];
  char* dst[kMaxCopyBlocks];
  long long sstride[kMaxCopyBlocks], dstride[kMaxCopyBlocks], row_bytes[kMaxCopyBlocks];
  int rows[kMaxCopyBlocks];
};
template <typename V>
__global__ void __launch_bounds__(256) copy_blocks_kernel(const CopyBlocks p) {
  const int b = blockIdx.y;
  const long long per_row = p.row_bytes[b] / (long long)sizeof(V), total = per_row * p.rows[b];
  const char* __restrict__ src = p.src[b];
  char* __restrict__ dst = p.dst[b];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / per_row, c = i - r * per_row;
    *reinterpret_cast<V*>(dst + r * p.dstride[b] + c * (long long)sizeof(V)) =
        *reinterpret_cast<const V*>(src + r * p.sstride[b] + c * (long long)sizeof(V));
  }
}
}  // namespace ac

extern "C" int ac_copy_blocks(int n, const void* const* src_host, const int64_t* src_stride_bytes_host, void* const* dst_host,
                              const int64_t* dst_stride_bytes_host, const int32_t* rows_host, const int64_t* row_bytes_host,
                              ac_stream_t stream) {
  if (n < 0 || n > ac::kMaxCopyBlocks) return AC_ERR_UNSUPPORTED;
  if (n == 0) return AC_OK;
  if (!src_host || !dst_host || !src_stride_bytes_host || !dst_stride_bytes_host || !rows_host || !row_bytes_host) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  ac::CopyBlocks p;
  memset(&p, 0, sizeof(p));
  bool v16 = true;
  long long most = 0;
  for (int b = 0; b < n; ++b) {
    if (!src_host[b] || !dst_host[b] || rows_host[b] < 0 || row_bytes_host[b] < 0 || row_bytes_host[b] % 4 != 0) return AC_ERR_INVALID;
    p.src[b] = (const char*)src_host[b];
    p.dst[b] = (char*)dst_host[b];
    p.sstride[b] = src_stride_bytes_host[b];
    p.dstride[b] = dst_stride_bytes_host[b];
    p.rows[b] = rows_host[b];
    p.row_bytes[b] = row_bytes_host[b];
    v16 = v16 && ((reinterpret_cast<uintptr_t>(src_host[b]) | reinterpret_cast<uintptr_t>(dst_host[b]) | (uintptr_t)p.sstride[b] |
                   (uintptr_t)p.dstride[b] | (uintptr_t)p.row_bytes[b]) % 16 == 0);
    most = std::max(most, (long long)rows_host[b] * row_bytes_host[b]);
  }
  if (most == 0) return AC_OK;
  const long long elems = most / (v16 ? 16 : 4);
  dim3 grid((unsigned)std::min<long long>((elems + 255) / 256, 148LL * 2), (unsigned)n);
  if (v16) ac::copy_blocks_kernel<uint4><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  else ac::copy_blocks_kernel<unsigned int><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  AC_LAUNCH_CHECK();
  return AC_OK;
}
