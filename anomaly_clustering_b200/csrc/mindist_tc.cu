// Stage 2: patch-versus-bank nearest neighbour on the 5th-gen tensor cores (tcgen05 / TMEM / TMA).
//
// Replaces the torch.cdist + torch.min(dim=1) loops of Weight_Distance_Unsupervised / _Supervised
// (reference: Anomaly-Clustering/models/patchcore/utils.py:222-237).
//
//   dmin[j, r] = sqrt(max(0, |q_r|^2 + min_{c in image j} (|b_c|^2 - 2 q_r . b_c)))
//
// Structure (one persistent CTA pair per two SMs, cta_group::2 MMAs):
//   warp 0      TMA producer: 128B-swizzled K-major operand tiles -> kStages-deep smem ring; in the leader CTA it
//               also CLAIMS the work units (global atomic counter) and publishes them to the other roles through
//               a small smem queue (the peer CTA's copy is written with st.shared::cluster)
//   warp 1      MMA issuer:   tcgen05.mma kind::f16, fp32 accumulators in TMEM (2 x 256 columns,
//               double buffered so the epilogue of tile i overlaps the MMAs of tile i+1)
//   warps 2-5   epilogue: tcgen05.ld 32 lanes x 32 columns, d2 = bn2[c] - 2*acc, running row-min in
//               registers across the tiles of one bank image (each thread owns one query row, so
//               the row-min needs no shuffles), one coalesced store per (row, bank image).
//   The [Mq, Nb*P] distance matrix never exists in memory.
// Work unit = (block of 2*kTileM = 256 query rows, one kTileM half per CTA of the pair, bank image).  A bank image is cut into nt tiles
// of <= 256 rows whose widths are multiples of 16 (P=784 -> 208+208+208+160), so no tile straddles
// two images; excess columns of the last tile are masked with +inf norms.
// Units are rasterised so that concurrently resident units share A blocks and bank images in L2.
// The X3 precision modes run 3 K-segments (hi*hi, lo*hi, hi*lo) into the same accumulator.
// Symmetric mode (ac_min_dist_sym): only the units of image pairs the query image OWNS are enumerated (device-built
// raster list); the epilogue additionally reduces every column over the 32 rows of its warp (butterfly
// transpose-min) and atomicMin's the result, so cdist(Zi,Zj) and cdist(Zj,Zi) come from one tile.
#include "common.cuh"
#include <cuda.h>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>

namespace ac {

static constexpr int kTcThreads = 192;
static constexpr int kBlockK = 64;         // elements per K block = one 128-byte swizzle row (2-byte operands)
static constexpr int kUmmaK = 16;
static constexpr int kTileM = 128;         // rows per CTA; a CTA pair multiplies 2 * kTileM query rows
static constexpr int kMaxN = 256;
static constexpr int kBRows = kMaxN / 2;   // bank rows staged per CTA per stage (each CTA holds half of the N tile)
static constexpr int kStages = 6;
static constexpr int kGM = 16;             // query blocks per raster group: 16 x 2 MB of A + the streaming bank images stay L2-resident (tuned on B200)
static constexpr int kTmemCols = 512;
static constexpr long long kWatchdogCycles = 20000000000LL;  // ~10 s

struct __align__(64) TcParams {
  CUtensorMap mapA[2];       // [0] hi, [1] lo
  CUtensorMap mapBmain[2];
  CUtensorMap mapBlast[2];
  const float* qn2;
  const float* bn2;
  float* dmin;
  int* err;
  long long Mq;
  long long total_units;
  int nb_img, P, D;
  int nkb;                   // K blocks per segment
  int nseg;                  // 1 or 3
  int nt, wmain, wlast;      // tiles per bank image, widths (multiples of 16)
  int n_mblocks;
  uint32_t idesc_main, idesc_last;
  // symmetric (self-bank) mode: every unordered image pair is multiplied once
  int sym;                   // 0 = every (query block, bank image) unit; 1 = only pairs owned by the query image
  int q_img0;                // global image index of query row 0 (query slice of a sharded run)
  int KU;                    // units per query block in sym mode
  unsigned int* colmin;      // [nq_img, nb_img*P] squared distances (fp32 bits), atomicMin target
  const int2* units;         // sym mode: explicit (query block, bank image) list in raster order (device-built)
  const long long* n_units;  // sym mode: length of that list (device memory)
  int win_begin, win_count;  // sym mode: only bank images in the circular window [win_begin, win_begin + win_count)
  unsigned long long* counter;   // next unclaimed unit (work stealing)
  // arg-min tracking (kArg kernels; the exact re-evaluation of ac_refine_min_dist needs WHICH bank row won)
  // per-category banks in one launch (the reference runs one make_category_data per category, examples/main.py:353):
  // groups[2*j], groups[2*j+1] = first image and image count of the category of bank image j; pairs exist only inside
  // a category and ownership is the circular rule inside it.  null = one category (all images).
  const int* groups;
  // sharded runs: bank_ready[j] != 0 once bank image j (operand rows + norms) has landed in this GPU's memory; the producer
  // waits for it before the first load of a unit.  null = the whole bank is resident.
  const int* bank_ready;
  int img_rot;                   // all-pairs form: the raster starts at this bank image (the first one that is resident in a sharded run)
  int* rowarg;                   // [nb_img, Mq] row inside bank image j that is nearest to query row r
  unsigned long long* colkey;    // sym: [nq_img, nb_img*P] (fp32 bits of d2 << 32) | row inside the query image, atomicMin target
};

// Ownership of the unordered pair {i, j} of N images: the image that sees the other one within the
// next floor((N-1)/2) positions of the circular order (ties at N/2 go to the smaller index).
__host__ __device__ inline bool pair_owned(int i, int j, int N) {
  int d = j - i;
  if (d < 0) d += N;
  if (d == 0) return false;
  if (2 * d < N) return true;
  if (2 * d == N) return i < j;
  return false;
}

// ownership with categories: image i owns the pair {i, j} iff both lie in the category of j and i owns it there
__host__ __device__ inline bool pair_owned_grouped(const int* groups, int i, int j, int N) {
  if (!groups) return pair_owned(i, j, N);
#ifdef __CUDA_ARCH__
  const int g0 = __ldg(groups + 2 * j), gn = __ldg(groups + 2 * j + 1);
#else
  const int g0 = groups[2 * j], gn = groups[2 * j + 1];
#endif
  if (i < g0 || i >= g0 + gn) return false;
  return pair_owned(i - g0, j - g0, gn);
}

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
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
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > kWatchdogCycles) {  // pipeline deadlock: report and kill the launch, never hang the GPU
      if (err) *reinterpret_cast<volatile int*>(err) = code;   // host-mapped flag: still readable after the trap (ac_last_watchdog)
      __threadfence_system();
      __trap();
    }
  }
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (clock64() - t0 > kWatchdogCycles) {
      if (err) *reinterpret_cast<volatile int*>(err) = code;
      __threadfence_system();
      __trap();
    }
  }
}
__device__ __forceinline__ void st_cluster_s64(uint32_t cluster_addr, long long v) {
  asm volatile("st.shared::cluster.b64 [%0], %1;" ::"r"(cluster_addr), "l"(v) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// data lands in this CTA's shared memory, completion bytes are signalled on the LEADER CTA's barrier
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// tcgen05.commit: the mbarrier receives one arrival once all previously issued MMAs have completed;
// multicast to the same barrier offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

#define AC_TMEM_LD16(taddr, v)                                                                                          \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];" \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),        \
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])   \
               : "r"(taddr))
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor: 8-row x 128-byte atoms, SBO = 1024 B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);   // start address, 16-byte units
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
  return d;
}

// unit index -> (query block, bank image); false when the unit carries no work (sym mode: no row of
// the block owns the pair).  Every warp role evaluates this identically, so skipped units touch no barrier.
// r[i] = this lane's value for column i (32 columns x 32 lanes).  Returns min over all lanes of
// column `lane`: at each butterfly level a lane keeps the half of the columns whose index bit matches
// its own lane bit and hands the other half to its partner.
__device__ __forceinline__ float warp_transpose_min(float (&r)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float keep = up ? r[i + off] : r[i];
      const float send = up ? r[i] : r[i + off];
      r[i] = fminf(keep, __shfl_xor_sync(0xffffffffu, send, off));
    }
  }
  return r[0];
}

// same butterfly on 64-bit keys (distance bits << 32 | row): the min carries the arg-min with it
__device__ __forceinline__ unsigned long long warp_transpose_min_u64(unsigned long long (&r)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const unsigned long long keep = up ? r[i + off] : r[i];
      const unsigned long long send = up ? r[i] : r[i + off];
      const unsigned long long got = __shfl_xor_sync(0xffffffffu, send, off);
      r[i] = keep < got ? keep : got;
    }
  }
  return r[0];
}

// sharded runs (TcParams::bank_ready): spin until bank image img has landed; a flag that never comes kills the launch (code 7)
__device__ __forceinline__ void wait_bank_ready(const TcParams& p, int img) {
  const int* fl = p.bank_ready + img;
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(fl) : "memory");
  if (v != 0) return;
  const long long t0 = clock64();
  do {
    __nanosleep(200);
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(fl) : "memory");
    if (v == 0 && clock64() - t0 > kWatchdogCycles) {
      if (p.err) *p.err = 7;
      __threadfence_system();
      __trap();
    }
  } while (v == 0);
}

__device__ __forceinline__ bool decode_unit(const TcParams& p, long long u, int& mb, int& img) {
  if (p.sym) {
    // compact host-built list (only units that carry work), so all CTA pairs stay in lock-step on the
    // same few bank images and query blocks -- skipped slots would let them drift apart and thrash L2
    const int2 un = __ldg(p.units + u);
    mb = un.x;
    img = un.y;
    return true;
  }
  const int per_mb = p.nb_img;
  const long long per_group = (long long)kGM * per_mb;
  const int mg = (int)(u / per_group);
  const long long rem = u - (long long)mg * per_group;
  const int gm_cur = min(kGM, p.n_mblocks - mg * kGM);
  const int k = (int)(rem / gm_cur);
  mb = mg * kGM + (int)(rem - (long long)k * gm_cur);
  img = k + p.img_rot;
  if (img >= p.nb_img) img -= p.nb_img;
  return true;
}

// ------------------------------------------------------------------------------------------------
template <bool kArg>
__global__ void __launch_bounds__(kTcThreads, 1) mindist_tc_kernel(const __grid_constant__ TcParams p) {
  constexpr uint32_t kABytes = kTileM * kBlockK * 2;        // 16 KB
  constexpr uint32_t kBBytes = kBRows * kBlockK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment is required by SWIZZLE_128B; the launch adds 1 KB of slack
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* s_bn2 = reinterpret_cast<float*>(smem + kStages * kStageBytes);            // [2][kMaxN]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_bn2 + 2 * kMaxN);
  uint64_t* full_bar = s_bar;                 // [kStages]
  uint64_t* empty_bar = s_bar + kStages;      // [kStages]
  uint64_t* tfull_bar = s_bar + 2 * kStages;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;       // [2]
  constexpr int kQD = 4;                                   // depth of the unit queue
  uint64_t* qfull_bar = tempty_bar + 2;                    // [kQD]
  uint64_t* qempty_bar = qfull_bar + kQD;                  // [kQD] (the leader CTA's copy collects both CTAs' readers)
  long long* s_qunit = reinterpret_cast<long long*>(qempty_bar + kQD);   // [kQD]
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_qunit + kQD);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = (rank == 0);
  const long long total_units = p.sym ? __ldg(p.n_units) : p.total_units;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tfull_bar[b]), 1);
      mbar_init(smem_u32(&tempty_bar[b]), 4 * 2);  // one arrival per epilogue warp of both CTAs of the pair
    }
    for (int i = 0; i < kQD; ++i) {
      mbar_init(smem_u32(&qfull_bar[i]), 1);
      mbar_init(smem_u32(&qempty_bar[i]), 5 * 2);  // readers: MMA warp (or the peer's producer) + 4 epilogue warps per CTA
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(s_tmem), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // ---- unit sequence: the leader's producer claims units from a global counter and publishes them through a kQD-deep
  // smem queue to every other role of the pair.
  const uint32_t qempty_leader0 = mapa_rank(smem_u32(&qempty_bar[0]), 0);
  auto queue_read = [&](uint32_t& qs, uint32_t& qph) -> long long {   // one lane per reader warp
    mbar_wait_cluster(smem_u32(&qfull_bar[qs]), qph, p.err, 5);
    const long long u = *reinterpret_cast<volatile long long*>(&s_qunit[qs]);
    mbar_arrive_cluster(qempty_leader0 + qs * 8);
    if (++qs == kQD) { qs = 0; qph ^= 1; }
    return u;
  };

  if (warp == 0) {
    // ================================================================ TMA producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      const uint32_t full0 = mapa_rank(smem_u32(&full_bar[0]), 0);
      uint32_t qs = 0, qph = 0;
      for (;;) {
        long long u;
        if (leader) {
          mbar_wait_cluster(smem_u32(&qempty_bar[qs]), qph ^ 1, p.err, 6);   // slot free in both CTAs
          const unsigned long long c = atomicAdd(p.counter, 1ull);
          u = (c < (unsigned long long)total_units) ? (long long)c : -1;
          s_qunit[qs] = u;
          asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&qfull_bar[qs])) : "memory");
          st_cluster_s64(mapa_rank(smem_u32(&s_qunit[qs]), 1), u);
          mbar_arrive_cluster(mapa_rank(smem_u32(&qfull_bar[qs]), 1));
          if (++qs == kQD) { qs = 0; qph ^= 1; }
        } else {
          u = queue_read(qs, qph);
        }
        if (u < 0) break;
        int mb, img;
        if (!decode_unit(p, u, mb, img)) continue;
        if (p.bank_ready) {
          // the shard that holds this bank image may still be travelling (copy-engine pull on another stream): wait for its flag,
          // then order the flag read before the TMA (async proxy) reads of the landed rows
          wait_bank_ready(p, img);
          asm volatile("fence.proxy.async;" ::: "memory");
        }
        const int arow = mb * (kTileM * 2) + (int)rank * kTileM;
        for (int t = 0; t < p.nt; ++t) {
          const bool last = (t == p.nt - 1);
          const int width = last ? p.wlast : p.wmain;
          const int brow = img * p.P + t * p.wmain + (int)rank * (width / 2);
          const uint32_t bbytes = (uint32_t)(width / 2) * kBlockK * 2;
          for (int seg = 0; seg < p.nseg; ++seg) {
            const CUtensorMap* ma = &p.mapA[seg == 1 ? 1 : 0];
            const CUtensorMap* mbp = last ? &p.mapBlast[seg == 2 ? 1 : 0] : &p.mapBmain[seg == 2 ? 1 : 0];
            for (int kb = 0; kb < p.nkb; ++kb) {
              mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1, p.err, 1);
              if (leader) mbar_expect_tx(smem_u32(&full_bar[stage]), (kABytes + bbytes) * 2);
              const uint32_t fb = full0 + stage * 8;
              uint8_t* sa = smem + stage * kStageBytes;
              tma_load_2d(smem_u32(sa), ma, fb, kb * kBlockK, arow);
              tma_load_2d(smem_u32(sa + kABytes), mbp, fb, kb * kBlockK, brow);
              if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (leader CTA only)
    if (leader && elect_one()) {
      uint32_t stage = 0, phase = 0;
      uint32_t tile_ctr = 0;
      uint32_t qs = 0, qph = 0;
      for (;;) {
        const long long u = queue_read(qs, qph);
        if (u < 0) break;
        int mb_, img_;
        if (!decode_unit(p, u, mb_, img_)) continue;
        for (int t = 0; t < p.nt; ++t, ++tile_ctr) {
          const uint32_t buf = tile_ctr & 1, tphase = (tile_ctr >> 1) & 1;
          const uint32_t idesc = (t == p.nt - 1) ? p.idesc_last : p.idesc_main;
          mbar_wait(smem_u32(&tempty_bar[buf]), tphase ^ 1, p.err, 2);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * kMaxN;
          const int nk_total = p.nseg * p.nkb;
          for (int kb = 0; kb < nk_total; ++kb) {
            mbar_wait(smem_u32(&full_bar[stage]), phase, p.err, 3);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + stage * kStageBytes);
            const uint64_t adesc = make_smem_desc(sa);
            const uint64_t bdesc = make_smem_desc(sa + kABytes);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              // advance 32 bytes (16 elements) along K inside the 128-byte swizzle row
              umma_f16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit(smem_u32(&empty_bar[stage]));     // frees the smem slot once these MMAs retire
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          umma_commit(smem_u32(&tfull_bar[buf]));         // accumulator complete -> epilogue
        }
      }
    }
  } else {
    // ================================================================ epilogue (warps 2..5)
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int et = q * 32 + lane;                 // row inside the CTA tile == TMEM lane
    const int eidx = threadIdx.x - 64;            // 0..127
    const uint32_t tempty0 = mapa_rank(smem_u32(&tempty_bar[0]), 0);
    uint32_t tile_ctr = 0;
    uint32_t qs = 0, qph = 0;
    for (;;) {
      long long uu = 0;
      if (lane == 0) uu = queue_read(qs, qph);
      else if (++qs == kQD) { qs = 0; qph ^= 1; }      // keep every lane's queue cursor in step
      const long long u = __shfl_sync(0xffffffffu, uu, 0);
      if (u < 0) break;
      int mb, img;
      if (!decode_unit(p, u, mb, img)) continue;
      if (p.bank_ready) {
        // the norms of this bank image are read below, ahead of the accumulator: they travel with the rows, wait for the flag too
        if (lane == 0) wait_bank_ready(p, img);
        __syncwarp();
      }
      const long long row = (long long)mb * (kTileM * 2) + rank * kTileM + et;
      const bool rvalid = row < p.Mq;
      // sym mode: this row contributes (row-min and column-min) only if its image owns the pair
      const int irow = p.q_img0 + (int)((rvalid ? row : p.Mq - 1) / p.P);
      const bool act = rvalid && (!p.sym || pair_owned_grouped(p.groups, irow, img, p.nb_img));
      const float qn = rvalid ? __ldg(p.qn2 + row) : 0.f;
      // images covered by this warp's 32 consecutive rows (at most two when P >= 32)
      const long long wrow0 = row - lane;
      const int ilo = p.q_img0 + (int)(min(wrow0, p.Mq - 1) / p.P);
      const int ihi = p.q_img0 + (int)(min(wrow0 + 31, p.Mq - 1) / p.P);
      float best = INFINITY;
      int bestc = 0;                                        // kArg: column (row inside bank image img) of the running min
      // kArg, sym: this row's index inside its query image rides in the low half of the column-min keys
      const unsigned int rin = (unsigned int)((rvalid ? row : 0) - (long long)(irow - p.q_img0) * p.P);
      for (int t = 0; t < p.nt; ++t, ++tile_ctr) {
        const uint32_t buf = tile_ctr & 1, tphase = (tile_ctr >> 1) & 1;
        const int width = (t == p.nt - 1) ? p.wlast : p.wmain;
        const int valid = min(width, p.P - t * p.wmain);
        const int cbase = t * p.wmain;
        const long long col0 = (long long)img * p.P + cbase;
        float* bn = s_bn2 + buf * kMaxN;
        for (int c = eidx; c < width; c += 128) bn[c] = (c < valid) ? __ldcg(p.bn2 + col0 + c) : INFINITY;   // L2: may have landed during the launch
        asm volatile("bar.sync 1, 128;" ::: "memory");
        mbar_wait(smem_u32(&tfull_bar[buf]), tphase, p.err, 4);
        tc_fence_after();
        const uint32_t taddr = tmem_base + buf * kMaxN + ((uint32_t)(q * 32) << 16);
        for (int c0 = 0; c0 < width; c0 += 32) {
          uint32_t v0[16], v1[16];
          const bool two = (c0 + 16 < width);
          AC_TMEM_LD16(taddr + c0, v0);
          if (two) AC_TMEM_LD16(taddr + c0 + 16, v1);
          tmem_ld_wait();
          if (!p.sym) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float part = fmaf(-2.f, __uint_as_float(v0[i]), bn[c0 + i]);
              if (kArg) { if (part < best) { best = part; bestc = cbase + c0 + i; } }
              else best = fminf(best, part);
            }
            if (two) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float part = fmaf(-2.f, __uint_as_float(v1[i]), bn[c0 + 16 + i]);
                if (kArg) { if (part < best) { best = part; bestc = cbase + c0 + 16 + i; } }
                else best = fminf(best, part);
              }
            }
          } else {
            // row-min as above + column-min over the 32 rows of this warp.  A butterfly "transpose
            // reduction" leaves the min of column c0+l in lane l after 31 shuffles for 32 columns
            // (REDUX.MIN measured ~110 cycles per column here; this is ~4 instructions per column);
            // then one coalesced atomicMin per 32 columns.  Non-negative floats order like their bits.
            float e[32];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float part = fmaf(-2.f, __uint_as_float(v0[i]), bn[c0 + i]);
              if (kArg) { if (part < best) { best = part; bestc = cbase + c0 + i; } }
              else best = fminf(best, part);
              e[i] = fmaxf(part + qn, 0.f);
            }
            if (two) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float part = fmaf(-2.f, __uint_as_float(v1[i]), bn[c0 + 16 + i]);
                if (kArg) { if (part < best) { best = part; bestc = cbase + c0 + 16 + i; } }
                else best = fminf(best, part);
                e[16 + i] = fmaxf(part + qn, 0.f);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) e[16 + i] = INFINITY;
            }
            const bool in_lo = act && (irow == ilo), in_hi = act && (irow == ihi) && (ihi != ilo);
            const int c = c0 + lane;
            if (!kArg) {
              {
                float r[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) r[i] = in_lo ? e[i] : INFINITY;
                const float m = warp_transpose_min(r, lane);
                if (c < valid && m < 3.0e38f)
                  atomicMin(p.colmin + (long long)(ilo - p.q_img0) * ((long long)p.nb_img * p.P) + col0 + c, __float_as_uint(m));
              }
              if (ihi != ilo) {   // warp-uniform: this warp's rows straddle two query images
                float r[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) r[i] = in_hi ? e[i] : INFINITY;
                const float m = warp_transpose_min(r, lane);
                if (c < valid && m < 3.0e38f)
                  atomicMin(p.colmin + (long long)(ihi - p.q_img0) * ((long long)p.nb_img * p.P) + col0 + c, __float_as_uint(m));
              }
            } else {
              // same reduction on (distance bits << 32 | row inside the query image): the winner names its row
              constexpr unsigned long long kNone = ~0ull;
              {
                unsigned long long r[32];
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  r[i] = (in_lo && e[i] < 3.0e38f) ? (((unsigned long long)__float_as_uint(e[i]) << 32) | rin) : kNone;
                const unsigned long long m = warp_transpose_min_u64(r, lane);
                if (c < valid && m != kNone)
                  atomicMin(p.colkey + (long long)(ilo - p.q_img0) * ((long long)p.nb_img * p.P) + col0 + c, m);
              }
              if (ihi != ilo) {
                unsigned long long r[32];
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  r[i] = (in_hi && e[i] < 3.0e38f) ? (((unsigned long long)__float_as_uint(e[i]) << 32) | rin) : kNone;
                const unsigned long long m = warp_transpose_min_u64(r, lane);
                if (c < valid && m != kNone)
                  atomicMin(p.colkey + (long long)(ihi - p.q_img0) * ((long long)p.nb_img * p.P) + col0 + c, m);
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty0 + buf * 8);
      }
      if (act) {
        const float d2 = fmaxf(best + qn, 0.f);
        p.dmin[(long long)img * p.Mq + row] = p.sym ? d2 : sqrtf(d2);
        if (kArg) p.rowarg[(long long)img * p.Mq + row] = bestc;
      }
    }
  }

  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}


// ------------------------------------------------------------------------------------------------
// Device-side construction of the symmetric raster list.  (A host-built list needs an H2D copy, and
// copy-engine work queues behind any large transfer the application has in flight -- measured: +9 ms
// per launch while the next category's features were being uploaded.)
static constexpr int kUnitTab = 4096;     // query blocks whose image range the unit builder tabulates in shared memory
static constexpr int kUnitBlocks = 32;    // CTAs of the two unit-builder kernels (8 warps each)
static constexpr int kUnitWarps = kUnitBlocks * 8;

// Raster rows [ra, rb) of one warp: one lane per query block of the row's group, the activity mask of a row is a ballot.
// The image range of every query block is tabulated in shared memory first, so the row loop carries no 64-bit division.
// COUNT: returns the number of units of the run; otherwise emits them in raster order from position pos.
template <bool COUNT>
__device__ __forceinline__ long long walk_units(const TcParams& p, int2* units, long long pos) {
  __shared__ int s_i0[kUnitTab], s_i1[kUnitTab];
  const int tid = threadIdx.x, lane = tid & 31;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (tid >> 5), nw = gridDim.x * (blockDim.x >> 5);
  const long long rows_per_mb = (long long)kTileM * 2;
  const bool tab = p.n_mblocks <= kUnitTab;
  auto mb_range = [&](int mb, int& i0, int& i1) {
    const long long r0 = (long long)mb * rows_per_mb, r1 = min(p.Mq, r0 + rows_per_mb) - 1;
    i0 = p.q_img0 + (int)(r0 / p.P);
    i1 = p.q_img0 + (int)(r1 / p.P);
  };
  if (tab) {
    for (int mb = tid; mb < p.n_mblocks; mb += blockDim.x) mb_range(mb, s_i0[mb], s_i1[mb]);
  }
  __syncthreads();
  auto has_work = [&](int mb, int img) -> bool {
    int dw = img - p.win_begin;
    if (dw < 0) dw += p.nb_img;
    if (dw >= p.win_count) return false;          // bank image outside this launch's window
    int i0, i1;
    if (tab) { i0 = s_i0[mb]; i1 = s_i1[mb]; } else mb_range(mb, i0, i1);
    for (int i = i0; i <= i1; ++i)
      if (pair_owned_grouped(p.groups, i, img, p.nb_img)) return true;
    return false;
  };
  const int n_groups = (p.n_mblocks + kGM - 1) / kGM;
  const long long rows = (long long)n_groups * p.KU;
  // raster row = (group of kGM query blocks, candidate bank image); the candidates of a group are walked circularly
  // from the first image after the group's first query image (ownership looks forward in that order).
  // A contiguous slice of rows per warp keeps the raster order.
  const long long per = (rows + nw - 1) / nw;
  const long long ra = min(rows, (long long)gw * per), rb = min(rows, ra + per);
  long long cnt = 0;
  if (ra < rb) {
    int mg = (int)(ra / p.KU), k = (int)(ra - (long long)mg * p.KU);
    for (long long r = ra; r < rb; ++r) {
      const int gm_cur = min(kGM, p.n_mblocks - mg * kGM);
      int ig, i1_;
      if (tab) ig = s_i0[mg * kGM]; else mb_range(mg * kGM, ig, i1_);
      int img = ig + 1 + k;                       // < 2 * nb_img
      if (img >= p.nb_img) img -= p.nb_img;
      if (img >= p.nb_img) img -= p.nb_img;
      for (int m0 = 0; m0 < gm_cur; m0 += 32) {
        const int mi = m0 + lane, mb = mg * kGM + mi;
        const bool act = (mi < gm_cur) && has_work(mb, img);
        const unsigned mask = __ballot_sync(0xffffffffu, act);
        if (COUNT) {
          cnt += __popc(mask);
        } else {
          if (act) units[pos + __popc(mask & ((1u << lane) - 1u))] = make_int2(mb, img);
          pos += __popc(mask);
        }
      }
      if (++k == p.KU) { k = 0; ++mg; }
    }
  }
  return cnt;
}

// Two small multi-CTA launches instead of one CTA (which needed 46 us -- 3 % of an 8-GPU config-2 step -- whichever way its
// single SM was used): every warp counts the units of its run of raster rows, then every warp sums the counts of the runs
// before its own (fixed order) and emits.
__global__ void __launch_bounds__(256) count_units_kernel(TcParams p, long long* warp_cnt, int* err_flag) {
  if (blockIdx.x == 0 && threadIdx.x == 0 && err_flag) {
    *err_flag = 0;
    *reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(err_flag) + 128) = 0ull;   // unit claim counter
  }
  const long long cnt = walk_units<true>(p, nullptr, 0);
  if ((threadIdx.x & 31) == 0) warp_cnt[blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)] = cnt;
}

__global__ void __launch_bounds__(256) emit_units_kernel(TcParams p, const long long* __restrict__ warp_cnt, int2* units,
                                                         long long* n_units) {
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nw = gridDim.x * (blockDim.x >> 5);
  long long before = 0, all = 0;
  for (int w = lane; w < nw; w += 32) {
    const long long c = warp_cnt[w];
    all += c;
    if (w < gw) before += c;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    before += __shfl_xor_sync(0xffffffffu, before, off);
    all += __shfl_xor_sync(0xffffffffu, all, off);
  }
  if (gw == 0 && lane == 0) *n_units = all;
  walk_units<false>(p, units, before);
}

// grid-stride fill (SM-side replacement of cudaMemsetAsync: keeps the launch sequence off the copy engines)
__global__ void fill_u32_kernel(unsigned int* __restrict__ dst, long long n, unsigned int v) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dst[i] = v;
}

// ------------------------------------------------------------------------------------------------ host
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess || !ptr) return nullptr;
  fn = (PFN_encodeTiled)ptr;
  return fn;
}

static int make_map(CUtensorMap* m, const void* base, long long rows, int D, int box_rows, bool bf16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return AC_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)D * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims,
                   strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { g_last_cuda_error = 1000 + (int)r; return AC_ERR_CUDA; }
  return AC_OK;
}

static uint32_t make_idesc(int M, int N, bool bf16) {
  uint32_t d = 0;
  d |= 1u << 4;                       // accumulator format: F32
  d |= (bf16 ? 1u : 0u) << 7;         // A format
  d |= (bf16 ? 1u : 0u) << 10;        // B format
  // bits 13/14: no negate; bits 15/16: A and B K-major
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// Watchdog flag in pinned, mapped host memory (one per process, every device sees it through UVA): device memory cannot be
// read back once the kernel has trapped, this can.
static int* g_wd_host = nullptr;
static int* g_wd_dev = nullptr;
static std::once_flag g_wd_once;
static int* watchdog_flag() {
  std::call_once(g_wd_once, [] {
    int* h = nullptr;
    if (cudaHostAlloc((void**)&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); return; }
    *h = 0;
    int* d = nullptr;
    if (cudaHostGetDevicePointer((void**)&d, h, 0) != cudaSuccess) { (void)cudaGetLastError(); d = h; }
    g_wd_host = h;
    g_wd_dev = d;
  });
  return g_wd_dev;   // null when the allocation failed: the kernels then only trap
}

template <bool kArg>
static int launch_tc(const TcParams& prm, int num_sms, cudaStream_t st) {
  constexpr size_t kStageBytes = (size_t)kTileM * kBlockK * 2 + (size_t)kBRows * kBlockK * 2;
  const size_t smem = 1024 + kStages * kStageBytes + 2 * kMaxN * sizeof(float) + (2 * kStages + 4) * 8 + 256;
  auto kern = mindist_tc_kernel<kArg>;
  AC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int pairs = (int)std::min<long long>(num_sms / 2, prm.total_units);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pairs * 2);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AC_CUDA(cudaLaunchKernelEx(&cfg, kern, prm));
  __atomic_fetch_add(&g_kernel_launches, 1ull, __ATOMIC_RELAXED);
  return AC_OK;
}

int launch_mindist_tc(const void* Qhi, const void* Qlo, const float* Qn2, long long Mq, const void* Bhi, const void* Blo,
                      const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int* err_flag, cudaStream_t st,
                      int sym = 0, int q_img0 = 0, unsigned int* colmin = nullptr, void* unit_ws = nullptr, size_t unit_ws_bytes = 0,
                      int win_begin = 0, int win_count = -1, int* rowarg = nullptr, unsigned long long* colkey = nullptr,
                      const int* groups = nullptr, const int* bank_ready = nullptr, int img_rot = 0) {
  const bool bf16 = (precision == AC_PREC_BF16 || precision == AC_PREC_BF16X3);
  const bool x3 = (precision == AC_PREC_F16X3 || precision == AC_PREC_BF16X3);
  if (D % 8 != 0) return AC_ERR_UNSUPPORTED;  // TMA needs a 16-byte row pitch
  if (x3 && (!Qlo || !Blo)) return AC_ERR_INVALID;
  TcParams prm;
  memset(&prm, 0, sizeof(prm));
  // tile widths inside one bank image: multiples of 16, <= 256, as even as possible
  int nt = ceil_div(P, kMaxN);
  int wmain = std::min(kMaxN, ceil_div(ceil_div(P, nt), 16) * 16);
  nt = ceil_div(P, wmain);
  const int wlast = ceil_div(P - (nt - 1) * wmain, 16) * 16;
  prm.nt = nt; prm.wmain = wmain; prm.wlast = wlast;
  prm.qn2 = Qn2; prm.bn2 = Bn2; prm.dmin = dmin; prm.err = watchdog_flag();
  prm.Mq = Mq; prm.nb_img = nb_img; prm.P = P; prm.D = D;
  prm.nkb = ceil_div(D, kBlockK);
  prm.nseg = x3 ? 3 : 1;
  prm.n_mblocks = (int)ceil_div64(Mq, (long long)kTileM * 2);
  prm.counter = (unsigned long long*)((char*)err_flag + 128);   // inside the zeroed 256-byte workspace header
  prm.sym = sym; prm.q_img0 = q_img0; prm.colmin = colmin; prm.units = nullptr;
  prm.rowarg = rowarg; prm.colkey = colkey; prm.groups = groups; prm.bank_ready = bank_ready; prm.img_rot = sym ? 0 : img_rot;
  const bool arg = (rowarg != nullptr);
  if (arg && sym && !colkey) return AC_ERR_INVALID;
  prm.win_begin = win_begin; prm.win_count = (win_count < 0) ? nb_img : win_count;
  // bank images a raster group of kGM query blocks can own: N/2 after each of the images it spans (with categories the
  // group may end in the middle of one whose images wrap around: every bank image is a candidate)
  prm.KU = groups ? nb_img : std::min(nb_img, nb_img / 2 + (int)(((long long)kGM * kTileM * 2 - 1) / P) + 1);
  prm.total_units = (long long)prm.n_mblocks * nb_img;
  if (sym) {
    // raster order: groups of kGM query blocks; inside a group walk the bank images the group owns and,
    // per bank image, every block of the group that owns the pair (blocks sharing a bank image run
    // together).  Built on the device (count_units_kernel + emit_units_kernel).
    // a query block spans at most rows/P + 2 images, each owns at most half of its category (<= nb_img / 2 + 1 images)
    const long long span = ((long long)kTileM * 2 + P - 1) / P + 1;
    const long long max_units = (long long)prm.n_mblocks * std::min<long long>(nb_img, span * (nb_img / 2 + 1));
    if (!unit_ws || unit_ws_bytes < 16 + (size_t)max_units * sizeof(int2) + kUnitWarps * sizeof(long long)) return AC_ERR_WORKSPACE;
    long long* d_n = (long long*)unit_ws;
    int2* d_units = (int2*)((char*)unit_ws + 16);
    long long* d_cnt = (long long*)((char*)unit_ws + 16 + (size_t)max_units * sizeof(int2));     // one count per builder warp
    count_units_kernel<<<kUnitBlocks, 256, 0, st>>>(prm, d_cnt, err_flag);
    AC_LAUNCH_CHECK();
    emit_units_kernel<<<kUnitBlocks, 256, 0, st>>>(prm, d_cnt, d_units, d_n);
    AC_LAUNCH_CHECK();
    prm.units = d_units;
    prm.n_units = d_n;
    prm.total_units = max_units;   // upper bound (sizes the grid); the kernel reads the exact count
  }
  prm.idesc_main = make_idesc(kTileM * 2, wmain, bf16);
  prm.idesc_last = make_idesc(kTileM * 2, wlast, bf16);
  const long long brows = (long long)nb_img * P;
  int rc;
  if ((rc = make_map(&prm.mapA[0], Qhi, Mq, D, kTileM, bf16))) return rc;
  if ((rc = make_map(&prm.mapBmain[0], Bhi, brows, D, wmain / 2, bf16))) return rc;
  if ((rc = make_map(&prm.mapBlast[0], Bhi, brows, D, wlast / 2, bf16))) return rc;
  if (x3) {
    if ((rc = make_map(&prm.mapA[1], Qlo, Mq, D, kTileM, bf16))) return rc;
    if ((rc = make_map(&prm.mapBmain[1], Blo, brows, D, wmain / 2, bf16))) return rc;
    if ((rc = make_map(&prm.mapBlast[1], Blo, brows, D, wlast / 2, bf16))) return rc;
  } else {
    prm.mapA[1] = prm.mapA[0]; prm.mapBmain[1] = prm.mapBmain[0]; prm.mapBlast[1] = prm.mapBlast[0];
  }
  int dev = 0, num_sms = 0;
  AC_CUDA(cudaGetDevice(&dev));
  AC_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  return arg ? launch_tc<true>(prm, num_sms, st) : launch_tc<false>(prm, num_sms, st);
}

int launch_mindist_simt(const float* Q, long long Mq, const float* Bk, int nb_img, int P, int D, float* dmin, cudaStream_t st);

}  // namespace ac

using namespace ac;

extern "C" int ac_last_watchdog(void) {
  if (!g_wd_host) return 0;
  const int code = *reinterpret_cast<volatile int*>(g_wd_host);
  *reinterpret_cast<volatile int*>(g_wd_host) = 0;
  return code;
}

// w[r] = mean over the other images j of the category of sqrt(d2(r, j)), d2 taken from whichever of the two minima the
// ownership rule says was written.  A block handles 64 query rows x 4 quarters of the bank-image range (a sharded run has
// only ~10^4 rows per rank: one thread per row left most SMs idle and ran ~100 dependent loads per thread); the four
// partial sums are added in a fixed order, so the result does not depend on the launch geometry.
__global__ void __launch_bounds__(256) reduce_weights_sym_kernel(const float* __restrict__ rowmin, const float* __restrict__ colmin,
                                                                 long long Mq, int nb_img, int Pq, int q_img0,
                                                                 const int* __restrict__ groups, float* __restrict__ w) {
  __shared__ float s_part[4][64];
  const int rr = threadIdx.x & 63, part = threadIdx.x >> 6;
  const long long r = blockIdx.x * 64LL + rr;
  float s = 0.f;
  int j0 = 0, j1 = 0, i = 0;
  if (r < Mq) {
    i = q_img0 + (int)(r / Pq);
    j0 = groups ? groups[2 * i] : 0;                       // the image's own category
    j1 = groups ? j0 + groups[2 * i + 1] : nb_img;
    const int len = j1 - j0, chunk = (len + 3) >> 2;
    const int ja = j0 + part * chunk, jb = min(j1, ja + chunk);
    for (int jq = ja; jq < jb; jq += 8) {
      float d[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int j = jq + u;
        d[u] = -1.f;
        if (j < jb && j != i) {
          const float* src = pair_owned_grouped(groups, i, j, nb_img) ? rowmin : colmin;
          d[u] = __ldg(src + (long long)j * Mq + r);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (d[u] >= 0.f) s += sqrtf(d[u]);
    }
  }
  s_part[part][rr] = s;
  __syncthreads();
  if (part == 0 && r < Mq) {
    const int cnt = (j1 - j0) - ((i >= j0 && i < j1) ? 1 : 0);
    const float tot = ((s_part[0][rr] + s_part[1][rr]) + s_part[2][rr]) + s_part[3][rr];
    w[r] = cnt > 0 ? tot / (float)cnt : nanf("");
  }
}

static int min_dist_sym_impl(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                             const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                             int bank_count, int init_colmin, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                             const int32_t* groups, void* ws, size_t ws_bytes, ac_stream_t stream, const int32_t* bank_ready = nullptr) {
  const bool arg = (rowarg != nullptr);
  if (!Qhi || !Bhi || !Qn2 || !Bn2 || !rowmin_d2 || (!arg && !colmin_d2) || (arg && !colkey) || Mq < 0 || nb_img < 1 || P < 1 ||
      D < 1 || q_img0 < 0)
    return AC_ERR_INVALID;
  if (bank_begin < 0 || bank_begin >= nb_img || bank_count < 0 || bank_count > nb_img) return AC_ERR_INVALID;
  if (precision < AC_PREC_F16 || precision > AC_PREC_BF16X3) return AC_ERR_UNSUPPORTED;  // tensor-core modes only
  if (P < 32 || Mq % P != 0) return AC_ERR_UNSUPPORTED;  // a warp of 32 rows may span at most two query images
  if (q_img0 + Mq / P > nb_img) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (Mq == 0) return AC_OK;
  if (!ws || ws_bytes < 256) return AC_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  // column minima are accumulated with atomicMin on the fp32 bit pattern: start from a huge finite value
  if (init_colmin) {
    // float minima: one word per entry; (distance, row) keys: two words per entry -- same byte pattern, huge and finite
    const long long words = (long long)(Mq / P) * nb_img * P * (arg ? 2 : 1);
    const int blocks = (int)std::min<long long>((words + 1023) / 1024, 148LL * 8);
    fill_u32_kernel<<<blocks, 256, 0, st>>>(arg ? (unsigned int*)colkey : (unsigned int*)colmin_d2, words, 0x7f7f7f7fu);
    AC_LAUNCH_CHECK();
  }
  return launch_mindist_tc(Qhi, Qlo, Qn2, Mq, Bhi, Blo, Bn2, nb_img, P, D, precision, rowmin_d2, (int*)ws, st, 1, q_img0,
                           (unsigned int*)colmin_d2, (char*)ws + 256, ws_bytes - 256, bank_begin, bank_count, rowarg,
                           (unsigned long long*)colkey, groups, bank_ready);
}

extern "C" int ac_min_dist_sym(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                               const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                               int bank_count, int init_colmin, float* rowmin_d2, float* colmin_d2, void* ws, size_t ws_bytes,
                               ac_stream_t stream) {
  return min_dist_sym_impl(Qhi, Qlo, Qn2, Mq, q_img0, Bhi, Blo, Bn2, nb_img, P, D, precision, bank_begin, bank_count, init_colmin,
                           rowmin_d2, colmin_d2, nullptr, nullptr, nullptr, ws, ws_bytes, stream);
}

extern "C" int ac_min_dist_sym_ex(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                                  const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                                  int bank_count, int init, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                                  const int32_t* groups, void* ws, size_t ws_bytes, ac_stream_t stream) {
  if ((rowarg != nullptr) != (colkey != nullptr)) return AC_ERR_INVALID;
  return min_dist_sym_impl(Qhi, Qlo, Qn2, Mq, q_img0, Bhi, Blo, Bn2, nb_img, P, D, precision, bank_begin, bank_count, init,
                           rowmin_d2, colmin_d2, rowarg, colkey, groups, ws, ws_bytes, stream);
}

extern "C" int ac_min_dist_sym_ready(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                                     const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                                     int bank_count, int init, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                                     const int32_t* groups, const int32_t* bank_ready, void* ws, size_t ws_bytes, ac_stream_t stream) {
  if ((rowarg != nullptr) != (colkey != nullptr)) return AC_ERR_INVALID;
  return min_dist_sym_impl(Qhi, Qlo, Qn2, Mq, q_img0, Bhi, Blo, Bn2, nb_img, P, D, precision, bank_begin, bank_count, init,
                           rowmin_d2, colmin_d2, rowarg, colkey, groups, ws, ws_bytes, stream, bank_ready);
}

extern "C" int ac_min_dist_sym_arg(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                                   const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                                   int bank_count, int init_colkey, float* rowmin_d2, int32_t* rowarg, uint64_t* colkey, void* ws,
                                   size_t ws_bytes, ac_stream_t stream) {
  if (!rowarg || !colkey) return AC_ERR_INVALID;
  return min_dist_sym_impl(Qhi, Qlo, Qn2, Mq, q_img0, Bhi, Blo, Bn2, nb_img, P, D, precision, bank_begin, bank_count, init_colkey,
                           rowmin_d2, nullptr, rowarg, colkey, nullptr, ws, ws_bytes, stream);
}

extern "C" int ac_reduce_weights_sym_ex(const float* rowmin_d2, const float* colmin_d2, int64_t Mq, int nb_img, int Pq, int q_img0,
                                        const int32_t* groups, float* w, ac_stream_t stream) {
  if (!rowmin_d2 || !colmin_d2 || !w || Mq < 0 || nb_img < 1 || Pq < 1 || q_img0 < 0) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (Mq == 0) return AC_OK;
  reduce_weights_sym_kernel<<<(unsigned)((Mq + 63) / 64), 256, 0, (cudaStream_t)stream>>>(rowmin_d2, colmin_d2, Mq, nb_img, Pq, q_img0,
                                                                                            groups, w);
  AC_LAUNCH_CHECK();
  return AC_OK;
}

extern "C" int ac_reduce_weights_sym(const float* rowmin_d2, const float* colmin_d2, int64_t Mq, int nb_img, int Pq, int q_img0,
                                     float* w, ac_stream_t stream) {
  return ac_reduce_weights_sym_ex(rowmin_d2, colmin_d2, Mq, nb_img, Pq, q_img0, nullptr, w, stream);
}

extern "C" size_t ac_min_dist_workspace_bytes(int64_t Mq, int nb_img, int P, int D, int precision) {
  (void)D; (void)precision;
  // 256 B pipeline-watchdog flag + (symmetric form) the raster list of (query block, bank image) units
  // sized for 128-row query blocks: an upper bound for the 256-row blocks of the CTA pairs (more blocks, and a per-block
  // span bound at least that of launch_mindist_tc)
  const long long mblocks = (Mq + 127) / 128;
  const long long span = (256 + std::max(1, P) - 1) / std::max(1, P) + 1;
  const long long per_mb = std::min<long long>(nb_img, span * (nb_img / 2 + 1));
  return 256 + 16 + (size_t)(mblocks * per_mb) * sizeof(int2) + 4096;   // + the unit builder's per-warp counts
}

static int min_dist_impl(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                         const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int32_t* argmin, void* ws,
                         size_t ws_bytes, ac_stream_t stream, const int32_t* bank_ready = nullptr, int first_bank_image = 0) {
  if (!Qhi || !Bhi || !dmin || Mq < 0 || nb_img < 1 || P < 1 || D < 1) return AC_ERR_INVALID;
  if (first_bank_image < 0 || first_bank_image >= nb_img) return AC_ERR_INVALID;
  if (bank_ready && precision == AC_PREC_F32) return AC_ERR_UNSUPPORTED;   // arrival flags: tensor-core kernel only
  if (argmin && precision == AC_PREC_F32) return AC_ERR_UNSUPPORTED;   // the exact kernel needs no refinement
  if (precision < AC_PREC_F16 || precision > AC_PREC_F32) return AC_ERR_INVALID;
  int rc = check_device();
  if (rc) return rc;
  if (Mq == 0) return AC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == AC_PREC_F32)
    return launch_mindist_simt((const float*)Qhi, Mq, (const float*)Bhi, nb_img, P, D, dmin, st);
  if (!Qn2 || !Bn2) return AC_ERR_INVALID;
  if (!ws || ws_bytes < 256) return AC_ERR_WORKSPACE;
  fill_u32_kernel<<<1, 64, 0, st>>>((unsigned int*)ws, 64, 0u);   // watchdog flag (no copy-engine memset)
  AC_LAUNCH_CHECK();
  return launch_mindist_tc(Qhi, Qlo, Qn2, Mq, Bhi, Blo, Bn2, nb_img, P, D, precision, dmin, (int*)ws, st, 0, 0, nullptr, nullptr, 0, 0,
                           -1, argmin, nullptr, nullptr, bank_ready, first_bank_image);
}

extern "C" int ac_min_dist_ready(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                                 const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int32_t* argmin,
                                 const int32_t* bank_ready, int first_bank_image, void* ws, size_t ws_bytes, ac_stream_t stream) {
  return min_dist_impl(Qhi, Qlo, Qn2, Mq, Bhi, Blo, Bn2, nb_img, P, D, precision, dmin, argmin, ws, ws_bytes, stream, bank_ready,
                       first_bank_image);
}

extern "C" int ac_min_dist(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                           const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, void* ws, size_t ws_bytes,
                           ac_stream_t stream) {
  return min_dist_impl(Qhi, Qlo, Qn2, Mq, Bhi, Blo, Bn2, nb_img, P, D, precision, dmin, nullptr, ws, ws_bytes, stream);
}

extern "C" int ac_min_dist_arg(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                               const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int32_t* argmin, void* ws,
                               size_t ws_bytes, ac_stream_t stream) {
  if (!argmin) return AC_ERR_INVALID;
  return min_dist_impl(Qhi, Qlo, Qn2, Mq, Bhi, Blo, Bn2, nb_img, P, D, precision, dmin, argmin, ws, ws_bytes, stream);
}
