// lvo_extract.cuh — lvo_extract_features: the laserCloudHandler body, reference src/scanRegistration.cpp:127-411,
// as sm_100a kernels.  One launch sequence serves every lane (blockIdx.y = lane).
//
//   k_classify      :136-137 range/NaN filter, :166-200 ring id, :208 azimuth                 (A1, A2)
//   k_ring_count    :141-153 start/end azimuth, :209-236 halfPassed switch point as a min-index reduction,
//                   per-block ring histogram for the stable bucket                             (A3, A4)
//   k_ring_offsets  per-ring exclusive offsets, scanStartInd/scanEndInd :246-252               (A4)
//   k_ring_scatter  :238-240 relTime/intensity + stable counting sort by ring                  (A3, A4)
//   k_curvature     :256-266 11-tap curvature, plus the neighbour gap flags of :319-342         (A5)
//   k_sector_pick_fast / k_sector_pick   one CTA per ring: :277-399 sector sort + greedy sharp/flat picking, :392-407 less-flat
//                   gather and the per-ring 0.2 m voxel filter.  Fast kernel: register / warp-shuffle bitonic sorts, picks out of
//                   shared memory; generic kernel (block bitonic sorts in shared memory) for oversize rings       (A6-A10)
//   k_feature_compact  concatenation of the per-sector / per-ring results in reference order   (A7-A9)
//
// Exactness (SURVEY Appendix A): this TU is compiled with -fmad=false, every float expression is written in the
// reference's association order, float-vs-double-literal comparisons widen the float first.
#pragma once
#include "lvo_internal.h"
#include "lvo_prims.cuh"
#include <float.h>
#include <limits.h>

#define LVO_EX_THREADS 256
#define LVO_PICK_THREADS 128
#define LVO_PICK_SMEM_KEYS 3072  // 6 x 512 padded sector keys, or one ring's voxel keys (24 KB)
#define LVO_PICK_RING_SMEM 4096  // rings up to this many points keep their picked flags in shared memory

struct ExtractArgs {
  // input
  const unsigned char* const* in_ptr;  // [lanes] device pointers to raw point records
  const int* in_n;                     // [lanes] (0 for an idle lane)
  const int* lane_flags;               // [lanes] LVO_LANE_* of the step: the kernels below leave an idle lane's state alone
  int in_stride, in_off_xyz;
  const LaneConfig* lcfg;              // [lanes] n_scans and (float)MINIMUM_RANGE of each lane
  int max_scans;                       // lvo_config::n_scans: sizes the per-ring grids only; rings at or above a lane's n_scans are empty
  int P;                               // capacity per lane
  int nblk_cap;                        // ceil(P / LVO_EX_THREADS)
  LaneState* ls;
  // per-lane arrays of stride P
  signed char* ring;       // -2 dropped by range/NaN, -1 rejected by ring test, else ring id
  float* ori;
  int* blkcnt;             // [lanes][nblk_cap][64]
  float4* full;
  float* curv;
  unsigned char* gapbig;
  int* sort_ind; int* picked; int* label;
  // sector results: [lanes][64][6][...]
  int* slot_sharp;   // 2 per sector
  int* slot_lsharp;  // 20 per sector
  int* slot_flat;    // 4 per sector
  int* slot_cnt;     // 3 per sector: n_sharp, n_less_sharp, n_flat
  float4* lf_ring;   // per-ring voxel-filtered less-flat, stored at ring_start[ring]
  int* lf_cnt;       // [lanes][64]
  unsigned long long* sort_scratch;  // [lanes][2P] global fallback for oversize sorts
  int* ring_done;                    // [lanes][64] 1 = k_sector_pick_fast handled the ring
  // outputs (stride P except sharp/flat which have their own caps)
  float4* sharp; float4* less_sharp; float4* flat; float4* less_flat;
  int cap_sharp, cap_lsharp, cap_flat;
};

// ring id, literal C++ conversions of scanRegistration.cpp:166-200 (see oracle/scan_registration.hpp ring_of)
__device__ __forceinline__ int ring_of_dev(float x, float y, float z, int N_SCANS) {
  float angle = (float)((double)(lvo_atanf(z / sqrtf(x * x + y * y)) * 180) / LVO_PI);
  int scanID;
  if (N_SCANS == 16) {
    scanID = int((angle + 15) / 2 + 0.5);
    if (scanID > (N_SCANS - 1) || scanID < 0) return -1;
  } else if (N_SCANS == 32) {
    scanID = int((angle + 92.0 / 3.0) * 3.0 / 4.0);
    if (scanID > (N_SCANS - 1) || scanID < 0) return -1;
  } else {
    if (angle >= -8.83) scanID = int((2 - angle) * 3.0 + 0.5);
    else scanID = N_SCANS / 2 + int((-8.83 - angle) * 2.0 + 0.5);
    if (angle > 2 || angle < -24.33 || scanID > 50 || scanID < 0) return -1;
  }
  return scanID;
}

__device__ __forceinline__ float3 load_xyz(const unsigned char* base, int stride, int off, int i) {
  const float* p = reinterpret_cast<const float*>(base + (size_t)i * stride + off);
  return make_float3(p[0], p[1], p[2]);
}

__global__ void k_extract_reset(ExtractArgs a) {
  LaneState& s = a.ls[blockIdx.x];
  if (threadIdx.x == 0 && lane_active(a.lane_flags, blockIdx.x)) {
    s.n_in = a.in_n[blockIdx.x];
    s.first_kept = INT_MAX; s.last_kept = -1; s.switch_idx = INT_MAX; s.n_kept = 0;
    s.n_sharp = s.n_less_sharp = s.n_flat = s.n_less_flat = 0;
  }
}

__global__ void __launch_bounds__(LVO_EX_THREADS) k_classify(ExtractArgs a) {
  const int lane = blockIdx.y;
  const int n = a.in_n[lane];
  const LaneConfig lc = a.lcfg[lane];
  const int i = blockIdx.x * LVO_EX_THREADS + threadIdx.x;
  bool kept = false;
  if (i < n) {
    float3 p = load_xyz(a.in_ptr[lane], a.in_stride, a.in_off_xyz, i);
    kept = isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && !(p.x * p.x + p.y * p.y + p.z * p.z < lc.thres * lc.thres);
    int ring = -2;
    float ori = 0.f;
    if (kept) {
      ring = ring_of_dev(p.x, p.y, p.z, lc.n_scans);
      ori = -lvo_atan2f(p.y, p.x);
    }
    a.ring[(size_t)lane * a.P + i] = (signed char)ring;
    a.ori[(size_t)lane * a.P + i] = ori;
  }
  // first / last kept index
  int mn = kept ? i : INT_MAX, mx = kept ? i : -1;
  mn = __reduce_min_sync(0xffffffffu, mn);
  mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0) {
    if (mn != INT_MAX) atomicMin(&a.ls[lane].first_kept, mn);
    if (mx >= 0) atomicMax(&a.ls[lane].last_kept, mx);
  }
}

// start / end azimuth of the sweep, scanRegistration.cpp:141-153
__device__ __forceinline__ void sweep_ori(const ExtractArgs& a, int lane, float* startOri, float* endOri) {
  const LaneState& s = a.ls[lane];
  float so = 0.f, eo = 0.f;
  if (s.last_kept >= 0) {
    so = a.ori[(size_t)lane * a.P + s.first_kept];
    eo = (float)((double)a.ori[(size_t)lane * a.P + s.last_kept] + 2 * LVO_PI);
    if (eo - so > 3 * LVO_PI) eo = (float)((double)eo - 2 * LVO_PI);
    else if (eo - so < LVO_PI) eo = (float)((double)eo + 2 * LVO_PI);
  }
  *startOri = so; *endOri = eo;
}

__global__ void __launch_bounds__(LVO_EX_THREADS) k_ring_count(ExtractArgs a) {
  __shared__ int h[LVO_MAX_RINGS];
  __shared__ float s_ori[2];
  const int lane = blockIdx.y;
  const int n = a.in_n[lane];
  if (blockIdx.x * LVO_EX_THREADS >= n) return;
  if (threadIdx.x < LVO_MAX_RINGS) h[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    sweep_ori(a, lane, &s_ori[0], &s_ori[1]);
    if (blockIdx.x == 0) { a.ls[lane].start_ori = s_ori[0]; a.ls[lane].end_ori = s_ori[1]; }
  }
  __syncthreads();
  const float startOri = s_ori[0];
  const int i = blockIdx.x * LVO_EX_THREADS + threadIdx.x;
  int sw = INT_MAX;
  if (i < n) {
    int ring = a.ring[(size_t)lane * a.P + i];
    if (ring >= 0) {
      atomicAdd(&h[ring], 1);
      float ori = a.ori[(size_t)lane * a.P + i];
      // the unwrapping every point gets while !halfPassed (:211-218); the first point for which the test of :220
      // fires is where the sequential flag flips
      if (ori < startOri - LVO_PI / 2) ori = (float)((double)ori + 2 * LVO_PI);
      else if (ori > startOri + LVO_PI * 3 / 2) ori = (float)((double)ori - 2 * LVO_PI);
      if (ori - startOri > LVO_PI) sw = i;
    }
  }
  sw = __reduce_min_sync(0xffffffffu, sw);
  if ((threadIdx.x & 31) == 0 && sw != INT_MAX) atomicMin(&a.ls[lane].switch_idx, sw);
  __syncthreads();
  if (threadIdx.x < LVO_MAX_RINGS) a.blkcnt[((size_t)lane * a.nblk_cap + blockIdx.x) * LVO_MAX_RINGS + threadIdx.x] = h[threadIdx.x];
}

__global__ void k_ring_offsets(ExtractArgs a) {
  const int lane = blockIdx.x;
  LaneState& s = a.ls[lane];
  const int n = a.in_n[lane];
  if (!lane_active(a.lane_flags, lane)) return;
  const int nblk = (n + LVO_EX_THREADS - 1) / LVO_EX_THREADS;
  const int r = threadIdx.x;  // 64 threads
  int run = 0;
  int* col = a.blkcnt + (size_t)lane * a.nblk_cap * LVO_MAX_RINGS + r;
  for (int b = 0; b < nblk; ++b) {
    int c = col[(size_t)b * LVO_MAX_RINGS];
    col[(size_t)b * LVO_MAX_RINGS] = run;
    run += c;
  }
  s.ring_count[r] = run;
  __syncthreads();
  if (r == 0) {
    const int ns = a.lcfg[lane].n_scans;
    int acc = 0;
    for (int k = 0; k < LVO_MAX_RINGS; ++k) {
      s.ring_start[k] = acc;
      if (k < ns) s.scan_start[k] = acc + 5;   // :249
      acc += s.ring_count[k];
      if (k < ns) s.scan_end[k] = acc - 6;     // :251
    }
    s.ring_start[LVO_MAX_RINGS] = acc;
    s.n_kept = acc;
    s.stats.n_in = n;
    s.stats.n_kept = acc;
  }
}

__global__ void __launch_bounds__(LVO_EX_THREADS) k_ring_scatter(ExtractArgs a) {
  __shared__ int wcnt[LVO_EX_THREADS / 32][LVO_MAX_RINGS];
  const int lane = blockIdx.y;
  const int n = a.in_n[lane];
  if (blockIdx.x * LVO_EX_THREADS >= n) return;
  const LaneState& s = a.ls[lane];
  for (int k = threadIdx.x; k < (LVO_EX_THREADS / 32) * LVO_MAX_RINGS; k += LVO_EX_THREADS) (&wcnt[0][0])[k] = 0;
  __syncthreads();
  const int i = blockIdx.x * LVO_EX_THREADS + threadIdx.x;
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  int ring = -1;
  if (i < n) ring = a.ring[(size_t)lane * a.P + i];
  const unsigned m = __match_any_sync(0xffffffffu, ring);
  const int rank = __popc(m & ((1u << ln) - 1u));
  if (ring >= 0 && rank == 0) wcnt[w][ring] = __popc(m);
  __syncthreads();
  if (threadIdx.x < LVO_MAX_RINGS) {
    int run = 0;
    for (int ww = 0; ww < LVO_EX_THREADS / 32; ++ww) { int t = wcnt[ww][threadIdx.x]; wcnt[ww][threadIdx.x] = run; run += t; }
  }
  __syncthreads();
  if (ring >= 0) {
    const float startOri = s.start_ori, endOri = s.end_ori;
    float ori = a.ori[(size_t)lane * a.P + i];
    if (i <= s.switch_idx) {   // processed while !halfPassed (:209-224)
      if (ori < startOri - LVO_PI / 2) ori = (float)((double)ori + 2 * LVO_PI);
      else if (ori > startOri + LVO_PI * 3 / 2) ori = (float)((double)ori - 2 * LVO_PI);
    } else {                   // :225-236
      ori = (float)((double)ori + 2 * LVO_PI);
      if (ori < endOri - LVO_PI * 3 / 2) ori = (float)((double)ori + 2 * LVO_PI);
      else if (ori > endOri + LVO_PI / 2) ori = (float)((double)ori - 2 * LVO_PI);
    }
    float relTime = (ori - startOri) / (endOri - startOri);  // :238
    float3 p = load_xyz(a.in_ptr[lane], a.in_stride, a.in_off_xyz, i);
    const int dst = s.ring_start[ring] + a.blkcnt[((size_t)lane * a.nblk_cap + blockIdx.x) * LVO_MAX_RINGS + ring] + wcnt[w][ring] + rank;
    a.full[(size_t)lane * a.P + dst] = make_float4(p.x, p.y, p.z, (float)(ring + 0.1 * relTime));  // :239 scanPeriod = 0.1
  }
}

__global__ void __launch_bounds__(LVO_EX_THREADS) k_curvature(ExtractArgs a) {
  const int lane = blockIdx.y;
  const int n = a.ls[lane].n_kept;                   // an idle lane's n_kept is its last frame's
  const bool active = lane_active(a.lane_flags, lane);   // (loaded together with n_kept: no extra latency on the way to the work)
  const int i = blockIdx.x * LVO_EX_THREADS + threadIdx.x;
  if (i >= n || !active) return;
  const float4* P = a.full + (size_t)lane * a.P;
  float c = 0.f;
  const float4 p0 = P[i];
  if (i >= 5 && i < n - 5) {  // :256-266, strictly left to right
    float4 m5 = P[i - 5], m4 = P[i - 4], m3 = P[i - 3], m2 = P[i - 2], m1 = P[i - 1];
    float4 p1 = P[i + 1], p2 = P[i + 2], p3 = P[i + 3], p4 = P[i + 4], p5 = P[i + 5];
    float diffX = m5.x + m4.x + m3.x + m2.x + m1.x - 10 * p0.x + p1.x + p2.x + p3.x + p4.x + p5.x;
    float diffY = m5.y + m4.y + m3.y + m2.y + m1.y - 10 * p0.y + p1.y + p2.y + p3.y + p4.y + p5.y;
    float diffZ = m5.z + m4.z + m3.z + m2.z + m1.z - 10 * p0.z + p1.z + p2.z + p3.z + p4.z + p5.z;
    c = diffX * diffX + diffY * diffY + diffZ * diffZ;
  }
  unsigned char g = 0;
  if (i + 1 < n) {  // gap test of :321-324 between points i and i+1 (the squared distance is symmetric)
    float4 q = P[i + 1];
    float dx = q.x - p0.x, dy = q.y - p0.y, dz = q.z - p0.z;
    g = (dx * dx + dy * dy + dz * dz > 0.05) ? 1 : 0;
  }
  const size_t o = (size_t)lane * a.P + i;
  a.curv[o] = c; a.gapbig[o] = g;
  a.sort_ind[o] = (i >= 5 && i < n - 5) ? i : 0;
  a.picked[o] = 0; a.label[o] = 0;
}

// ascending bitonic sort of keys[0..npad), npad a power of two; whole block participates
__device__ __forceinline__ void block_bitonic_sort(unsigned long long* keys, int npad) {
  for (int k = 2; k <= npad; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < npad; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          unsigned long long x = keys[i], y = keys[ixj];
          const bool up = (i & k) == 0;
          if ((x > y) == up) { keys[i] = y; keys[ixj] = x; }
        }
      }
      __syncthreads();
    }
}
__device__ __forceinline__ int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
// nseg independent ascending sorts of npad keys each (segment s at keys + s * npad), one block barrier per network step
__device__ __forceinline__ void block_bitonic_sort_multi(unsigned long long* keys, int nseg, int npad) {
  const int half = npad >> 1, total = nseg * half;
  for (int k = 2; k <= npad; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int sg = t / half, u = t - sg * half;
        const int i = ((u & ~(j - 1)) << 1) | (u & (j - 1));   // u-th index with bit j clear
        unsigned long long* kk = keys + sg * npad;
        const unsigned long long x = kk[i], y = kk[i | j];
        const bool up = (i & k) == 0;
        if ((x > y) == up) { kk[i] = y; kk[i | j] = x; }
      }
      __syncthreads();
    }
}

// Marks the neighbours of a picked point (:319-342 / :365-388).  Called by a full warp.
// cloudNeighborPicked of one ring: shared memory while the picks run (written back afterwards), global for oversize rings
struct PickedRef {
  volatile unsigned char* sm; volatile int* gl; int r0; bool use_sm;
  __device__ __forceinline__ int get(int i) const { return use_sm ? (int)sm[i - r0] : gl[i]; }
  __device__ __forceinline__ void set(int i) const { if (use_sm) sm[i - r0] = 1; else gl[i] = 1; }
};
__device__ __forceinline__ void mark_neighbours(const PickedRef& picked, const unsigned char* gapbig, int ind, unsigned ln) {
  // lanes 0..4: l = 1..5 forward, gap between ind+l-1 and ind+l ; lanes 8..12: l = -1..-5, gap between ind+l and ind+l+1
  bool brk = false;
  int tgt = -1;
  if (ln < 5) { int l = (int)ln + 1; brk = gapbig[ind + l - 1] != 0; tgt = ind + l; }
  else if (ln >= 8 && ln < 13) { int l = -((int)ln - 8) - 1; brk = gapbig[ind + l] != 0; tgt = ind + l; }
  const unsigned b = __ballot_sync(0xffffffffu, brk);
  const unsigned bf = b & 0x1fu, bb = (b >> 8) & 0x1fu;
  const int stopf = bf ? (__ffs(bf) - 1) : 5, stopb = bb ? (__ffs(bb) - 1) : 5;
  if (ln < 5 && (int)ln < stopf) picked.set(tgt);
  if (ln >= 8 && ln < 13 && (int)(ln - 8) < stopb) picked.set(tgt);
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// Fast path of k_sector_pick: rings of at most LVO_PICK_RING_SMEM points whose sectors hold at most 512 points (every ring of a
// 16/32/64-beam sweep at 10 Hz).  Differences to the generic kernel below, same results bit for bit:
//   * sorts run in REGISTERS: 16 keys per thread, a warp owns 512 keys (one sector), compare-exchanges between a thread's own
//     registers for strides < 16, warp shuffles for strides 16..256, shared memory only for strides >= 512 (the ring-wide sort of
//     the voxel filter, up to 4096 keys over 8 warps).  No block barrier inside a sector sort;
//   * the six sector sorts run concurrently (one warp each);
//   * the sequential greedy picks read (curvature, index) keys, picked flags, gap flags and labels from shared memory, so one
//     pick costs a few shared-memory round trips instead of a chain of dependent global loads.
#define LVO_SECSORT_THREADS (32 * LVO_SECTORS)   // k_sector_sort: one warp per sector
#define LVO_PICKW_THREADS 128                    // k_sector_pick_warp: four rings per CTA
#define LVO_PICKF_SEC_STRIDE 544                 // 512 keys + 1 pad slot per 16 (bank-conflict-free for the 16-per-thread layout)
#define LVO_PICKF_KEYS (4096 + 256)              // padded capacity of the block-wide sort (34 KB)
__device__ __forceinline__ int pad16(int e) { return e + (e >> 4); }
__device__ __forceinline__ void ce64(unsigned long long& a, unsigned long long& b, bool up) {
  const bool sw = (a > b) == up;
  const unsigned long long x = sw ? b : a, y = sw ? a : b;
  a = x; b = y;
}
// Ascending bitonic sort of npad (power of two, <= 4096) keys; element e = warp * 512 + lane * 16 + r lives in k[r] of that
// thread.  npad <= 512: warp-local, no barrier (warps may call it independently).  npad > 512: every thread of the block must
// call it with the same npad; xbuf is the padded exchange buffer (LVO_PICKF_KEYS keys).
template <bool WARP_LOCAL>
__device__ __forceinline__ void bitonic_regs16(unsigned long long (&k)[16], int npad, unsigned long long* xbuf) {
  const unsigned ln = threadIdx.x & 31, w = WARP_LOCAL ? 0u : (threadIdx.x >> 5);   // warp-local sorts are all ascending
  const int ebase = (int)((w << 9) | (ln << 4));
  // warps that hold only padding keep the barriers and skip the work.  The test is per WARP: a warp that holds any key below npad runs
  // the network with all 32 lanes (the full-mask shuffles below need every lane; lanes past npad hold ~0ull padding and only ever
  // exchange with each other, npad being a power of two) — a per-thread test deadlocks the shuffles when npad < 512 (sparse rings).
  const bool active = WARP_LOCAL || (int)(w << 9) < npad;
  // K = 2, 4, 8: direction depends on the register index only
#pragma unroll
  for (int K = 2; K <= 8; K <<= 1) {
    if (K > npad) return;
    if (active) {
#pragma unroll
      for (int J = K >> 1; J > 0; J >>= 1)
#pragma unroll
        for (int r = 0; r < 16; ++r)
          if ((r & J) == 0) ce64(k[r], k[r | J], (r & K) == 0);
    }
  }
  for (int K = 16; K <= npad; K <<= 1) {
    const bool up = (ebase & K) == 0;
    for (int J = K >> 1; J >= 512; J >>= 1) {      // partner in another warp: through shared memory
      if (active) {
#pragma unroll
        for (int r = 0; r < 16; ++r) xbuf[pad16(ebase + r)] = k[r];
      }
      __syncthreads();
      if (active) {
        const bool keep_min = ((ebase & J) == 0) == up;
        const int pb = ebase ^ J;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          const unsigned long long o = xbuf[pad16(pb + r)];
          k[r] = keep_min ? (o < k[r] ? o : k[r]) : (o > k[r] ? o : k[r]);
        }
      }
      __syncthreads();
    }
    if (!active) continue;
    for (int J = min(K >> 1, 256); J >= 16; J >>= 1) {   // partner in another lane
      const int lj = J >> 4;
      const bool keep_min = ((ln & lj) == 0) == up;
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, k[r], lj);
        k[r] = keep_min ? (o < k[r] ? o : k[r]) : (o > k[r] ? o : k[r]);
      }
    }
#pragma unroll
    for (int J = 8; J > 0; J >>= 1)                       // partner in this thread
#pragma unroll
      for (int r = 0; r < 16; ++r)
        if ((r & J) == 0) ce64(k[r], k[r | J], up);
  }
}

// ---- fast path, kernel 1 of 3: the six sector sorts of one ring, one warp each, in registers (:288) -------------------------
// Decides whether the ring takes the fast path (ring_done) and zeroes the ring's counters for either path.
__global__ void __launch_bounds__(LVO_SECSORT_THREADS, 4) k_sector_sort(ExtractArgs a) {
  __shared__ unsigned long long stage[LVO_SECTORS][LVO_PICKF_SEC_STRIDE];   // per-warp transpose buffer for coalesced stores
  const int lane = blockIdx.y, ring = blockIdx.x;
  const LaneState& s = a.ls[lane];
  const size_t lo = (size_t)lane * a.P;
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int sbase = (lane * LVO_MAX_RINGS + ring) * LVO_SECTORS;
  const int S = s.scan_start[ring], E = s.scan_end[ring];
  const int ns = a.lcfg[lane].n_scans;
  // a ring at or above the lane's n_scans holds no point and the lane's steps never write its scan_start / scan_end: no kernel of the
  // ring runs (k_sector_pick_warp, k_lessflat_voxel and k_sector_pick return for it too)
  if (!lane_active(a.lane_flags, lane) || ring >= ns) return;
  if (threadIdx.x == 0) a.lf_cnt[lane * LVO_MAX_RINGS + ring] = 0;
  if (threadIdx.x < LVO_SECTORS * 3) a.slot_cnt[sbase * 3 + threadIdx.x] = 0;
  const int RL = (E + 6) - (S - 5) + 1;          // the ring occupies [S - 5, E + 6]
  const int mmax = (E - S + 5) / 6 + 1;
  const bool mine = E - S < 6 || (RL <= LVO_PICK_RING_SMEM && mmax <= 512);
  if (threadIdx.x == 0) a.ring_done[lane * LVO_MAX_RINGS + ring] = mine ? 1 : 0;
  if (!mine || E - S < 6) return;                // :279-280, or left to the generic kernel
  const float* curv = a.curv + lo;
  const int sp = S + (E - S) * (int)w / 6, ep = S + (E - S) * ((int)w + 1) / 6 - 1;   // :284-285
  const int m = ep - sp + 1;
  unsigned long long k[16];
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int u = (int)ln * 16 + r;
    k[r] = u < m ? (((unsigned long long)__float_as_uint(curv[sp + u]) << 32) | (unsigned)(sp + u)) : ~0ull;  // curvature >= 0: bit order == value order
  }
  bitonic_regs16<true>(k, 512, nullptr);
#pragma unroll
  for (int r = 0; r < 16; ++r) stage[w][pad16((int)ln * 16 + r)] = k[r];
  __syncwarp();
  unsigned long long* keys = a.sort_scratch + (size_t)lane * 2 * a.P;   // sorted (curvature, index) keys at the positions of cloudSortInd
  for (int u = (int)ln; u < m; u += 32) {
    const unsigned long long v = stage[w][pad16(u)];
    keys[sp + u] = v;
    a.sort_ind[lo + sp + u] = (int)(unsigned)(v & 0xffffffffull);         // cloudSortInd (parity probe)
  }
}

// ---- fast path, kernel 2 of 3: the greedy picks of :291-390, ONE WARP per ring ----------------------------------------------------
// The picks of a ring are sequential by definition (every pick suppresses its neighbours, :317-342); the parallelism is across
// rings and lanes.  cloudNeighborPicked and the gap flags of the ring live in shared memory as bit masks (1 KB per warp), 32
// candidates are examined per step, and no block barrier is involved, so an SM keeps up to 48 rings in flight.
__device__ __forceinline__ void bits_set_range(volatile unsigned* bits, int lo_i, int hi_i) {   // set bits lo_i..hi_i (inclusive, at most 5)
  if (hi_i < lo_i) return;
  const int w0 = lo_i >> 5, w1 = hi_i >> 5;
  const unsigned m_lo = 0xffffffffu << (lo_i & 31), m_hi = 0xffffffffu >> (31 - (hi_i & 31));
  if (w0 == w1) bits[w0] |= (m_lo & m_hi);
  else { bits[w0] |= m_lo; bits[w1] |= m_hi; }
}
__global__ void __launch_bounds__(LVO_PICKW_THREADS) k_sector_pick_warp(ExtractArgs a) {
  __shared__ unsigned s_bits[LVO_PICKW_THREADS / 32][2][LVO_PICK_RING_SMEM / 32 + 1];   // [warp][picked | gap][word] (+1: the 10-bit gap window reads two words)
  const int lane = blockIdx.y;
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int ring = blockIdx.x * (LVO_PICKW_THREADS / 32) + (int)w;
  const LaneState& s = a.ls[lane];
  const int S = s.scan_start[ring], E = s.scan_end[ring];   // ring < LVO_MAX_RINGS: the grid covers at most the context's n_scans
  const bool active = lane_active(a.lane_flags, lane);
  if (!active || ring >= a.lcfg[lane].n_scans || E - S < 6 || !a.ring_done[lane * LVO_MAX_RINGS + ring]) return;
  const size_t lo = (size_t)lane * a.P;
  const int sbase = (lane * LVO_MAX_RINGS + ring) * LVO_SECTORS;
  const int R0 = S - 5, RL = (E + 6) - R0 + 1;
  volatile unsigned* pk = s_bits[w][0];
  unsigned* gap = s_bits[w][1];
  for (int base = 0; base < RL; base += 32) {
    const int t = base + (int)ln;
    const unsigned g = __ballot_sync(0xffffffffu, t < RL && a.gapbig[lo + R0 + t] != 0);
    if (ln == 0) { gap[base >> 5] = g; pk[base >> 5] = 0u; }
  }
  __syncwarp();
  const unsigned long long* keys = a.sort_scratch + (size_t)lane * 2 * a.P;
  int* label = a.label + lo;
  // marks of :319-342 / :365-388 around `ind` (relative index i = ind - R0): forward l = 1..5 until the gap between ind+l-1 and
  // ind+l is big, backward l = -1..-5 until the gap between ind+l and ind+l+1 is big.  Executed by lane 0.
  auto mark = [&](int i) {
    // bits i-5 .. i+4 of the gap mask -> 10-bit window (bit 5 + x <-> gap[i + x])
    const int b0 = i - 5;
    const unsigned long long two = ((unsigned long long)gap[(b0 >> 5) + 1] << 32) | gap[b0 >> 5];
    const unsigned win = (unsigned)(two >> (b0 & 31)) & 0x3ffu;
    const unsigned fw = win >> 5;                    // bit x: gap[i + x], x = 0..4  (gap between i+x and i+x+1)
    const unsigned bw = __brev(win & 0x1fu) >> 27;   // bit x: gap[i - 1 - x], x = 0..4
    const int stopf = fw ? (__ffs(fw) - 1) : 5, stopb = bw ? (__ffs(bw) - 1) : 5;
    bits_set_range(pk, i + 1, i + stopf);
    bits_set_range(pk, i - stopb, i - 1);
  };
  for (int j = 0; j < LVO_SECTORS; ++j) {
    const int sp = S + (E - S) * j / 6;            // :284
    const int ep = S + (E - S) * (j + 1) / 6 - 1;  // :285
    int nsharp = 0, nls = 0, largest = 0;
    int pos = ep;
    while (pos >= sp) {  // :292-344, k = ep .. sp
      const int k = pos - (int)ln;
      const bool valid = k >= sp;
      const unsigned long long key = valid ? __ldg(keys + k) : 0ull;
      const int ind = (int)(unsigned)(key & 0xffffffffull);
      const float c = __uint_as_float((unsigned)(key >> 32));
      const bool big = valid && ((double)c > 0.1);
      const bool ok = big && ((pk[(ind - R0) >> 5] >> ((ind - R0) & 31)) & 1u) == 0;
      const unsigned bo = __ballot_sync(0xffffffffu, ok);
      if (bo == 0) {
        if (__ballot_sync(0xffffffffu, valid && !big)) break;  // sorted: nothing further can exceed 0.1
        pos -= 32;
        continue;
      }
      const int first = __ffs(bo) - 1;
      const int sel = __shfl_sync(0xffffffffu, ind, first);
      largest++;
      if (largest <= 2) {
        if (ln == 0) { label[sel] = 2; a.slot_sharp[sbase * 2 + j * 2 + nsharp] = sel; a.slot_lsharp[sbase * 20 + j * 20 + nls] = sel; }
        nsharp++; nls++;
      } else if (largest <= 20) {
        if (ln == 0) { label[sel] = 1; a.slot_lsharp[sbase * 20 + j * 20 + nls] = sel; }
        nls++;
      } else {
        break;
      }
      if (ln == 0) { bits_set_range(pk, sel - R0, sel - R0); mark(sel - R0); }
      __syncwarp();
      pos = pos - first - 1;
    }
    int nflat = 0;
    pos = sp;
    while (pos <= ep) {  // :347-390, k = sp .. ep
      const int k = pos + (int)ln;
      const bool valid = k <= ep;
      const unsigned long long key = valid ? __ldg(keys + k) : 0ull;
      const int ind = (int)(unsigned)(key & 0xffffffffull);
      const float c = __uint_as_float((unsigned)(key >> 32));
      const bool small = valid && ((double)c < 0.1);
      const bool ok = small && ((pk[(ind - R0) >> 5] >> ((ind - R0) & 31)) & 1u) == 0;
      const unsigned bo = __ballot_sync(0xffffffffu, ok);
      if (bo == 0) {
        if (__ballot_sync(0xffffffffu, valid && !small)) break;
        pos += 32;
        continue;
      }
      const int first = __ffs(bo) - 1;
      const int sel = __shfl_sync(0xffffffffu, ind, first);
      if (ln == 0) { label[sel] = -1; a.slot_flat[sbase * 4 + j * 4 + nflat] = sel; }
      nflat++;
      if (nflat >= 4) break;  // :359-362 before the marking
      if (ln == 0) { bits_set_range(pk, sel - R0, sel - R0); mark(sel - R0); }
      __syncwarp();
      pos = pos + first + 1;
    }
    if (ln == 0) { a.slot_cnt[(sbase + j) * 3 + 0] = nsharp; a.slot_cnt[(sbase + j) * 3 + 1] = nls; a.slot_cnt[(sbase + j) * 3 + 2] = nflat; }
    __syncwarp();
  }
  for (int t = (int)ln; t < RL; t += 32)   // cloudNeighborPicked (parity probe; zeroed by k_curvature)
    if ((pk[t >> 5] >> (t & 31)) & 1u) a.picked[lo + R0 + t] = 1;
}

// dynamic shared memory of k_lessflat_voxel<NT>: NT * 17 sort keys, NT * 16 voxel ids, NT * 16 offsets, NT * 16 + 2 run heads
#define LVO_LFV_SMEM(NT) ((NT) * 17 * sizeof(unsigned long long) + (NT) * 16 * sizeof(unsigned) + ((NT) * 32 + 2) * sizeof(unsigned short))
// ---- fast path, kernel 3 of 3: :392-398 less-flat candidates (label <= 0, index order) and :401-407 VoxelGrid(0.2) of one ring -----
// NT threads x 16 keys: NT = 128 takes the rings with at most 2048 candidates, NT = 256 those with 2049..4096.
template <int NT>
__global__ void __launch_bounds__(NT, NT == 128 ? 5 : 3) k_lessflat_voxel(ExtractArgs a) {
  extern __shared__ unsigned long long skeys[];  // NT * 17 keys (padded)
  __shared__ float s_red[6][NT / 32];
  __shared__ int s_i[2];
  __shared__ unsigned s_scan[64];
  int ph = 0;   // double-buffer phase of block_flag_rank
  const int lane = blockIdx.y, ring = blockIdx.x;
  const LaneState& s = a.ls[lane];
  const int S = s.scan_start[ring], E = s.scan_end[ring];
  const bool active = lane_active(a.lane_flags, lane);
  const int ns = a.lcfg[lane].n_scans;
  if (!active || ring >= ns || E - S < 6 || !a.ring_done[lane * LVO_MAX_RINGS + ring]) return;
  if (NT == 256 && E - S <= 2048) return;       // candidates come from [S, E - 1]: at most 2048 of them, the other instantiation's ring
  const size_t lo = (size_t)lane * a.P;
  const float4* P = a.full + lo;
  const int* label = a.label + lo;
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int cnt = 0;
  for (int k = S + threadIdx.x; k <= E - 1; k += NT) {
    if (label[k] <= 0) {
      const float4 p = P[k];
      mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
      mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
      cnt++;
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    for (int o = 16; o > 0; o >>= 1) { mn[c] = fminf(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o)); mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o)); }
    if (ln == 0) { s_red[c][w] = mn[c]; s_red[3 + c][w] = mx[c]; }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (threadIdx.x == 0) s_i[0] = 0;
  __syncthreads();
  if (ln == 0) atomicAdd(&s_i[0], cnt);
  __syncthreads();
  const int ncand = s_i[0];
  if (ncand == 0) return;
  if (NT == 128 ? ncand > 2048 : ncand <= 2048) return;   // the other instantiation's ring
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float a0 = s_red[c][0], b0 = s_red[3 + c][0];
    for (int ww = 1; ww < NT / 32; ++ww) { a0 = fminf(a0, s_red[c][ww]); b0 = fmaxf(b0, s_red[3 + c][ww]); }
    mn[c] = a0; mx[c] = b0;
  }
  const float inv = 1.0f / 0.2f;  // inverse_leaf_size_ for setLeafSize(0.2, 0.2, 0.2)
  const long long ddx = (long long)((mx[0] - mn[0]) * inv) + 1, ddy = (long long)((mx[1] - mn[1]) * inv) + 1, ddz = (long long)((mx[2] - mn[2]) * inv) + 1;
  const bool passthrough = (ddx * ddy * ddz) > (long long)INT_MAX;
  const int min_b0 = (int)floorf(mn[0] * inv), min_b1 = (int)floorf(mn[1] * inv), min_b2 = (int)floorf(mn[2] * inv);
  const int max_b0 = (int)floorf(mx[0] * inv), max_b1 = (int)floorf(mx[1] * inv);
  const int div0 = max_b0 - min_b0 + 1, div1 = max_b1 - min_b1 + 1;
  // Candidates in ring order with their voxel idx.  Consecutive returns of a ring mostly fall into the same 0.2 m voxel (3 cm apart at
  // 10 m), so the sort below ranks RUNS of equal idx instead of points: key = (voxel idx, position of the run's first candidate, run
  // length).  Runs of one voxel come out in position order and a run's candidates are consecutive, so walking them visits the voxel's
  // points in original index order — the very sequence a stable sort of all (idx, offset) pairs gives — with a 3-6 times smaller network.
  unsigned* cand_idx = reinterpret_cast<unsigned*>(skeys + NT * 17);          // [NT * 16]
  unsigned short* cand_off = reinterpret_cast<unsigned short*>(cand_idx + NT * 16);   // [NT * 16] offset of the candidate inside the ring
  int carry = 0;
  for (int base = S; base <= E - 1; base += NT) {   // stable compaction of the candidates
    const int k = base + threadIdx.x;
    const bool c = (k <= E - 1) && label[k] <= 0;
    unsigned tot;
    const unsigned ex = block_flag_rank(c, s_scan, ph++, &tot);
    if (c) {
      const float4 p = P[k];
      unsigned idx;
      if (passthrough) idx = (unsigned)(carry + ex);
      else {
        const int ijk0 = (int)(floorf(p.x * inv) - (float)min_b0);
        const int ijk1 = (int)(floorf(p.y * inv) - (float)min_b1);
        const int ijk2 = (int)(floorf(p.z * inv) - (float)min_b2);
        idx = (unsigned)(ijk0 + ijk1 * div0 + ijk2 * div0 * div1);
      }
      cand_idx[carry + (int)ex] = idx;
      cand_off[carry + (int)ex] = (unsigned short)(k - S);
    }
    carry += (int)tot;
  }
  __syncthreads();
  // run heads -> keys (the run length is filled in once the next head is known: head positions first)
  unsigned short* run_pos = cand_off + NT * 16;   // [NT * 16 + 1] positions of the run heads
  carry = 0;
  for (int base = 0; base < ncand; base += NT) {
    const int t = base + threadIdx.x;
    const bool head = t < ncand && (t == 0 || cand_idx[t] != cand_idx[t - 1]);
    unsigned tot;
    const unsigned ex = block_flag_rank(head, s_scan, ph++, &tot);
    if (head) run_pos[carry + (int)ex] = (unsigned short)t;
    carry += (int)tot;
  }
  const int nruns = carry;
  if (threadIdx.x == 0) run_pos[nruns] = (unsigned short)ncand;
  __syncthreads();
  const int npad = next_pow2(nruns);
  {
    unsigned long long k[16];
    const int e0 = (int)threadIdx.x * 16;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      unsigned long long key = ~0ull;
      if (e0 + r < nruns) {
        const unsigned pos = run_pos[e0 + r], len = run_pos[e0 + r + 1] - pos;
        key = ((unsigned long long)cand_idx[pos] << 32) | (pos << 16) | len;
      }
      k[r] = key;
    }
    __syncthreads();
    bitonic_regs16<false>(k, npad, skeys);
#pragma unroll
    for (int r = 0; r < 16; ++r) if (e0 + r < npad) skeys[pad16(e0 + r)] = k[r];
    __syncthreads();
  }
  // one centroid per voxel: its runs in sorted order, each run's candidates in order, accumulated in float (PCL's CentroidPoint)
  float4* out = a.lf_ring + lo + s.ring_start[ring];
  carry = 0;
  for (int base = 0; base < nruns; base += NT) {
    const int t = base + threadIdx.x;
    bool head = false;
    if (t < nruns) head = (t == 0) || ((skeys[pad16(t)] >> 32) != (skeys[pad16(t - 1)] >> 32));
    unsigned tot;
    const unsigned ex = block_flag_rank(head, s_scan, ph++, &tot);
    if (head) {
      const unsigned long long v = skeys[pad16(t)] >> 32;
      float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
      int cnt = 0;
      for (int u = t; u < nruns; ++u) {
        const unsigned long long ku = skeys[pad16(u)];
        if ((ku >> 32) != v) break;
        const int pos = (int)((ku >> 16) & 0xffffull), len = (int)(ku & 0xffffull);
        for (int q = pos; q < pos + len; ++q) {
          const float4 p = P[S + (int)cand_off[q]];
          sx += p.x; sy += p.y; sz += p.z; si += p.w;
        }
        cnt += len;
      }
      const float c = (float)cnt;
      out[carry + ex] = make_float4(sx / c, sy / c, sz / c, si / c);
    }
    carry += (int)tot;
  }
  if (threadIdx.x == 0) a.lf_cnt[lane * LVO_MAX_RINGS + ring] = carry;
}

// Generic kernel: any ring size (block bitonic sorts in shared memory, global scratch for oversize sorts).  Runs after the fast
// kernel and only handles the rings that one left (ring_done == 0).
__global__ void __launch_bounds__(LVO_PICK_THREADS) k_sector_pick(ExtractArgs a) {
  extern __shared__ unsigned long long skeys[];  // LVO_PICK_SMEM_KEYS
  __shared__ float s_red[6][LVO_PICK_THREADS / 32];
  __shared__ int s_i[8];
  __shared__ unsigned s_scan[33];
  __shared__ unsigned char s_picked[LVO_PICK_RING_SMEM];   // cloudNeighborPicked of this ring while the greedy picks run
  const int lane = blockIdx.y, ring = blockIdx.x;
  const bool active = lane_active(a.lane_flags, lane);
  LaneState& s = a.ls[lane];
  const size_t lo = (size_t)lane * a.P;
  const float4* P = a.full + lo;
  const float* curv = a.curv + lo;
  const unsigned char* gapbig = a.gapbig + lo;
  int* sort_ind = a.sort_ind + lo;
  volatile int* picked = a.picked + lo;
  int* label = a.label + lo;
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int sbase = (lane * LVO_MAX_RINGS + ring) * LVO_SECTORS;
  const int S = s.scan_start[ring], E = s.scan_end[ring];
  const int ns = a.lcfg[lane].n_scans;
  if (!active || ring >= ns || a.ring_done[lane * LVO_MAX_RINGS + ring]) return;   // idle lane / empty ring / handled by k_sector_pick_fast
  if (threadIdx.x == 0) a.lf_cnt[lane * LVO_MAX_RINGS + ring] = 0;
  if (threadIdx.x < LVO_SECTORS * 3) a.slot_cnt[sbase * 3 + threadIdx.x] = 0;
  if (E - S < 6) return;  // :279-280
  const int R0 = S - 5, RL = (E + 6) - R0 + 1;   // the ring occupies [S - 5, E + 6]
  const bool sp_ok = RL <= LVO_PICK_RING_SMEM;
  if (sp_ok) for (int t = threadIdx.x; t < RL; t += blockDim.x) s_picked[t] = 0;
  const PickedRef pk{s_picked, picked, R0, sp_ok};

  // ---- :288 sort cloudSortInd[sp..ep] by (curvature, index) ascending.  When six padded sectors fit in shared memory
  // they are sorted together (one block barrier per network step instead of six).
  const int mmax = (E - S + 5) / 6 + 1;
  const int npad_all = next_pow2(mmax);
  const bool joint = LVO_SECTORS * npad_all <= LVO_PICK_SMEM_KEYS;
  if (joint) {
    for (int t = threadIdx.x; t < LVO_SECTORS * npad_all; t += blockDim.x) {
      const int j = t / npad_all, u = t - j * npad_all;
      const int sp = S + (E - S) * j / 6, ep = S + (E - S) * (j + 1) / 6 - 1;
      unsigned long long k = ~0ull;
      if (u <= ep - sp) k = ((unsigned long long)__float_as_uint(curv[sp + u]) << 32) | (unsigned)(sp + u);  // curvature >= 0: bit order == value order
      skeys[t] = k;
    }
    __syncthreads();
    block_bitonic_sort_multi(skeys, LVO_SECTORS, npad_all);
    for (int t = threadIdx.x; t < LVO_SECTORS * npad_all; t += blockDim.x) {
      const int j = t / npad_all, u = t - j * npad_all;
      const int sp = S + (E - S) * j / 6, ep = S + (E - S) * (j + 1) / 6 - 1;
      if (u <= ep - sp) sort_ind[sp + u] = (int)(unsigned)(skeys[t] & 0xffffffffull);
    }
    __syncthreads();
  }
  for (int j = 0; j < LVO_SECTORS; ++j) {
    const int sp = S + (E - S) * j / 6;            // :284
    const int ep = S + (E - S) * (j + 1) / 6 - 1;  // :285
    const int m = ep - sp + 1;
    if (!joint) {
      const int npad = next_pow2(m);
      unsigned long long* keys = (npad <= LVO_PICK_SMEM_KEYS) ? skeys : (a.sort_scratch + (size_t)lane * 2 * a.P + 2 * (size_t)sp);
      for (int t = threadIdx.x; t < npad; t += blockDim.x) {
        unsigned long long k = ~0ull;
        if (t < m) k = ((unsigned long long)__float_as_uint(curv[sp + t]) << 32) | (unsigned)(sp + t);
        keys[t] = k;
      }
      __syncthreads();
      if (npad <= LVO_PICK_SMEM_KEYS) block_bitonic_sort(skeys, npad); else block_bitonic_sort(keys, npad);
      for (int t = threadIdx.x; t < m; t += blockDim.x) sort_ind[sp + t] = (int)(unsigned)(keys[t] & 0xffffffffull);
      __syncthreads();
    }
    // ---- greedy picks, warp 0 (sequential semantics, 32 candidates examined per step)
    if (w == 0) {
      int nsharp = 0, nls = 0, largest = 0;
      int pos = ep;
      while (pos >= sp) {  // :292-344, k = ep .. sp
        const int k = pos - (int)ln;
        const bool valid = k >= sp;
        const int ind = valid ? sort_ind[k] : 0;
        const float c = valid ? curv[ind] : 0.f;
        const bool big = valid && ((double)c > 0.1);
        const bool ok = big && pk.get(ind) == 0;
        const unsigned bo = __ballot_sync(0xffffffffu, ok);
        if (bo == 0) {
          if (__ballot_sync(0xffffffffu, valid && !big)) break;  // sorted: nothing further can exceed 0.1
          pos -= 32;
          continue;
        }
        const int first = __ffs(bo) - 1;
        const int sel = __shfl_sync(0xffffffffu, ind, first);
        largest++;
        if (largest <= 2) {
          if (ln == 0) { label[sel] = 2; a.slot_sharp[sbase * 2 + j * 2 + nsharp] = sel; a.slot_lsharp[sbase * 20 + j * 20 + nls] = sel; }
          nsharp++; nls++;
        } else if (largest <= 20) {
          if (ln == 0) { label[sel] = 1; a.slot_lsharp[sbase * 20 + j * 20 + nls] = sel; }
          nls++;
        } else {
          break;
        }
        if (ln == 0) pk.set(sel);
        __syncwarp();
        mark_neighbours(pk, gapbig, sel, ln);
        pos = pos - first - 1;
      }
      int nflat = 0;
      pos = sp;
      while (pos <= ep) {  // :347-390, k = sp .. ep
        const int k = pos + (int)ln;
        const bool valid = k <= ep;
        const int ind = valid ? sort_ind[k] : 0;
        const float c = valid ? curv[ind] : 0.f;
        const bool small = valid && ((double)c < 0.1);
        const bool ok = small && pk.get(ind) == 0;
        const unsigned bo = __ballot_sync(0xffffffffu, ok);
        if (bo == 0) {
          if (__ballot_sync(0xffffffffu, valid && !small)) break;
          pos += 32;
          continue;
        }
        const int first = __ffs(bo) - 1;
        const int sel = __shfl_sync(0xffffffffu, ind, first);
        if (ln == 0) { label[sel] = -1; a.slot_flat[sbase * 4 + j * 4 + nflat] = sel; }
        nflat++;
        if (nflat >= 4) break;  // :359-362 before the marking
        if (ln == 0) pk.set(sel);
        __syncwarp();
        mark_neighbours(pk, gapbig, sel, ln);
        pos = pos + first + 1;
      }
      if (ln == 0) { a.slot_cnt[(sbase + j) * 3 + 0] = nsharp; a.slot_cnt[(sbase + j) * 3 + 1] = nls; a.slot_cnt[(sbase + j) * 3 + 2] = nflat; }
    }
    __syncthreads();
  }
  __threadfence_block();
  __syncthreads();
  if (sp_ok) for (int t = threadIdx.x; t < RL; t += blockDim.x) if (s_picked[t]) picked[R0 + t] = 1;   // probe array (cloudNeighborPicked)

  // ---- :392-398 less-flat candidates k in [S, E-1] with label <= 0, in index order; then :401-407 VoxelGrid(0.2)
  // pass 1: bounding box of the candidates
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int cnt = 0;
  for (int k = S + threadIdx.x; k <= E - 1; k += blockDim.x) {
    if (label[k] <= 0) {
      float4 p = P[k];
      mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
      mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
      cnt++;
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    for (int o = 16; o > 0; o >>= 1) { mn[c] = fminf(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o)); mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o)); }
    if (ln == 0) { s_red[c][w] = mn[c]; s_red[3 + c][w] = mx[c]; }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  __syncthreads();
  if (threadIdx.x == 0) s_i[0] = 0;
  __syncthreads();
  if (ln == 0) atomicAdd(&s_i[0], cnt);
  __syncthreads();
  const int ncand = s_i[0];
  if (ncand == 0) return;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float a0 = s_red[c][0], b0 = s_red[3 + c][0];
    for (int ww = 1; ww < LVO_PICK_THREADS / 32; ++ww) { a0 = fminf(a0, s_red[c][ww]); b0 = fmaxf(b0, s_red[3 + c][ww]); }
    mn[c] = a0; mx[c] = b0;
  }
  const float inv = 1.0f / 0.2f;  // inverse_leaf_size_ for setLeafSize(0.2, 0.2, 0.2)
  const long long ddx = (long long)((mx[0] - mn[0]) * inv) + 1, ddy = (long long)((mx[1] - mn[1]) * inv) + 1, ddz = (long long)((mx[2] - mn[2]) * inv) + 1;
  const bool passthrough = (ddx * ddy * ddz) > (long long)INT_MAX;
  const int min_b0 = (int)floorf(mn[0] * inv), min_b1 = (int)floorf(mn[1] * inv), min_b2 = (int)floorf(mn[2] * inv);
  const int max_b0 = (int)floorf(mx[0] * inv), max_b1 = (int)floorf(mx[1] * inv);
  const int div0 = max_b0 - min_b0 + 1, div1 = max_b1 - min_b1 + 1;
  // pass 2: keys (voxel idx, candidate rank) — the rank makes the sort stable and addresses the point
  const int npad = next_pow2(ncand);
  unsigned long long* keys = (npad <= LVO_PICK_SMEM_KEYS) ? skeys : (a.sort_scratch + (size_t)lane * 2 * a.P + 2 * (size_t)S);
  // stable compaction of the candidates: block scan over chunks of the ring
  int carry = 0;
  for (int base = S; base <= E - 1; base += blockDim.x) {
    const int k = base + threadIdx.x;
    const bool c = (k <= E - 1) && label[k] <= 0;
    unsigned tot;
    const unsigned ex = block_excl_scan(c ? 1u : 0u, s_scan, &tot);
    if (c) {
      float4 p = P[k];
      unsigned idx;
      if (passthrough) idx = (unsigned)(carry + ex);
      else {
        int ijk0 = (int)(floorf(p.x * inv) - (float)min_b0);
        int ijk1 = (int)(floorf(p.y * inv) - (float)min_b1);
        int ijk2 = (int)(floorf(p.z * inv) - (float)min_b2);
        idx = (unsigned)(ijk0 + ijk1 * div0 + ijk2 * div0 * div1);
      }
      // low word: offset of the point inside the ring (k - S) — ascending with the candidate rank
      keys[carry + ex] = ((unsigned long long)idx << 32) | (unsigned)(k - S);
    }
    carry += (int)tot;
  }
  for (int t = ncand + threadIdx.x; t < npad; t += blockDim.x) keys[t] = ~0ull;
  __syncthreads();
  if (npad <= LVO_PICK_SMEM_KEYS) block_bitonic_sort(skeys, npad); else block_bitonic_sort(keys, npad);
  // pass 3: one centroid per run of equal voxel idx, accumulated in sorted order (float, as PCL's CentroidPoint)
  float4* out = a.lf_ring + lo + s.ring_start[ring];
  carry = 0;
  for (int base = 0; base < ncand; base += blockDim.x) {
    const int t = base + threadIdx.x;
    bool head = false;
    if (t < ncand) head = (t == 0) || ((keys[t] >> 32) != (keys[t - 1] >> 32));
    unsigned tot;
    const unsigned ex = block_excl_scan(head ? 1u : 0u, s_scan, &tot);
    if (head) {
      const unsigned long long v = keys[t] >> 32;
      float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
      int u = t;
      for (; u < ncand && (keys[u] >> 32) == v; ++u) {
        const float4 p = P[S + (int)(unsigned)(keys[u] & 0xffffffffull)];
        sx += p.x; sy += p.y; sz += p.z; si += p.w;
      }
      const float c = (float)(u - t);
      out[carry + ex] = make_float4(sx / c, sy / c, sz / c, si / c);
    }
    carry += (int)tot;
  }
  if (threadIdx.x == 0) a.lf_cnt[lane * LVO_MAX_RINGS + ring] = carry;
}

// Concatenate per-sector picks and per-ring less-flat clouds in reference order.  One block (512 threads) per lane:
// thread k owns sector k (ring k / 6, sector k % 6); three block scans give the output offsets.
__global__ void __launch_bounds__(512) k_feature_compact(ExtractArgs a) {
  __shared__ unsigned sm[33];
  __shared__ int lfo[LVO_MAX_RINGS + 1];
  const int lane = blockIdx.x;
  LaneState& s = a.ls[lane];
  const int ns = a.lcfg[lane].n_scans;
  const int nsec = ns * LVO_SECTORS;
  const int k = threadIdx.x;
  const int r = k / LVO_SECTORS, j = k % LVO_SECTORS;
  const size_t sb = (size_t)(lane * LVO_MAX_RINGS + r) * LVO_SECTORS;
  int c0 = 0, c1 = 0, c2 = 0;
  if (k < nsec) { const int* c = a.slot_cnt + (sb + j) * 3; c0 = c[0]; c1 = c[1]; c2 = c[2]; }
  if (!lane_active(a.lane_flags, lane)) return;
  unsigned t0, t1, t2, tl;
  const unsigned o0 = block_excl_scan((unsigned)c0, sm, &t0);
  const unsigned o1 = block_excl_scan((unsigned)c1, sm, &t1);
  const unsigned o2 = block_excl_scan((unsigned)c2, sm, &t2);
  const int lc = k < ns ? a.lf_cnt[lane * LVO_MAX_RINGS + k] : 0;
  const unsigned ol = block_excl_scan((unsigned)lc, sm, &tl);
  if (k < ns) { lfo[k] = (int)ol; s.lf_ring_off[k] = (int)ol; }
  if (k == 0) {
    lfo[ns] = (int)tl; s.lf_ring_off[ns] = (int)tl;
    s.n_sharp = (int)t0; s.n_less_sharp = (int)t1; s.n_flat = (int)t2; s.n_less_flat = (int)tl;
    s.stats.n_sharp = (int)t0; s.stats.n_less_sharp = (int)t1; s.stats.n_flat = (int)t2; s.stats.n_less_flat = (int)tl;
  }
  __syncthreads();
  const float4* P = a.full + (size_t)lane * a.P;
  if (k < nsec) {
    for (int t = 0; t < c0; ++t) a.sharp[(size_t)lane * a.cap_sharp + o0 + t] = P[a.slot_sharp[sb * 2 + j * 2 + t]];
    for (int t = 0; t < c1; ++t) a.less_sharp[(size_t)lane * a.cap_lsharp + o1 + t] = P[a.slot_lsharp[sb * 20 + j * 20 + t]];
    for (int t = 0; t < c2; ++t) a.flat[(size_t)lane * a.cap_flat + o2 + t] = P[a.slot_flat[sb * 4 + j * 4 + t]];
  }
  // less-flat: warp w copies rings w, w + 16, ...
  const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
  for (int rr = w; rr < ns; rr += 16) {
    const int c = lfo[rr + 1] - lfo[rr];
    const float4* src = a.lf_ring + (size_t)lane * a.P + s.ring_start[rr];
    for (int t = ln; t < c; t += 32) a.less_flat[(size_t)lane * a.P + lfo[rr] + t] = src[t];
  }
}

// once per process and device, before the first launch (dynamic shared memory above 48 KB needs the opt-in)
static inline void lvo_extract_kernel_attributes() {
  cudaFuncSetAttribute(k_lessflat_voxel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LVO_LFV_SMEM(128));
  cudaFuncSetAttribute(k_lessflat_voxel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LVO_LFV_SMEM(256));
}

static inline void lvo_launch_extract(cudaStream_t st, const ExtractArgs& a, int lanes, int max_n_in, long long* launches, LvoStageTimer* tm = nullptr) {
  if (max_n_in < 1) max_n_in = 1;
  dim3 gpts(lvo_div_up(max_n_in, LVO_EX_THREADS), lanes);
  LVO_MARK(tm, LVO_ST_REG_PREPARE, st);
  k_extract_reset<<<lanes, 32, 0, st>>>(a);
  k_classify<<<gpts, LVO_EX_THREADS, 0, st>>>(a);
  k_ring_count<<<gpts, LVO_EX_THREADS, 0, st>>>(a);
  k_ring_offsets<<<lanes, LVO_MAX_RINGS, 0, st>>>(a);
  k_ring_scatter<<<gpts, LVO_EX_THREADS, 0, st>>>(a);
  k_curvature<<<gpts, LVO_EX_THREADS, 0, st>>>(a);
  LVO_MARK(tm, LVO_ST_REG_SORT, st);
  k_sector_sort<<<dim3(a.max_scans, lanes), LVO_SECSORT_THREADS, 0, st>>>(a);
  LVO_MARK(tm, LVO_ST_REG_SEPARATE, st);
  k_sector_pick_warp<<<dim3(lvo_div_up(a.max_scans, LVO_PICKW_THREADS / 32), lanes), LVO_PICKW_THREADS, 0, st>>>(a);
  k_lessflat_voxel<128><<<dim3(a.max_scans, lanes), 128, LVO_LFV_SMEM(128), st>>>(a);
  k_lessflat_voxel<256><<<dim3(a.max_scans, lanes), 256, LVO_LFV_SMEM(256), st>>>(a);
  k_sector_pick<<<dim3(a.max_scans, lanes), LVO_PICK_THREADS, LVO_PICK_SMEM_KEYS * sizeof(unsigned long long), st>>>(a);
  k_feature_compact<<<lanes, 512, 0, st>>>(a);
  if (launches) *launches += 12;
}
