// Multi-scalar multiplication sum_i s_i * P_i over BN254 G1 and G2 -- signed-digit Pippenger on precomputed
// window tables.
//
// Replaces (upstream, not vendored: yarn.lock:408-416, 1132-1135) ffjavascript src/engine_multiexp.js
// (G1.multiExpAffine / G2.multiExpAffine: window size pTSizes[log2 N], one _multiExpChunk task per window and point
// chunk on the worker pool, then Horner by doubling) and wasmcurves build_multiexp.js g1m_multiexpAffine_chunk.
// Inputs follow the same contract: bases are affine, Montgomery-form, (0,0) = infinity (zkey sections 5-9);
// scalars are 32-byte little-endian *plain* integers < r (the witness, or the from-Montgomery h vector).
// The sum is an exact group element, so its affine form is bit-identical to the reference's.
//
// B200 design.  The bases of a proving key never change, and a B200 has 180 GB of HBM, so every base section is
// expanded ONCE (at zkey load) into a window table  T[w][i] = 2^(c w) P_i  (16 x the section: 5.6 GB for the NZCP
// key).  With it  sum_i s_i P_i = sum_{i,w} d_{i,w} T[w][i]  is a single bucket problem: all windows share one set
// of 2^(c-1) buckets, there is no per-window reduction and no Horner pass.  One MSM is a stream-ordered chain:
//   sort (once per scalar vector, shared by A / B1 / B2 / C which all use the witness):
//     1 digits/count   signed c-bit digits (c = 16 at 2^20), histogram over 2^15 buckets in per-SM shared memory
//     2 scan           exclusive prefix sum of the bucket counts
//     3 scatter        (w * n + i) | sign << 31 written into the bucket's slot range
//     4 plan + tasks   bucket offsets of the pair rounds (below); every bucket's remaining list is cut into tasks of <= 64
//                      points, so the 0/1-heavy witness distribution (a quarter of all wires land in bucket "1") still
//                      load-balances
//   run (per base section):
//     5a pair rounds   (large MSMs) up to three batched-affine rounds: each halves every bucket's list with affine
//                      additions that share one inversion per thread (msm_pair.cuh): 6 + 50/K products per addition
//                      instead of 10, for 7/8 of all additions
//     5b accumulate    one thread per task: XYZZ accumulator in registers, 8M+2S mixed adds over what the rounds left
//                      (or, without rounds, over table entries gathered by index, next one prefetched into L1)
//     6 combine        one thread per bucket sums its (<= 16) task partials; buckets with more go through a two-stage
//                      block-wide sum (chunks of 512 partials, then the chunk results)
//     7 reduce         sum_v v * B_v through marginal sums per base-32 digit of the bucket id (two launches, no level tree)
//     8 host           T + sum_k 32^k S_k: ten doublings and four additions
#include <atomic>

#include "common.cuh"
#include "msm_pair.cuh"

#ifndef NZCP_G2_ACC_BLOCKS
#define NZCP_G2_ACC_BLOCKS 3
#endif

namespace nzcp {

#ifndef NZCP_TASK_LEN_MAX
#define NZCP_TASK_LEN_MAX 64
#endif
static constexpr int kTaskLenMax = NZCP_TASK_LEN_MAX;  // entries per accumulate task: 8..64, picked on the device from the entry
static_assert((NZCP_TASK_LEN_MAX & (NZCP_TASK_LEN_MAX - 1)) == 0 && NZCP_TASK_LEN_MAX >= 8, "task length must be a power of two");
static constexpr int kTaskLenMin = 8;      //   count so that the tasks about fill the GPU once (flags[4])
#ifndef NZCP_TARGET_TASKS
#define NZCP_TARGET_TASKS (148 * 640)
#endif
static constexpr int kTargetTasks = NZCP_TARGET_TASKS;  // resident accumulate threads of a B200 (G1: 5 blocks of 128 per SM)
#ifndef NZCP_HEAVY_TASKS
#define NZCP_HEAVY_TASKS 16
#endif
static constexpr int kHeavyTasks = NZCP_HEAVY_TASKS;  // buckets with more tasks than this go to the block-wide combine
static constexpr int kHeavyThreads = 128;
static constexpr int kHeavyChunk = 512;     // task partials per stage-1 block of the heavy combine
static constexpr int kMaxDigits = 4;        // base-32 digits of a bucket id (c <= 20)
static constexpr int kCopiesGlobal = 16;   // global-atomic histogram (c > 16): private copies of every bucket counter
static constexpr int kSmemHistBuckets = 1 << 15;  // shared-memory histogram path: <= 2^15 buckets (128 KB), c <= 16
static constexpr int kSmemHistThreads = 1024;
static constexpr int kScanBlock = 1024;    // elements per block of the multi-block scan

struct DigitParams {
  uint32_t n_copies;  // private copies of every bucket counter (counter index = bucket * n_copies + copy)
  uint32_t n_points;  // scalars in this launch
  uint32_t stride;    // points per window of the table the entries index (>= n_points)
  int c;
  int n_windows;
  uint32_t n_buckets;     // buckets per group = 2^(c-1): the largest digit magnitude
  uint32_t group_stride;  // 0: every window feeds the same bucket set (window-table mode); 2^(c-1): window w owns bucket
                          // group w (table-free mode: entries index the raw bases, the windows are combined at the end)
  uint32_t n_total;       // all buckets = n_buckets * (group_stride ? n_windows : 1)
};

__device__ __forceinline__ uint32_t scalar_bits(const uint32_t* s, int pos, int c) {
  if (pos >= 256) return 0;
  int idx = pos >> 5, sh = pos & 31;
  uint64_t lo = s[idx];
  uint64_t hi = (idx + 1 < 8) ? s[idx + 1] : 0;
  uint64_t v = (lo | (hi << 32)) >> sh;
  return (uint32_t)v & ((1u << c) - 1);
}

// ------------------------------------------------------------------------------------------------ window table
template <class F>
__global__ void __launch_bounds__(128)
msm_table_kernel(const Affine<F>* __restrict__ src, size_t n_src, size_t pad_front, Affine<F>* __restrict__ table,
                 size_t n_points, int c, int n_windows) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_points) return;
  Affine<F> p = i < pad_front ? Affine<F>::inf() : src[i - pad_front];
  table[i] = p;
  for (int w = 1; w < n_windows; w++) {
    if (!p.is_inf()) {
      XYZZ<F> acc = xyzz_dbl_affine(p);
      for (int k = 1; k < c; k++) acc = xyzz_dbl(acc);
      p = xyzz_to_affine(acc);
    }
    table[(size_t)w * n_points + i] = p;
  }
}

// ------------------------------------------------------------------------------------------------ sort
// COUNT pass: histogram.  SCATTER pass: cursors start at the bucket offsets; write the entry list.
template <bool SCATTER>
__global__ void __launch_bounds__(256)
msm_digits_kernel(const Fr* __restrict__ scalars, DigitParams p, uint32_t* __restrict__ counts_or_cursors,
                  uint32_t* __restrict__ entries, uint32_t* __restrict__ flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  // No early exits: every lane of the warp takes part in the __match_any_sync below (inactive ones with zero digits).
  bool valid = i < p.n_points;
  uint32_t s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (valid) {
    const uint4* q = reinterpret_cast<const uint4*>(scalars + i);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    s[0] = a.x; s[1] = a.y; s[2] = a.z; s[3] = a.w;
    s[4] = b.x; s[5] = b.y; s[6] = b.z; s[7] = b.w;
    // scalars must be canonical (< r); anything else is a malformed witness
    bool ge = true;
#pragma unroll
    for (int k = 7; k >= 0; k--) {
      uint32_t m = FrParams::mod(k);
      if (s[k] != m) {
        ge = s[k] > m;
        break;
      }
    }
    if (ge) {
      if (!SCATTER) atomicOr(&flags[1], 1u);
#pragma unroll
      for (int k = 0; k < 8; k++) s[k] = 0;
    }
  }
  // Counter (d-1) * n_copies + copy: a bucket's sub-ranges stay adjacent, so its entries are still one contiguous run.
  // Lanes of a warp that hit the same counter (the 0/1-heavy witness: digit 1 in window 0) are merged into one atomic.
  const uint32_t copy = blockIdx.x % p.n_copies;
  const uint32_t lane = threadIdx.x & 31;
  const unsigned active = 0xffffffffu;
  uint32_t carry = 0;
  for (int w = 0; w < p.n_windows; w++) {
    uint32_t d = scalar_bits(s, w * p.c, p.c) + carry;
    uint32_t neg = 0;
    if (d > p.n_buckets) {
      d = (1u << p.c) - d;
      neg = 1;
      carry = 1;
    } else {
      carry = 0;
    }
    const uint32_t key = d ? d : 0x80000000u + lane;     // zero digits: singleton groups, no atomic
    const unsigned peers = __match_any_sync(active, key);
    const uint32_t leader = __ffs(peers) - 1;
    const uint32_t rank = __popc(peers & ((1u << lane) - 1));
    uint32_t base = 0;
    if (d && lane == leader)
      base = atomicAdd(&counts_or_cursors[(size_t)(d - 1 + (uint32_t)w * p.group_stride) * p.n_copies + copy], (uint32_t)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    if (SCATTER && d) entries[base + rank] = ((uint32_t)w * p.stride + i) | (neg << 31);
  }
  if (!SCATTER && carry) atomicOr(&flags[1], 2u);
}

// Shared-memory histogram variant (<= 2^15 buckets): one block per SM owns a contiguous chunk of the scalars and a
// private 128 KB histogram, so the per-digit atomics never leave the SM.  COUNT writes its column of the
// [bucket][block] counter matrix; after the scan SCATTER reloads that column as its private cursors, so the entries of
// a bucket are ordered by block -- the layout (and the MSM result) is the same as with global atomics.
template <bool SCATTER>
__global__ void __launch_bounds__(kSmemHistThreads, 1)
msm_digits_smem_kernel(const Fr* __restrict__ scalars, DigitParams p, uint32_t* __restrict__ counts_or_offsets,
                       uint32_t* __restrict__ entries, uint32_t* __restrict__ flags) {
  extern __shared__ uint32_t hist[];
  for (uint32_t b = threadIdx.x; b < p.n_total; b += blockDim.x)
    hist[b] = SCATTER ? counts_or_offsets[b * p.n_copies + blockIdx.x] : 0u;
  __syncthreads();
  const uint32_t per_block = ((p.n_points + gridDim.x - 1) / gridDim.x + 31) & ~31u;   // whole warps stay together
  const uint32_t begin = blockIdx.x * per_block;
  const uint32_t end = begin + per_block < p.n_points ? begin + per_block : p.n_points;
  uint32_t bad = 0;
  for (uint32_t i0 = begin; i0 < end; i0 += blockDim.x) {
    const uint32_t i = i0 + threadIdx.x;
    uint32_t s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (i < end) {
      const uint4* q = reinterpret_cast<const uint4*>(scalars + i);
      uint4 a = __ldg(q), b = __ldg(q + 1);
      s[0] = a.x; s[1] = a.y; s[2] = a.z; s[3] = a.w;
      s[4] = b.x; s[5] = b.y; s[6] = b.z; s[7] = b.w;
      bool ge = true;   // canonical (< r)?
#pragma unroll
      for (int k = 7; k >= 0; k--) {
        uint32_t m = FrParams::mod(k);
        if (s[k] != m) {
          ge = s[k] > m;
          break;
        }
      }
      if (ge) {
        bad |= 1u;
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = 0;
      }
    }
    uint32_t carry = 0;
    for (int w = 0; w < p.n_windows; w++) {
      uint32_t d = scalar_bits(s, w * p.c, p.c) + carry;
      uint32_t neg = 0;
      if (d > p.n_buckets) {
        d = (1u << p.c) - d;
        neg = 1;
        carry = 1;
      } else {
        carry = 0;
      }
      if (d) {   // shared-memory atomics: same-address lanes (the witness's digit 1) serialise on the SM, cheaply
        const uint32_t pos = atomicAdd(&hist[d - 1 + (uint32_t)w * p.group_stride], 1u);
        if (SCATTER) entries[pos] = ((uint32_t)w * p.stride + i) | (neg << 31);
      }
    }
    if (carry) bad |= 2u;
  }
  if (!SCATTER) {
    if (bad) atomicOr(&flags[1], bad);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < p.n_total; b += blockDim.x) counts_or_offsets[b * p.n_copies + blockIdx.x] = hist[b];
  }
}

// Multi-block exclusive scan of the n_buckets * n_copies counters (3 launches: block sums, scan of the sums, rescan).
__global__ void __launch_bounds__(256) msm_scan_sums_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ sums, uint32_t n) {
  __shared__ uint32_t sh[8];
  uint32_t base = blockIdx.x * kScanBlock;
  uint32_t acc = 0;
  for (uint32_t i = threadIdx.x; i < kScanBlock; i += 256)
    if (base + i < n) acc += in[base + i];
  for (int off = 16; off >= 1; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int k = 0; k < 8; k++) t += sh[k];
    sums[blockIdx.x] = t;
  }
}

// out/out2[i] = exclusive prefix of in[] (out2 may be null); block_off = exclusive scan of the block sums.
__global__ void __launch_bounds__(256)
msm_scan_apply_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ block_off, uint32_t* __restrict__ out,
                      uint32_t* __restrict__ out2, uint32_t n) {
  __shared__ uint32_t sh[256];
  const uint32_t base = blockIdx.x * kScanBlock + threadIdx.x * 4;
  uint32_t v[4], acc = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    v[k] = base + k < n ? in[base + k] : 0;
    acc += v[k];
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int off = 1; off < 256; off <<= 1) {
    uint32_t t = threadIdx.x >= (uint32_t)off ? sh[threadIdx.x - off] : 0;
    __syncthreads();
    sh[threadIdx.x] += t;
    __syncthreads();
  }
  uint32_t run = block_off[blockIdx.x] + (threadIdx.x ? sh[threadIdx.x - 1] : 0);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (base + k < n) {
      out[base + k] = run;
      if (out2) out2[base + k] = run;
    }
    run += v[k];
  }
}

// Single-block exclusive scan: out[i] = sum_{j<i} f(in[j]), out[n] = total.  f = identity or ceil(x / task_len).
// TASKS mode first picks the task length from the entry total in flags[3] and publishes it in flags[4].
// Chunks of 4096 values: coalesced loads (four consecutive values per thread), warp-shuffle scans, one carry between
// chunks -- this kernel sits alone on the latency path of every sort (2^15 buckets = 8 chunks).
template <bool TASKS>
__global__ void __launch_bounds__(1024)
msm_scan_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, uint32_t* __restrict__ total,
                uint32_t* __restrict__ flags) {
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t chunk_total;
  uint32_t tl = kTaskLenMax;
  if (TASKS) {
    uint32_t per_thread = flags[5] / kTargetTasks;   // points left after the pair rounds
    while (tl > (uint32_t)kTaskLenMin && tl > per_thread) tl >>= 1;
    if (threadIdx.x == 0) flags[4] = tl;
  }
  const uint32_t tsh = 31 - __clz(tl);   // task lengths are powers of two: ceil(v / tl) without the integer division
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t carry = 0;
  for (uint32_t base = 0; base < n; base += 4096) {
    const uint32_t i0 = base + threadIdx.x * 4;
    uint32_t v[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint32_t x = i0 + k < n ? in[i0 + k] : 0u;
      v[k] = TASKS ? (x + tl - 1) >> tsh : x;
      s += v[k];
    }
    uint32_t incl = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= (uint32_t)d) incl += y;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const uint32_t w = wsum[lane];
      uint32_t z = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, z, d);
        if (lane >= (uint32_t)d) z += y;
      }
      wsum[lane] = z - w;
      if (lane == 31) chunk_total = z;
    }
    __syncthreads();
    uint32_t run = carry + wsum[warp] + (incl - s);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (i0 + k < n) out[i0 + k] = run;
      run += v[k];
    }
    carry += chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[n] = carry;
    if (total) *total = carry;
  }
}

// Round plan (one block; it sits where the per-bucket count kernel used to): from the scanned sub-counters take every
// bucket's entry count len_0, derive len_r = ceil(len_{r-1} / 2) for the R pair rounds, and write the R + 1 exclusive
// prefix sums round_off[r][b] (round_off[r][n_buckets] = points in round r) plus red_count[b] = len_R.
// Chunks of 4096 buckets, four per thread, warp-shuffle scans of all R + 1 channels at once.
template <int R>
__global__ void __launch_bounds__(1024)
msm_round_plan_kernel(const uint32_t* __restrict__ offsets, uint32_t n_copies, uint32_t n_buckets,
                      uint32_t* __restrict__ round_off, uint32_t* __restrict__ red_count, uint32_t* __restrict__ flags) {
  constexpr int C = R + 1;
  __shared__ uint32_t wsum[C][32];
  __shared__ uint32_t chunk_total[C];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t pitch = n_buckets + 1;
  uint32_t carry[C];
#pragma unroll
  for (int r = 0; r < C; r++) carry[r] = 0;
  for (uint32_t base = 0; base < n_buckets; base += 4096) {
    const uint32_t b0 = base + threadIdx.x * 4;
    uint32_t v[C][4], sum[C], incl[C];
#pragma unroll
    for (int r = 0; r < C; r++) sum[r] = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t b = b0 + k;
      uint32_t len = b < n_buckets ? offsets[(size_t)(b + 1) * n_copies] - offsets[(size_t)b * n_copies] : 0u;
#pragma unroll
      for (int r = 0; r < C; r++) {
        v[r][k] = len;
        sum[r] += len;
        len = (len + 1) >> 1;
      }
      if (b < n_buckets) red_count[b] = v[R][k];
    }
#pragma unroll
    for (int r = 0; r < C; r++) {
      incl[r] = sum[r];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl[r], d);
        if (lane >= (uint32_t)d) incl[r] += y;
      }
      if (lane == 31) wsum[r][warp] = incl[r];
    }
    __syncthreads();
    if (warp < (uint32_t)C) {
      const uint32_t w = wsum[warp][lane];
      uint32_t z = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, z, d);
        if (lane >= (uint32_t)d) z += y;
      }
      wsum[warp][lane] = z - w;
      if (lane == 31) chunk_total[warp] = z;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < C; r++) {
      uint32_t run = carry[r] + wsum[r][warp] + (incl[r] - sum[r]);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (b0 + k < n_buckets) round_off[(size_t)r * pitch + b0 + k] = run;
        run += v[r][k];
      }
      carry[r] += chunk_total[r];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int r = 0; r < C; r++) round_off[(size_t)r * pitch + n_buckets] = carry[r];
    flags[5] = carry[R];
  }
}

// One thread per task: find its bucket by binary search in task_off, then (first entry, length).
__global__ void __launch_bounds__(256)
msm_task_fill_kernel(const uint32_t* __restrict__ bcount, const uint32_t* __restrict__ offsets,
                     const uint32_t* __restrict__ task_off, uint2* __restrict__ tasks, uint32_t n_buckets,
                     const uint32_t* __restrict__ flags) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= flags[2]) return;
  const uint32_t tl = flags[4];
  uint32_t lo = 0, hi = n_buckets;  // task_off[lo] <= t < task_off[hi]
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (task_off[mid] <= t) lo = mid; else hi = mid;
  }
  // balanced split: the bucket's k = ceil(count / tl) tasks get count / k entries each (+1 for the first count % k), so
  // the lanes of a warp finish together instead of waiting for full-length neighbours of a short remainder task
  (void)tl;
  const uint32_t k = task_off[lo + 1] - task_off[lo], j = t - task_off[lo];
  const uint32_t cnt = bcount[lo], base = cnt / k, rem = cnt % k;
  tasks[t] = make_uint2(offsets[lo] + j * base + (j < rem ? j : rem), base + (j < rem ? 1u : 0u));
}

// ------------------------------------------------------------------------------------------------ run
template <class T>
__device__ __forceinline__ void prefetch_l1(const T* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
  if (sizeof(T) > 64) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(p) + 64));
}

template <class F> struct AccumOcc { static constexpr int kBlocks = 5; };   // G1: <= 102 registers
template <> struct AccumOcc<Fq2> { static constexpr int kBlocks = NZCP_G2_ACC_BLOCKS; };

// DRAM traffic (ncu): 128 bytes per 64-byte G1 point, 1.05 x 128 bytes per G2 point -- random reads cost a full 128-byte
// line on this part.  Tried and measured without effect on bytes or time: staging the point with 16-byte cp.async
// (LDGSTS.BYPASS) instead of the L1 prefetch, and cudaLimitMaxL2FetchGranularity = 32 / 64 (DESIGN.md section 5).
template <class F>
__global__ void __launch_bounds__(128, AccumOcc<F>::kBlocks)
msm_accumulate_kernel(const Affine<F>* __restrict__ table, const uint32_t* __restrict__ entries,
                      const uint2* __restrict__ tasks, const uint32_t* __restrict__ flags, XYZZ<F>* __restrict__ partial, int pf) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= flags[2]) return;
  uint2 tk = tasks[t];
  XYZZ<F> acc = XYZZ<F>::inf();
  uint32_t e = entries[tk.x];
  if (pf & 1) prefetch_l1(table + (e & 0x7fffffffu));
  for (uint32_t k = 0; k < tk.y; k++) {
    uint32_t en = e;
    if (k + 1 < tk.y) {
      en = entries[tk.x + k + 1];
      if (pf & 1) prefetch_l1(table + (en & 0x7fffffffu));
    }
    Affine<F> q;
#if defined(__CUDA_ARCH__)
    if (sizeof(F) == sizeof(Fq) && (pf & 4)) q = gather_hinted<Affine<F>>(table + (e & 0x7fffffffu));   // "gather_hint": see msm_pair.cuh
    else
#endif
      q = table[e & 0x7fffffffu];
    if (!q.is_inf()) xyzz_madd(acc, q, (e >> 31) != 0);
    e = en;
  }
  partial[t] = acc;
}

// The same accumulation over what the pair rounds left: the task's points are contiguous in the last round's array.
template <class F>
__global__ void __launch_bounds__(128, AccumOcc<F>::kBlocks)
msm_accumulate_pts_kernel(const Affine<F>* __restrict__ pts, const uint2* __restrict__ tasks,
                          const uint32_t* __restrict__ flags, XYZZ<F>* __restrict__ partial) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= flags[2]) return;
  uint2 tk = tasks[t];
  XYZZ<F> acc = XYZZ<F>::inf();
  for (uint32_t k = 0; k < tk.y; k++) {
    Affine<F> q = pts[tk.x + k];
    if (!q.is_inf()) xyzz_madd(acc, q, false);
  }
  partial[t] = acc;
}

// One pair round (msm_pair.cuh) = forward, invert, backward; thread t of forward / backward owns K consecutive points of
// the round, thread g of invert owns 32 consecutive thread products.
static constexpr int kPairInvGroup = 32;
#ifndef NZCP_PAIR_FWD_BLOCKS
#define NZCP_PAIR_FWD_BLOCKS 1
#endif
template <class F, bool FROM_TABLE, int K>
__global__ void __launch_bounds__(128, (sizeof(F) == sizeof(Fq) ? NZCP_PAIR_FWD_BLOCKS : 1))
msm_pair_forward_kernel(const Affine<F>* __restrict__ src, const uint32_t* __restrict__ entries,
                        const uint32_t* __restrict__ off_in, const uint32_t* __restrict__ off_out, uint32_t n_buckets,
                        F* __restrict__ scratch, F* __restrict__ prod, int pf, Affine<F>* __restrict__ ops) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  PairSource<F, FROM_TABLE> ps{src, entries, pf};
  msm_pair_forward_body<F, FROM_TABLE, K>(t, gridDim.x * blockDim.x, ps, off_in, off_out, n_buckets, scratch, prod, ops);
}

template <class F, int K>
__global__ void __launch_bounds__(64)
msm_pair_invert_kernel(F* __restrict__ prod, const uint32_t* __restrict__ off_out, uint32_t n_buckets) {
  const uint32_t n_out = off_out[n_buckets];
  const uint32_t n_prod = pair_n_prod<K>(n_out);    // threads of the forward kernel that had work
  msm_pair_invert_body<F, kPairInvGroup>(blockIdx.x * blockDim.x + threadIdx.x, prod, n_prod);
}

template <class F, bool FROM_TABLE, int K>
__global__ void __launch_bounds__(128)
msm_pair_backward_kernel(const Affine<F>* __restrict__ src, const uint32_t* __restrict__ entries,
                         const uint32_t* __restrict__ off_in, const uint32_t* __restrict__ off_out, uint32_t n_buckets,
                         Affine<F>* __restrict__ dst, const F* __restrict__ scratch, const F* __restrict__ inv_prod, int pf,
                         const Affine<F>* __restrict__ ops) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  PairSource<F, FROM_TABLE> ps{src, entries, pf};
  msm_pair_backward_body<F, FROM_TABLE, K>(t, gridDim.x * blockDim.x, ps, off_in, off_out, n_buckets, dst, scratch, inv_prod,
                                           ops);
}

// L2-coherent load of an object another block of the same grid wrote (after its __threadfence + counter increment).
template <class T>
__device__ __forceinline__ T load_cg(const T* p) {
  static_assert(sizeof(T) % 16 == 0, "16-byte granules");
  T r;
  const uint4* s = reinterpret_cast<const uint4*>(p);
  uint4* d = reinterpret_cast<uint4*>(&r);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = __ldcg(s + i);
  return r;
}

template <class T>
__device__ __forceinline__ T shfl_down_obj(const T& v, unsigned delta) {
  T r;
  const uint32_t* s = reinterpret_cast<const uint32_t*>(&v);
  uint32_t* d = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) d[i] = __shfl_down_sync(0xffffffffu, s[i], delta);
  return r;
}

// One thread per bucket sums the bucket's (few) task partials; buckets with many tasks go to the block-wide kernel.
template <class F>
__global__ void __launch_bounds__(128)
msm_combine_kernel(const uint32_t* __restrict__ task_off, const XYZZ<F>* __restrict__ partial,
                   XYZZ<F>* __restrict__ buckets, uint32_t n_buckets, uint32_t* __restrict__ heavy_list,
                   uint32_t* __restrict__ heavy_count) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_buckets) return;
  const uint32_t t0 = task_off[b], nt = task_off[b + 1] - t0;
  if (nt > (uint32_t)kHeavyTasks) {
    heavy_list[atomicAdd(heavy_count, 1u)] = b;
    return;
  }
  XYZZ<F> acc = XYZZ<F>::inf();
  for (uint32_t j = 0; j < nt; j++) xyzz_add(acc, partial[t0 + j]);
  buckets[b] = acc;
}

// Heavy buckets (more than kHeavyTasks task partials; the witness's bucket "1" has ~15 000) are summed in two stages
// so that no single block walks a long dependent chain: stage 1 reduces chunks of kHeavyChunk partials (one block per
// chunk, all chunks of all heavy buckets in one grid), stage 2 sums each bucket's chunk results.
// chunk_off[h] = exclusive prefix of ceil(tasks(heavy bucket h) / kHeavyChunk), h <= n_heavy.  One block; the heavy
// list is short (a few hundred buckets for the witness, none for dense scalars).
__global__ void __launch_bounds__(1024)
msm_heavy_scan_kernel(const uint32_t* __restrict__ task_off, const uint32_t* __restrict__ heavy_list,
                      uint32_t* __restrict__ heavy_count, uint32_t* __restrict__ chunk_off) {
  __shared__ uint32_t sums[1024];
  const uint32_t n = heavy_count[0];
  const uint32_t per = (n + 1023) / 1024;
  const uint32_t b = threadIdx.x * per;
  const uint32_t e = b + per < n ? b + per : n;
  auto chunks = [&](uint32_t h) {
    uint32_t bk = heavy_list[h];
    return (task_off[bk + 1] - task_off[bk] + kHeavyChunk - 1) / kHeavyChunk;
  };
  uint32_t acc = 0;
  for (uint32_t h = b; h < e; h++) acc += chunks(h);
  sums[threadIdx.x] = acc;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    uint32_t v = threadIdx.x >= (uint32_t)off ? sums[threadIdx.x - off] : 0;
    __syncthreads();
    sums[threadIdx.x] += v;
    __syncthreads();
  }
  uint32_t run = threadIdx.x ? sums[threadIdx.x - 1] : 0;
  for (uint32_t h = b; h < e; h++) {
    chunk_off[h] = run;
    run += chunks(h);
  }
  if (threadIdx.x == 1023) {
    chunk_off[n] = sums[1023];
    heavy_count[1] = sums[1023];
  }
}

template <class F>
__device__ __forceinline__ XYZZ<F> block_sum(XYZZ<F> acc, XYZZ<F>* sm) {
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (uint32_t stride = blockDim.x / 2; stride >= 1; stride >>= 1) {
    if (threadIdx.x < stride) {
      XYZZ<F> a = sm[threadIdx.x];
      xyzz_add(a, sm[threadIdx.x + stride]);
      sm[threadIdx.x] = a;
    }
    __syncthreads();
  }
  XYZZ<F> r = sm[0];
  __syncthreads();
  return r;
}

template <class F>
__global__ void __launch_bounds__(kHeavyThreads)
msm_combine_heavy_kernel(const uint32_t* __restrict__ task_off, const XYZZ<F>* __restrict__ partial,
                         const uint32_t* __restrict__ heavy_list, const uint32_t* __restrict__ heavy_count,
                         const uint32_t* __restrict__ chunk_off, XYZZ<F>* __restrict__ chunk_partial,
                         XYZZ<F>* __restrict__ buckets) {
  extern __shared__ unsigned char heavy_sm_raw[];
  XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(heavy_sm_raw);
  const uint32_t n_heavy = *heavy_count;
  const uint32_t total = chunk_off[n_heavy];
  for (uint32_t ch = blockIdx.x; ch < total; ch += gridDim.x) {
    // heavy bucket h with chunk_off[h] <= ch < chunk_off[h + 1]
    uint32_t lo = 0, hi = n_heavy;
    while (hi - lo > 1) {
      uint32_t mid = (lo + hi) >> 1;
      if (chunk_off[mid] <= ch) lo = mid; else hi = mid;
    }
    const uint32_t b = heavy_list[lo];
    const uint32_t c = ch - chunk_off[lo];
    const uint32_t t0 = task_off[b] + c * kHeavyChunk;
    const uint32_t left = task_off[b + 1] - t0;
    const uint32_t cnt = left < (uint32_t)kHeavyChunk ? left : (uint32_t)kHeavyChunk;
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t j = threadIdx.x; j < cnt; j += blockDim.x) xyzz_add(acc, partial[t0 + j]);
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) {
      if (chunk_off[lo + 1] - chunk_off[lo] == 1) buckets[b] = acc;   // one chunk: this is the bucket's sum
      else chunk_partial[ch] = acc;
    }
  }
}

template <class F>
__global__ void __launch_bounds__(kHeavyThreads)
msm_combine_heavy2_kernel(const uint32_t* __restrict__ heavy_list, const uint32_t* __restrict__ heavy_count,
                          const uint32_t* __restrict__ chunk_off, const XYZZ<F>* __restrict__ chunk_partial,
                          XYZZ<F>* __restrict__ buckets) {
  extern __shared__ unsigned char heavy_sm_raw[];
  XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(heavy_sm_raw);
  const uint32_t n_heavy = *heavy_count;
  for (uint32_t h = blockIdx.x; h < n_heavy; h += gridDim.x) {
    const uint32_t c0 = chunk_off[h], nc = chunk_off[h + 1] - c0;
    if (nc <= 1) continue;                                             // stage 1 already wrote the bucket
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t j = threadIdx.x; j < nc; j += blockDim.x) xyzz_add(acc, chunk_partial[c0 + j]);
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) buckets[heavy_list[h]] = acc;
  }
}

// Bucket reduction  sum_v v * B_v  without a dependent tree of levels.  Write the bucket id v-1 in base 32,
// v-1 = sum_k d_k 32^k.  Then  sum_v (v-1) B_v = sum_k 32^k * sum_j j * M_k[j]  with the marginal sums
// M_k[j] = sum of all buckets whose k-th digit is j.  Stage 1 computes every M_k[j] as an independent block-wide tree
// sum (fully parallel, chain ~ log); stage 2 turns each digit's 32 marginals into sum_j j M_k[j] with one warp
// (suffix scan + tree sum through shuffles); the host finishes with  T + sum_k 32^k S_k  (T = sum of all buckets).
static constexpr int kMargThreads = 128;

// Suffix scan + tree sum of one digit's 32 marginals by one warp: returns sum_j j * M[j] (lane 0), *total = sum_j M[j].
template <class F>
__device__ __forceinline__ XYZZ<F> warp_weighted_sum(XYZZ<F> run, uint32_t lane, XYZZ<F>* total) {
  for (uint32_t d = 1; d < 32; d <<= 1) {
    XYZZ<F> o = shfl_down_obj(run, d);
    if (lane + d < 32) xyzz_add(run, o);
  }
  *total = run;                                                  // lane 0: sum of all 32
  XYZZ<F> leaf = lane >= 1 ? run : XYZZ<F>::inf();              // sum_{j>=1} suffix_j = sum_j j M[j]
  for (uint32_t off = 16; off >= 1; off >>= 1) {
    XYZZ<F> o = shfl_down_obj(leaf, off);
    xyzz_add(leaf, o);
  }
  return leaf;
}

// Grid = n_groups * n_digits * 32 blocks: block (g, k, j) sums the buckets of group g whose k-th base-32 digit is j.  The
// LAST of a digit's 32 blocks to finish (a counter per (g, k), reset by that block for the next launch) also folds the 32
// marginals into S_k = sum_j j M_k[j] with its first warp -- the former second launch (three lone warps, ~115 us on the
// critical path of every MSM) now starts the moment its inputs exist.
// out[g * (n_digits + 1) + k] = S_k of group g, out[g * (n_digits + 1) + n_digits] = T = sum of the group's buckets.
template <class F>
__global__ void __launch_bounds__(kMargThreads)
msm_marginal_kernel(const XYZZ<F>* __restrict__ buckets, XYZZ<F>* __restrict__ marg, XYZZ<F>* __restrict__ out,
                    uint32_t* __restrict__ done, uint32_t bits, uint32_t n_digits) {
  extern __shared__ unsigned char heavy_sm_raw[];
  XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(heavy_sm_raw);
  __shared__ uint32_t is_last;
  const uint32_t gk = blockIdx.x >> 5, j = blockIdx.x & 31;     // (group, digit position), digit value
  const uint32_t g = gk / n_digits, k = gk - g * n_digits;
  const XYZZ<F>* bk = buckets + ((size_t)g << bits);
  const uint32_t lo_bits = 5 * k;
  const uint32_t dig_bits = bits - lo_bits < 5 ? bits - lo_bits : 5;
  XYZZ<F> acc = XYZZ<F>::inf();
  if (j < (1u << dig_bits)) {
    const uint32_t count = 1u << (bits - dig_bits);              // buckets with d_k == j
    const uint32_t lo_mask = (1u << lo_bits) - 1;
    for (uint32_t idx = threadIdx.x; idx < count; idx += blockDim.x) {
      const uint32_t v = (idx & lo_mask) | (j << lo_bits) | ((idx >> lo_bits) << (lo_bits + dig_bits));
      xyzz_add(acc, bk[v]);
    }
  }
  acc = block_sum(acc, sm);
  if (threadIdx.x == 0) {
    marg[blockIdx.x] = acc;
    __threadfence();
    const uint32_t prev = atomicAdd(&done[gk], 1u);
    is_last = prev == 31u;
    if (is_last) done[gk] = 0;                                   // ready for the next launch on this stream
  }
  __syncthreads();
  if (!is_last || threadIdx.x >= 32) return;
  __threadfence();
  const uint32_t lane = threadIdx.x;
  XYZZ<F> total;
  XYZZ<F> leaf = warp_weighted_sum(load_cg(marg + gk * 32 + lane), lane, &total);   // marginals beyond the digit's range are infinity
  if (lane == 0) {
    out[g * (n_digits + 1) + k] = leaf;
    if (k == 0) out[g * (n_digits + 1) + n_digits] = total;
  }
}

// sum_g 2^(c g) * (T_g + sum_k 32^k S_{g,k}) on the device (one warp; lane l folds the groups [l G, (l+1) G) by Horner,
// G = ceil(n_groups / 32), then a shuffle tree applies the 2^(c G off) factors by repeated doubling).  The prover finishes
// on the host instead (a dozen group operations are faster there); this kernel exists for results that must stay in
// HBM: the per-rank partial sums of a split MSM.
template <class F>
__global__ void __launch_bounds__(32)
msm_finish_kernel(const XYZZ<F>* __restrict__ out, XYZZ<F>* __restrict__ result, uint32_t n_groups, uint32_t n_digits, int c) {
  const uint32_t lane = threadIdx.x;
  const uint32_t per = (n_groups + 31) / 32;
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int g = (int)((lane + 1) * per) - 1; g >= (int)(lane * per); g--) {
    if (!acc.is_inf())
      for (int d = 0; d < c; d++) acc = xyzz_dbl(acc);
    if ((uint32_t)g >= n_groups) continue;
    const XYZZ<F>* w = out + (size_t)g * (n_digits + 1);
    XYZZ<F> r = XYZZ<F>::inf();
    for (int k = (int)n_digits - 1; k >= 0; k--) {
      if (!r.is_inf())
        for (int d = 0; d < 5; d++) r = xyzz_dbl(r);
      xyzz_add(r, w[k]);
    }
    xyzz_add(r, w[n_digits]);
    xyzz_add(acc, r);
  }
  // tree: acc[l] += 2^(c * per * off) * acc[l + off]
  for (uint32_t off = 1; off < 32; off <<= 1) {
    XYZZ<F> o = shfl_down_obj(acc, off);
    if ((lane & (2 * off - 1)) == 0 && (lane + off) * per < n_groups && !o.is_inf()) {
      for (uint32_t d = 0; d < (uint32_t)c * per * off; d++) o = xyzz_dbl(o);
      xyzz_add(acc, o);
    }
  }
  if (lane == 0) *result = acc;
}

// result = sum of `count` points (the gathered per-rank partials of a split MSM): one block, tree in shared memory.
template <class F>
__global__ void __launch_bounds__(kHeavyThreads)
msm_sum_points_kernel(const XYZZ<F>* __restrict__ pts, uint32_t count, XYZZ<F>* __restrict__ result) {
  extern __shared__ unsigned char heavy_sm_raw[];
  XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(heavy_sm_raw);
  XYZZ<F> acc = XYZZ<F>::inf();
  for (uint32_t j = threadIdx.x; j < count; j += blockDim.x) xyzz_add(acc, pts[j]);
  acc = block_sum(acc, sm);
  if (threadIdx.x == 0) *result = acc;
}

// ---------------------------------------------------------------------------------------------- host side
int msm_pick_window(size_t n) {
  int lg = 0;
  while (((size_t)2 << lg) <= n) lg++;
  if (lg <= 6) return 4;
  if (lg <= 9) return 6;
  if (lg <= 12) return 8;
  if (lg <= 14) return 10;
  if (lg <= 16) return 12;
  if (lg <= 18) return 14;
  return 16;
}

// Table-free path: every window has its own 2^(c-1) buckets, reduced separately, so the optimum is a little below the
// shared-bucket one.  Cost model in Fq products: W * (10 n + 2^(c-1) * 14 * (digits + 1)), W * 2^(c-1) <= 2^19.
int msm_pick_window_free(size_t n) {
  int best = 2;
  double best_cost = 1e300;
  for (int c = 2; c <= 16; c++) {
    const int w = msm_num_windows(c);
    const double nb = (double)((size_t)1 << (c - 1));
    if (w * nb > (double)(1 << 19)) break;
    const double cost = w * (10.0 * (double)n + nb * 14.0 * ((c - 1 + 4) / 5 + 1));
    if (cost < best_cost) {
      best_cost = cost;
      best = c;
    }
  }
  return best;
}

int msm_num_windows(int c) {
  int w = (254 + c - 1) / c;
  if (w * c < 255) w++;  // one spare bit so the top signed digit never carries out
  return w;
}

// Tuning knobs (nzcp_tuning_set): pair rounds per MSM (-1 = msm_pick_rounds) and additions per thread in round 1, 2, 3.
std::atomic<int> g_tune_rounds{-1};
std::atomic<int> g_tune_rounds_w{-1}, g_tune_rounds_h{-1};   // prover: witness MSMs / H MSM (-1 = default)
std::atomic<int> g_tune_pair_k[kMsmMaxRounds] = {{16}, {16}, {16}};
std::atomic<int> g_tune_pair_prefetch[2] = {{0}, {0}};   // forward / backward pair kernels: 0 none, 1 L1, 2 L2 (msm_pair.cuh)
// "pair_stage" = 1: round 1's forward pass also writes the operands it gathered (coalesced) and the backward pass streams
// them instead of gathering a second time.  Measured on the B200: it LOSES 4 % (126 vs 131 proofs/s,
// profiles/r02_window_rounds_sweep.md) -- the 2 x 1 GB of extra streaming per H MSM and a forward pass that now carries
// whole points through its registers cost more than the second gather saves.  Kept as an opt-in, off by default.
std::atomic<int> g_tune_pair_stage{0};
std::atomic<int> g_tune_sort_threads{1024};
std::atomic<int> g_tune_gather_hint{0};                  // experiment: .L2::64B fetch-size qualifier on the round-1 gathers
std::atomic<int> g_tune_acc_prefetch{1};                 // XYZZ accumulate kernel: prefetch the next table point to L1

// Pair rounds are OFF for the standalone MSMs unless asked for (nzcp_tuning_set "msm_rounds"); provers turn them on
// (msm_pick_rounds_prover; "prover_rounds_*" override).  History of the measurement on the B200 (profiles/r02_pair_rounds.md,
// r02_window_rounds_sweep.md): with the operands of the next pair prefetched to L1 the H accumulation took 3.1 ms with
// rounds against 2.75 ms for the XYZZ kernel (an affine addition needs each operand twice, and round 1 gathers them from
// the 1 GB window table); without that prefetch and with a thread's additions interleaved across its warp it takes
// 2.58 ms, executes a quarter fewer products, and the whole proof gains 11 %.
int msm_pick_rounds(size_t n_points, int c) {
  (void)n_points;
  (void)c;
  const int forced = g_tune_rounds.load();
  if (forced >= 0) return forced > kMsmMaxRounds ? kMsmMaxRounds : forced;
  return 0;
}

// The prover's MSMs: three pair rounds once an MSM has a few million entries -- below that the rounds' nine extra launches
// cost more than the products they save.
int msm_pick_rounds_prover(size_t n_points, int c) {
  const int forced = g_tune_rounds.load();
  if (forced >= 0) return forced > kMsmMaxRounds ? kMsmMaxRounds : forced;
  return n_points * (size_t)msm_num_windows(c) >= ((size_t)1 << 22) ? kMsmMaxRounds : 0;
}

void msm_table_create(MsmTable* t, const void* d_bases, size_t n_src, size_t pad_front, bool g2, int c, cudaStream_t st) {
  *t = MsmTable();
  if (c < 2 || c > 20) throw std::runtime_error("msm: window size out of range");
  t->n_points = n_src + pad_front;
  t->c = c;
  t->n_windows = msm_num_windows(c);
  t->g2 = g2;
  size_t psz = g2 ? sizeof(G2Affine) : sizeof(G1Affine);
  if ((size_t)t->n_windows * t->n_points >= ((size_t)1 << 31)) throw std::runtime_error("msm: too many points");
  t->bytes = (size_t)t->n_windows * (t->n_points ? t->n_points : 1) * psz;
  t->pts = t->res.device<unsigned char>(t->bytes);
  if (t->n_points == 0) return;
  unsigned grid = div_up(t->n_points, 128);
  if (g2)
    msm_table_kernel<Fq2><<<grid, 128, 0, st>>>(reinterpret_cast<const G2Affine*>(d_bases), n_src, pad_front,
                                               reinterpret_cast<G2Affine*>(t->pts), t->n_points, c, t->n_windows);
  else
    msm_table_kernel<Fq><<<grid, 128, 0, st>>>(reinterpret_cast<const G1Affine*>(d_bases), n_src, pad_front,
                                              reinterpret_cast<G1Affine*>(t->pts), t->n_points, c, t->n_windows);
  NZCP_LAUNCH_CHECK();
}

void msm_table_view(MsmTable* t, void* d_bases, size_t n_points, bool g2, int c) {
  *t = MsmTable();
  t->pts = d_bases;
  t->n_points = n_points;
  t->c = c;
  t->n_windows = 1;
  t->g2 = g2;
}

void msm_sort_create(MsmSort* s, size_t n_points, int c, int rounds, bool table_free) {
  *s = MsmSort();
  if (c < 2 || c > 20) throw std::runtime_error("msm: window size out of range");
  s->n_points = n_points;
  s->c = c;
  s->rounds = rounds < 0 ? msm_pick_rounds(n_points, c) : (rounds > kMsmMaxRounds ? kMsmMaxRounds : rounds);
  s->n_windows = msm_num_windows(c);
  s->table_free = table_free;
  s->n_groups = table_free ? s->n_windows : 1;
  s->group_buckets = (size_t)1 << (c - 1);
  s->n_buckets = s->group_buckets * s->n_groups;
  if (s->n_buckets > ((size_t)1 << 19)) throw std::runtime_error("msm: too many buckets (window size too large for the table-free path)");
  size_t max_entries = (size_t)s->n_windows * n_points;
  if (max_entries >= ((size_t)1 << 31)) throw std::runtime_error("msm: too many points");
  // task length L = clamp(pow2_floor(entries / kTargetTasks), 8, 64)  =>  tasks <= n_buckets + max(2 * target, entries / 64)
  size_t by_len = max_entries / kTaskLenMax, by_target = 2 * (size_t)kTargetTasks;
  if (max_entries / kTaskLenMin < by_target) by_target = max_entries / kTaskLenMin;
  s->max_tasks = s->n_buckets + (by_len > by_target ? by_len : by_target) + 1;
  s->smem_hist = s->n_buckets <= (size_t)kSmemHistBuckets;
  s->n_copies = s->smem_hist ? 148 : kCopiesGlobal;
  size_t n_ctr = s->n_buckets * s->n_copies;
  s->counts = s->res.device<uint32_t>(n_ctr + 1);
  s->offsets = s->res.device<uint32_t>(n_ctr + 1);
  s->cursors = s->res.device<uint32_t>(n_ctr + 1);
  s->red_count = s->res.device<uint32_t>(s->n_buckets + 1);
  s->round_off = s->res.device<uint32_t>((size_t)(kMsmMaxRounds + 1) * (s->n_buckets + 1));
  s->round_max[0] = max_entries;
  for (int r = 1; r <= kMsmMaxRounds; r++) s->round_max[r] = (s->round_max[r - 1] + s->n_buckets) / 2 + 1;
  s->block_sums = s->res.device<uint32_t>(2 * (n_ctr / kScanBlock + 2));
  if (s->smem_hist) {  // function attributes are per device: set them whenever a plan is created on the current one
    NZCP_CUDA(cudaFuncSetAttribute(msm_digits_smem_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemHistBuckets * 4));
    NZCP_CUDA(cudaFuncSetAttribute(msm_digits_smem_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemHistBuckets * 4));
  }
  s->entries = s->res.device<uint32_t>(max_entries ? max_entries : 1);
  s->task_off = s->res.device<uint32_t>(s->n_buckets + 1);
  s->tasks = s->res.device<uint2>(s->max_tasks);
  s->flags = s->res.device<uint32_t>(8);
  s->flags_host = s->res.pinned<uint32_t>(8);
  memset(s->flags_host, 0, 8 * sizeof(uint32_t));
  s->scratch_bytes = s->res.device_bytes();
}

void msm_sort_launch(MsmSort* s, const Fr* scalars, size_t n_points, cudaStream_t st) {
  if (n_points > s->n_points) throw std::runtime_error("msm: sort plan too small");
  const uint32_t nb = (uint32_t)s->n_buckets;
  NZCP_CUDA(cudaMemsetAsync(s->flags, 0, 8 * sizeof(uint32_t), st));
  if (n_points) {
    // shared-memory histogram: one block per SM (fewer for small inputs); otherwise 16 global copies of the counters
    uint32_t n_copies = s->n_copies;
    if (s->smem_hist) {
      uint32_t want = div_up(n_points, kSmemHistThreads);   // one block per 1024 scalars at most, whatever its thread count
      if (want < n_copies) n_copies = want;
    }
    // "sort_threads": threads per block of the shared-memory histogram passes (one block per SM, 128 KB of shared memory).
    // A 1024-thread block needs a whole SM's thread slots and registers at once; a thinner one can be placed beside the
    // blocks of whatever kernel another stream is running.
    int sort_threads = g_tune_sort_threads.load();
    sort_threads = sort_threads >= 1024 ? 1024 : sort_threads >= 512 ? 512 : sort_threads >= 256 ? 256 : 128;
    const uint32_t n_ctr = nb * n_copies;
    // entries index the table of the plan's full point count, so a shorter scalar vector still addresses T[w][i]
    DigitParams dp{n_copies, (uint32_t)n_points, s->table_free ? 0u : (uint32_t)s->n_points, s->c, s->n_windows,
                   (uint32_t)s->group_buckets, s->table_free ? (uint32_t)s->group_buckets : 0u, nb};
    const unsigned gp = div_up(n_points, 256);
    const size_t hist_bytes = (size_t)nb * sizeof(uint32_t);
    if (s->smem_hist) {
      NZCP_CUDA(cudaMemsetAsync(s->counts + n_ctr, 0, sizeof(uint32_t), st));
      msm_digits_smem_kernel<false><<<n_copies, sort_threads, hist_bytes, st>>>(scalars, dp, s->counts, nullptr, s->flags);
    } else {
      NZCP_CUDA(cudaMemsetAsync(s->counts, 0, (n_ctr + 1) * sizeof(uint32_t), st));
      msm_digits_kernel<false><<<gp, 256, 0, st>>>(scalars, dp, s->counts, nullptr, s->flags);
    }
    NZCP_LAUNCH_CHECK();
    // exclusive scan of the sub-counters (counts[n_ctr] = 0 is scanned too, so offsets[n_ctr] = total)
    const uint32_t n_scan = n_ctr + 1;
    const uint32_t n_blk = div_up(n_scan, kScanBlock);
    uint32_t* blk_sum = s->block_sums;
    uint32_t* blk_off = s->block_sums + (s->n_buckets * s->n_copies / kScanBlock + 2);
    msm_scan_sums_kernel<<<n_blk, 256, 0, st>>>(s->counts, blk_sum, n_scan);
    NZCP_LAUNCH_CHECK();
    msm_scan_kernel<false><<<1, 1024, 0, st>>>(blk_sum, blk_off, n_blk, s->flags + 3, s->flags);
    NZCP_LAUNCH_CHECK();
    msm_scan_apply_kernel<<<n_blk, 256, 0, st>>>(s->counts, blk_off, s->offsets, s->smem_hist ? nullptr : s->cursors, n_scan);
    NZCP_LAUNCH_CHECK();
    if (s->smem_hist)
      msm_digits_smem_kernel<true><<<n_copies, sort_threads, hist_bytes, st>>>(scalars, dp, s->offsets, s->entries, s->flags);
    else
      msm_digits_kernel<true><<<gp, 256, 0, st>>>(scalars, dp, s->cursors, s->entries, s->flags);
    NZCP_LAUNCH_CHECK();
    switch (s->rounds) {
      case 0: msm_round_plan_kernel<0><<<1, 1024, 0, st>>>(s->offsets, n_copies, nb, s->round_off, s->red_count, s->flags); break;
      case 1: msm_round_plan_kernel<1><<<1, 1024, 0, st>>>(s->offsets, n_copies, nb, s->round_off, s->red_count, s->flags); break;
      case 2: msm_round_plan_kernel<2><<<1, 1024, 0, st>>>(s->offsets, n_copies, nb, s->round_off, s->red_count, s->flags); break;
      default: msm_round_plan_kernel<3><<<1, 1024, 0, st>>>(s->offsets, n_copies, nb, s->round_off, s->red_count, s->flags); break;
    }
    NZCP_LAUNCH_CHECK();
    msm_scan_kernel<true><<<1, 1024, 0, st>>>(s->red_count, s->task_off, nb, s->flags + 2, s->flags);
    NZCP_LAUNCH_CHECK();
    msm_task_fill_kernel<<<div_up(s->max_tasks, 256), 256, 0, st>>>(s->red_count, s->round_off + (size_t)s->rounds * (nb + 1),
                                                                     s->task_off, s->tasks, nb, s->flags);
    NZCP_LAUNCH_CHECK();
  } else {
    NZCP_CUDA(cudaMemsetAsync(s->task_off, 0, (nb + 1) * sizeof(uint32_t), st));
  }
  NZCP_CUDA(cudaMemcpyAsync(s->flags_host, s->flags, 8 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
}

uint32_t msm_sort_check(const MsmSort* s) {
  if (s->flags_host[1]) throw std::runtime_error("witness/scalar value is not a canonical field element (>= r)");
  return s->flags_host[3];
}

void msm_run_create(MsmRun* r, const MsmSort* sort, bool g2) {
  *r = MsmRun();
  r->g2 = g2;
  size_t psz = g2 ? sizeof(G2XYZZ) : sizeof(G1XYZZ);
  if (g2) {  // > 48 KB of dynamic shared memory; function attributes are per device
    NZCP_CUDA(cudaFuncSetAttribute(msm_combine_heavy_kernel<Fq2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(kHeavyThreads * sizeof(G2XYZZ))));
    NZCP_CUDA(cudaFuncSetAttribute(msm_combine_heavy2_kernel<Fq2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(kHeavyThreads * sizeof(G2XYZZ))));
    NZCP_CUDA(cudaFuncSetAttribute(msm_marginal_kernel<Fq2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(kMargThreads * sizeof(G2XYZZ))));
  }
  r->partial = r->res.device<unsigned char>(sort->max_tasks * psz);
  r->buckets = r->res.device<unsigned char>(sort->n_buckets * psz);
  r->n_groups = sort->n_groups;
  r->c = sort->c;
  r->marg = r->res.device<unsigned char>((size_t)r->n_groups * kMaxDigits * 32 * psz);
  r->marg_done = r->res.device<uint32_t>((size_t)r->n_groups * kMaxDigits);
  NZCP_CUDA(cudaMemset(r->marg_done, 0, (size_t)r->n_groups * kMaxDigits * sizeof(uint32_t)));
  r->result = r->res.device<unsigned char>(psz);
  r->heavy_list = r->res.device<uint32_t>(sort->n_buckets);
  r->heavy_count = r->res.device<uint32_t>(2);
  r->chunk_off = r->res.device<uint32_t>(sort->n_buckets + 1);
  r->chunk_partial = r->res.device<unsigned char>((sort->max_tasks / kHeavyChunk + sort->n_buckets + 1) * psz);
  r->out = r->res.device<unsigned char>((size_t)r->n_groups * (kMaxDigits + 1) * psz);
  r->out_host = r->res.pinned<unsigned char>((size_t)r->n_groups * (kMaxDigits + 1) * psz);
  memset(r->out_host, 0, (size_t)r->n_groups * (kMaxDigits + 1) * psz);
  r->n_digits = (sort->c - 1 + 4) / 5;
  NZCP_CUDA(cudaFuncSetAttribute(msm_sum_points_kernel<Fq2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(kHeavyThreads * sizeof(G2XYZZ))));
  if (sort->rounds > 0) {
    const size_t asz = g2 ? sizeof(G2Affine) : sizeof(G1Affine), fsz = asz / 2, pad = 128 * 64;
    r->round_pts[0] = r->res.device<unsigned char>((sort->round_max[1] + pad) * asz);
    if (sort->rounds > 1) r->round_pts[1] = r->res.device<unsigned char>((sort->round_max[2] + pad) * asz);
    r->round_prefix = r->res.device<unsigned char>((sort->round_max[1] + pad) * fsz);
    if (g_tune_pair_stage.load())   // opt-in ("pair_stage", read when the run is created): two operands per round-1 addition
      r->round_ops = r->res.device<unsigned char>((sort->round_max[1] + pad) * 2 * asz);
    r->round_prod = r->res.device<unsigned char>((sort->round_max[1] / 4 + pad) * fsz);   // >= 4 additions per thread
  }
  r->ev_acc0 = r->res.event();
  r->ev_acc1 = r->res.event();
  r->scratch_bytes = r->res.device_bytes();
}

template <class F>
static void msm_run_launch_t(MsmRun* r, const MsmSort* s, const MsmTable* t, cudaStream_t st) {
  if (t->c != s->c || t->n_points != s->n_points || t->n_windows != (s->table_free ? 1 : s->n_windows))
    throw std::runtime_error("msm: table and sort plan do not match");
  const uint32_t nb = (uint32_t)s->n_buckets;
  const size_t psz = sizeof(XYZZ<F>);
  XYZZ<F>* partial = reinterpret_cast<XYZZ<F>*>(r->partial);
  XYZZ<F>* buckets = reinterpret_cast<XYZZ<F>*>(r->buckets);
  XYZZ<F>* out = reinterpret_cast<XYZZ<F>*>(r->out);
  NZCP_CUDA(cudaMemsetAsync(r->heavy_count, 0, 2 * sizeof(uint32_t), st));
  NZCP_CUDA(cudaEventRecord(r->ev_acc0, st));
  if (s->rounds == 0) {
    msm_accumulate_kernel<F><<<div_up(s->max_tasks, 128), 128, 0, st>>>(reinterpret_cast<const Affine<F>*>(t->pts),
                                                                       s->entries, s->tasks, s->flags, partial,
                                                                       (g_tune_acc_prefetch.load() ? 1 : 0) | (g_tune_gather_hint.load() ? 4 : 0));
    NZCP_LAUNCH_CHECK();
  } else {
    // pair rounds: table -> pts[0] -> pts[1] -> pts[0]; then the XYZZ accumulation over the last array
    const Affine<F>* src = reinterpret_cast<const Affine<F>*>(t->pts);
    for (int rd = 1; rd <= s->rounds; rd++) {
      Affine<F>* dst = reinterpret_cast<Affine<F>*>(r->round_pts[(rd - 1) & 1]);
      const uint32_t* off_in = s->round_off + (size_t)(rd - 1) * (nb + 1);
      const uint32_t* off_out = s->round_off + (size_t)rd * (nb + 1);
      const int hint = g_tune_gather_hint.load() ? 4 : 0;
      const int pf_fwd = g_tune_pair_prefetch[0].load() | hint, pf_bwd = g_tune_pair_prefetch[1].load() | hint;
      int k = g_tune_pair_k[rd - 1].load();
      k = k >= 32 ? 32 : k >= 16 ? 16 : k >= 8 ? 8 : 4;
      const unsigned grid = div_up(div_up(s->round_max[rd], k) + kPairLanes, 128);   // + one warp: the last one may be partial in every lane
      const unsigned grid_inv = div_up(div_up((size_t)grid * 128, kPairInvGroup), 64);
      F* scratch = reinterpret_cast<F*>(r->round_prefix);
      F* prod = reinterpret_cast<F*>(r->round_prod);
      Affine<F>* ops = g_tune_pair_stage.load() ? reinterpret_cast<Affine<F>*>(r->round_ops) : nullptr;   // round 1 only;
                                                                                   // null unless the run was created with it
#define NZCP_PAIR_LAUNCH(TABLE, KK)                                                                                       \
      do {                                                                                                                \
        msm_pair_forward_kernel<F, TABLE, KK><<<grid, 128, 0, st>>>(src, s->entries, off_in, off_out, nb, scratch, prod, \
                                                                    pf_fwd, TABLE ? ops : nullptr);                       \
        NZCP_LAUNCH_CHECK();                                                                                              \
        msm_pair_invert_kernel<F, KK><<<grid_inv, 64, 0, st>>>(prod, off_out, nb);                                        \
        NZCP_LAUNCH_CHECK();                                                                                              \
        msm_pair_backward_kernel<F, TABLE, KK><<<grid, 128, 0, st>>>(src, s->entries, off_in, off_out, nb, dst, scratch,  \
                                                                     prod, pf_bwd, TABLE ? ops : nullptr);                \
        NZCP_LAUNCH_CHECK();                                                                                              \
      } while (0)
      if (rd == 1) {
        if (k == 32) NZCP_PAIR_LAUNCH(true, 32); else if (k == 16) NZCP_PAIR_LAUNCH(true, 16);
        else if (k == 8) NZCP_PAIR_LAUNCH(true, 8); else NZCP_PAIR_LAUNCH(true, 4);
      } else {
        if (k == 32) NZCP_PAIR_LAUNCH(false, 32); else if (k == 16) NZCP_PAIR_LAUNCH(false, 16);
        else if (k == 8) NZCP_PAIR_LAUNCH(false, 8); else NZCP_PAIR_LAUNCH(false, 4);
      }
#undef NZCP_PAIR_LAUNCH
      src = dst;
    }
    msm_accumulate_pts_kernel<F><<<div_up(s->max_tasks, 128), 128, 0, st>>>(src, s->tasks, s->flags, partial);
    NZCP_LAUNCH_CHECK();
  }
  NZCP_CUDA(cudaEventRecord(r->ev_acc1, st));
  msm_combine_kernel<F><<<div_up(nb, 128), 128, 0, st>>>(s->task_off, partial, buckets, nb, r->heavy_list,
                                                                     r->heavy_count);
  NZCP_LAUNCH_CHECK();
  msm_heavy_scan_kernel<<<1, 1024, 0, st>>>(s->task_off, r->heavy_list, r->heavy_count, r->chunk_off);
  NZCP_LAUNCH_CHECK();
  XYZZ<F>* chunk_partial = reinterpret_cast<XYZZ<F>*>(r->chunk_partial);
  // the chunk count is only known on the device: a grid large enough for "every bucket is heavy" (standalone MSMs of
  // 2^22+ points), whose surplus blocks exit at once in the prover's case (a few hundred heavy buckets at most)
  msm_combine_heavy_kernel<F><<<148 * 16, kHeavyThreads, kHeavyThreads * psz, st>>>(s->task_off, partial, r->heavy_list,
                                                                                    r->heavy_count, r->chunk_off, chunk_partial,
                                                                                    buckets);
  NZCP_LAUNCH_CHECK();
  msm_combine_heavy2_kernel<F><<<148, kHeavyThreads, kHeavyThreads * psz, st>>>(r->heavy_list, r->heavy_count, r->chunk_off,
                                                                                chunk_partial, buckets);
  NZCP_LAUNCH_CHECK();
  const uint32_t bits = (uint32_t)(s->c - 1);
  const uint32_t n_digits = (bits + 4) / 5;
  XYZZ<F>* marg = reinterpret_cast<XYZZ<F>*>(r->marg);
  msm_marginal_kernel<F><<<(unsigned)s->n_groups * n_digits * 32, kMargThreads, kMargThreads * psz, st>>>(buckets, marg, out,
                                                                                                      r->marg_done, bits, n_digits);
  NZCP_LAUNCH_CHECK();
  NZCP_CUDA(cudaMemcpyAsync(r->out_host, r->out, (size_t)s->n_groups * (n_digits + 1) * psz, cudaMemcpyDeviceToHost, st));
}

// After msm_run_launch on the same stream: fold the run's digit sums into ONE point that stays on the device.
void msm_run_finish_device(MsmRun* r, cudaStream_t st) {
  if (r->g2)
    msm_finish_kernel<Fq2><<<1, 32, 0, st>>>(reinterpret_cast<const G2XYZZ*>(r->out), reinterpret_cast<G2XYZZ*>(r->result),
                                             (uint32_t)r->n_groups, (uint32_t)r->n_digits, r->c);
  else
    msm_finish_kernel<Fq><<<1, 32, 0, st>>>(reinterpret_cast<const G1XYZZ*>(r->out), reinterpret_cast<G1XYZZ*>(r->result),
                                            (uint32_t)r->n_groups, (uint32_t)r->n_digits, r->c);
  NZCP_LAUNCH_CHECK();
}

// result (device, one XYZZ point) = sum of `count` XYZZ points in device memory.
void msm_sum_points(const void* d_pts, uint32_t count, bool g2, void* d_result, cudaStream_t st) {
  if (g2) {
    NZCP_CUDA(cudaFuncSetAttribute(msm_sum_points_kernel<Fq2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(kHeavyThreads * sizeof(G2XYZZ))));
    msm_sum_points_kernel<Fq2><<<1, kHeavyThreads, kHeavyThreads * sizeof(G2XYZZ), st>>>(
        reinterpret_cast<const G2XYZZ*>(d_pts), count, reinterpret_cast<G2XYZZ*>(d_result));
  } else {
    msm_sum_points_kernel<Fq><<<1, kHeavyThreads, kHeavyThreads * sizeof(G1XYZZ), st>>>(
        reinterpret_cast<const G1XYZZ*>(d_pts), count, reinterpret_cast<G1XYZZ*>(d_result));
  }
  NZCP_LAUNCH_CHECK();
}

void msm_run_launch(MsmRun* r, const MsmSort* sort, const MsmTable* table, cudaStream_t st) {
  if (r->g2 != table->g2) throw std::runtime_error("msm: run and table group mismatch");
  if (r->g2)
    msm_run_launch_t<Fq2>(r, sort, table, st);
  else
    msm_run_launch_t<Fq>(r, sort, table, st);
}

template <class F>
static XYZZ<F> msm_run_finish_t(const MsmRun* r) {
  // sum_v v B_v = T + sum_k 32^k S_k : Horner over the digit positions (a handful of host group operations)
  // table-free runs: one such sum per window, folded by Horner with c doublings per step (ffjavascript's own last step)
  XYZZ<F> res = XYZZ<F>::inf();
  for (int g = r->n_groups - 1; g >= 0; g--) {
    const XYZZ<F>* w = reinterpret_cast<const XYZZ<F>*>(r->out_host) + (size_t)g * (r->n_digits + 1);
    XYZZ<F> acc = XYZZ<F>::inf();
    for (int k = r->n_digits - 1; k >= 0; k--) {
      if (!acc.is_inf())
        for (int d = 0; d < 5; d++) acc = xyzz_dbl(acc);
      xyzz_add(acc, w[k]);
    }
    xyzz_add(acc, w[r->n_digits]);
    if (!res.is_inf())
      for (int d = 0; d < r->c; d++) res = xyzz_dbl(res);
    xyzz_add(res, acc);
  }
  return res;
}

G1XYZZ msm_run_finish_g1(const MsmRun* r) { return msm_run_finish_t<Fq>(r); }
G2XYZZ msm_run_finish_g2(const MsmRun* r) { return msm_run_finish_t<Fq2>(r); }

float msm_run_accumulate_ms(const MsmRun* r) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, r->ev_acc0, r->ev_acc1) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return ms;
}

}  // namespace nzcp
