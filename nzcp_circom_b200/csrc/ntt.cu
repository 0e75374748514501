// BN254-Fr number-theoretic transforms for the Groth16 H pipeline.
//
// Replaces (upstream, not vendored: yarn.lock:408-416, 1132-1135)
//   ffjavascript src/engine_fft.js  (Fr.fft / Fr.ifft: natural order in and out, worker fan-out of <=2^14 blocks,
//                                    frm_fft / frm_ifft / frm_fftJoin / frm_fftFinal in wasmcurves build_fft.js)
//   ffjavascript src/engine_applykey.js (Fr.batchApplyKey(buf, 1, inc): element i *= inc^i)
//   wasmcurves build_qap.js qap_joinABC + frm_batchFromMontgomery (joinABC in snarkjs src/groth16_prove.js)
// as called from snarkjs groth16_prove.js:  for X in A,B,C: ifft -> batchApplyKey -> fft ; joinABC.
//
// B200 design.  One polynomial is n x 32 B (32 MiB at n = 2^20).  Per polynomial the pipeline is
//     iNTT as decimation-in-frequency (natural in -> bit-reversed out)
//     x  n^-1 * inc^bitrev(p)            (the 1/n of the iNTT fused with batchApplyKey, one table)
//     NTT as decimation-in-time          (bit-reversed in -> natural out)
// so no bit-reversal pass is ever materialised.  Stages are grouped into passes of <= 10 radix-2 stages that run
// out of shared memory; the low DIF pass, the scale and the low DIT pass touch the same contiguous tile and are one
// kernel.  At n = 2^20 that is 3 launches (hi DIF, fused lo, hi DIT) = 3 read+write sweeps of HBM per polynomial,
// A/B/C batched through grid.y.  Shared tiles are limb-planar (8 planes of u32) with index padding l + l/32 so that
// both unit-stride and stride-2 butterflies are bank-conflict free.
#include "common.cuh"

namespace nzcp {

static constexpr int kNttThreads = 256;
#ifndef NZCP_NTT_MIN_BLOCKS
#define NZCP_NTT_MIN_BLOCKS 2
#endif
static constexpr int kMaxPassBits = 10;
std::atomic<int> g_tune_ntt_tma{1};   // "ntt_tma" knob: 1 = TMA-staged low pass (below), 0 = the thread-loaded one

__device__ __forceinline__ uint32_t pad_idx(uint32_t l) { return l + (l >> 5); }

__device__ __forceinline__ Fr sm_load(const uint32_t* sm, uint32_t plane, uint32_t l) {
  Fr r;
  uint32_t p = pad_idx(l);
#pragma unroll
  for (int k = 0; k < 8; k++) r.v[k] = sm[k * plane + p];
  return r;
}
__device__ __forceinline__ void sm_store(uint32_t* sm, uint32_t plane, uint32_t l, const Fr& x) {
  uint32_t p = pad_idx(l);
#pragma unroll
  for (int k = 0; k < 8; k++) sm[k * plane + p] = x.v[k];
}
__device__ __forceinline__ Fr g_load(const Fr* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  Fr r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
__device__ __forceinline__ void g_store(Fr* p, const Fr& x) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
  q[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
}

// One radix-2 stage on the shared tile.  sl = stage index inside the pass (global bit s = lo + sl).
// low_bits = the fixed low index bits of this tile below `lo` other than the `cb` column bits.
template <bool DIT>
__device__ __forceinline__ void tile_stage(uint32_t* sm, uint32_t plane, uint32_t tile_elems, const Fr* tw, int log_n,
                                           int lo, int sl, int cb, uint32_t low_bits) {
  const int lb = sl + cb;        // local bit that this stage pairs
  const int s = lo + sl;         // global bit
  const uint32_t cmask = (1u << cb) - 1;
  for (uint32_t b = threadIdx.x; b < (tile_elems >> 1); b += blockDim.x) {
    uint32_t l0 = ((b >> lb) << (lb + 1)) | (b & ((1u << lb) - 1));
    uint32_t l1 = l0 | (1u << lb);
    uint32_t t = l0 >> cb;
    uint32_t imod = ((t & ((1u << sl) - 1)) << lo) | low_bits | (l0 & cmask);  // global index mod 2^s
    uint32_t e = imod << (log_n - 1 - s);                                      // exponent of w, < n/2
    Fr u = sm_load(sm, plane, l0);
    Fr v = sm_load(sm, plane, l1);
    if (DIT) {
      if (e) v = fp_mul(v, g_load(tw + e));
      sm_store(sm, plane, l0, fp_add(u, v));
      sm_store(sm, plane, l1, fp_sub(u, v));
    } else {
      Fr d = fp_sub(u, v);
      if (e) d = fp_mul(d, g_load(tw + e));
      sm_store(sm, plane, l0, fp_add(u, v));
      sm_store(sm, plane, l1, d);
    }
  }
}

// Two radix-2 stages (sl and sl + 1) at once on four elements held in registers: half the shared-memory traffic and
// half the barriers of two tile_stage calls, same four twiddle products.  Elements l00, l01 (bit lb), l10, l11 (bit
// lb+1).  w1 = twiddle of stage s for this group; w2, w3 = twiddles of stage s+1 for the l00/l10 and l01/l11 pairs
// (w3 = w2 * w^(n/4)).
template <bool DIT>
__device__ __forceinline__ void tile_stage4(uint32_t* sm, uint32_t plane, uint32_t tile_elems, const Fr* tw, int log_n,
                                            int lo, int sl, int cb, uint32_t low_bits) {
  const int lb = sl + cb;
  const int s = lo + sl;
  const uint32_t cmask = (1u << cb) - 1;
  for (uint32_t g = threadIdx.x; g < (tile_elems >> 2); g += blockDim.x) {
    const uint32_t l00 = ((g >> lb) << (lb + 2)) | (g & ((1u << lb) - 1));
    const uint32_t l01 = l00 | (1u << lb), l10 = l00 | (2u << lb), l11 = l00 | (3u << lb);
    const uint32_t t = l00 >> cb;
    const uint32_t imod = ((t & ((1u << sl) - 1)) << lo) | low_bits | (l00 & cmask);  // global index mod 2^s
    const uint32_t e1 = imod << (log_n - 1 - s);
    const uint32_t e2 = imod << (log_n - 2 - s);
    const uint32_t e3 = e2 + (1u << (log_n - 2));
    Fr x0 = sm_load(sm, plane, l00), x1 = sm_load(sm, plane, l01);
    Fr x2 = sm_load(sm, plane, l10), x3 = sm_load(sm, plane, l11);
    if (DIT) {
      if (e1) {
        Fr w1 = g_load(tw + e1);
        x1 = fp_mul(x1, w1);
        x3 = fp_mul(x3, w1);
      }
      Fr s0 = fp_add(x0, x1), s1 = fp_sub(x0, x1), s2 = fp_add(x2, x3), s3 = fp_sub(x2, x3);
      if (e2) s2 = fp_mul(s2, g_load(tw + e2));
      s3 = fp_mul(s3, g_load(tw + e3));
      sm_store(sm, plane, l00, fp_add(s0, s2));
      sm_store(sm, plane, l10, fp_sub(s0, s2));
      sm_store(sm, plane, l01, fp_add(s1, s3));
      sm_store(sm, plane, l11, fp_sub(s1, s3));
    } else {
      Fr p0 = fp_add(x0, x2), p2 = fp_sub(x0, x2), p1 = fp_add(x1, x3), p3 = fp_sub(x1, x3);
      if (e2) p2 = fp_mul(p2, g_load(tw + e2));
      p3 = fp_mul(p3, g_load(tw + e3));
      Fr d0 = fp_sub(p0, p1), d1 = fp_sub(p2, p3);
      if (e1) {
        Fr w1 = g_load(tw + e1);
        d0 = fp_mul(d0, w1);
        d1 = fp_mul(d1, w1);
      }
      sm_store(sm, plane, l00, fp_add(p0, p1));
      sm_store(sm, plane, l01, d0);
      sm_store(sm, plane, l10, fp_add(p2, p3));
      sm_store(sm, plane, l11, d1);
    }
  }
}

// All ns stages of a pass on the shared tile, two at a time (one radix-2 stage left over when ns is odd).
template <bool DIT>
__device__ __forceinline__ void tile_stages(uint32_t* sm, uint32_t plane, uint32_t tile_elems, const Fr* tw, int log_n,
                                            int lo, int ns, int cb, uint32_t low_bits) {
  if (DIT) {
    int sl = 0;
    for (; sl + 1 < ns; sl += 2) {
      tile_stage4<true>(sm, plane, tile_elems, tw, log_n, lo, sl, cb, low_bits);
      __syncthreads();
    }
    if (sl < ns) {
      tile_stage<true>(sm, plane, tile_elems, tw, log_n, lo, sl, cb, low_bits);
      __syncthreads();
    }
  } else {
    int sl = ns - 1;
    if (ns & 1) {
      tile_stage<false>(sm, plane, tile_elems, tw, log_n, lo, sl, cb, low_bits);
      __syncthreads();
      sl--;
    }
    for (; sl >= 1; sl -= 2) {
      tile_stage4<false>(sm, plane, tile_elems, tw, log_n, lo, sl - 1, cb, low_bits);
      __syncthreads();
    }
  }
}

// Generic pass over global bits [lo, lo+ns).  Tile = 2^ns "rows" x 2^cb adjacent columns (cb <= lo).
// grid.x = n >> (ns + cb) tiles, grid.y = batch.
template <bool DIT>
__global__ void __launch_bounds__(kNttThreads, NZCP_NTT_MIN_BLOCKS)
ntt_pass_kernel(Fr* __restrict__ data, const Fr* __restrict__ tw, int log_n, int lo, int ns, int cb) {
  extern __shared__ uint32_t sm[];
  const uint32_t tile_elems = 1u << (ns + cb);
  const uint32_t plane = tile_elems + (tile_elems >> 5) + 1;
  Fr* x = data + ((size_t)blockIdx.y << log_n);
  const uint32_t lhi_bits = lo - cb;
  const uint32_t tile = blockIdx.x;
  const uint32_t lhi = tile & ((1u << lhi_bits) - 1);
  const uint32_t upper = tile >> lhi_bits;
  const uint32_t low_bits = lhi << cb;
  const uint32_t base = (upper << (lo + ns)) | low_bits;
  const uint32_t cmask = (1u << cb) - 1;
  for (uint32_t l = threadIdx.x; l < tile_elems; l += blockDim.x) {
    uint32_t gi = base | ((l >> cb) << lo) | (l & cmask);
    sm_store(sm, plane, l, g_load(x + gi));
  }
  __syncthreads();
  tile_stages<DIT>(sm, plane, tile_elems, tw, log_n, lo, ns, cb, low_bits);
  for (uint32_t l = threadIdx.x; l < tile_elems; l += blockDim.x) {
    uint32_t gi = base | ((l >> cb) << lo) | (l & cmask);
    g_store(x + gi, sm_load(sm, plane, l));
  }
}

// Low pass of the pipeline: DIF stages ns-1..0 (inverse twiddles), scale by n^-1 * inc^bitrev(p), DIT stages
// 0..ns-1 (forward twiddles).  Contiguous tile of 2^ns elements.
__global__ void __launch_bounds__(kNttThreads, NZCP_NTT_MIN_BLOCKS)
ntt_fused_lo_kernel(Fr* __restrict__ data, const Fr* __restrict__ tw_inv, const Fr* __restrict__ tw_fwd,
                    const Fr* __restrict__ scale, int log_n, int ns) {
  extern __shared__ uint32_t sm[];
  const uint32_t tile_elems = 1u << ns;
  const uint32_t plane = tile_elems + (tile_elems >> 5) + 1;
  Fr* x = data + ((size_t)blockIdx.y << log_n);
  const uint32_t base = blockIdx.x << ns;
  for (uint32_t l = threadIdx.x; l < tile_elems; l += blockDim.x) sm_store(sm, plane, l, g_load(x + base + l));
  __syncthreads();
  tile_stages<false>(sm, plane, tile_elems, tw_inv, log_n, 0, ns, 0, 0);
  for (uint32_t l = threadIdx.x; l < tile_elems; l += blockDim.x) {
    Fr v = sm_load(sm, plane, l);
    sm_store(sm, plane, l, fp_mul(v, g_load(scale + base + l)));
  }
  __syncthreads();
  tile_stages<true>(sm, plane, tile_elems, tw_fwd, log_n, 0, ns, 0, 0);
  for (uint32_t l = threadIdx.x; l < tile_elems; l += blockDim.x) g_store(x + base + l, sm_load(sm, plane, l));
}


// ------------------------------------------------------------------------------------------------ TMA-staged low pass
// The same low pass with its operands staged by the copy engine instead of by the threads (north_star: "TMA-staged,
// coalesced 128-bit HBM access"):
//   * persistent blocks (two per SM) walk the contiguous 32 KB tiles of all polynomials; while a tile is being transformed
//     the NEXT one is already in flight: one 1-D bulk copy (cp.async.bulk.shared::cluster.global, SASS UBLKCP) into a
//     staging buffer, completion counted in bytes on an mbarrier -- no thread issues a load for the data it will touch;
//   * the twiddles of the pass -- 512 of each direction, w^(j * n/1024): every stage of a 2^10-point tile draws from this
//     set -- are bulk-copied ONCE per block into shared memory and read from there in the butterflies, instead of one
//     L2 round trip per butterfly (ncu r01: long_scoreboard 1.1-1.5 in this kernel, all of it twiddle fetches).
// The staging buffer is array-of-structures (what a linear copy lands); one repack pass moves it into the limb-planar,
// padded compute tile (same 10 shared-memory instructions per element the direct global->shared load used to cost).
// The compact twiddle tables are stored PADDED in global memory (16 B after every 4 and every 32 entries), so that the
// power-of-two strides of the radix-4 sweeps are bank-conflict free for 128-bit shared loads; the bulk copy lands the
// padded layout as is.
static constexpr int kLoTmaBits = 10;
static constexpr uint32_t kLoTmaTile = 1u << kLoTmaBits;
static constexpr uint32_t kLoTmaTileBytes = kLoTmaTile * 32;
static constexpr uint32_t kLoTwEntries = kLoTmaTile / 2;
__host__ __device__ constexpr uint32_t tw_pad_off(uint32_t j) { return 32 * j + 16 * (j >> 2) + 16 * (j >> 5); }
static constexpr uint32_t kLoTwBytes = tw_pad_off(kLoTwEntries);   // 18 688
static constexpr uint32_t kLoPlane = kLoTmaTile + (kLoTmaTile >> 5) + 1;
static constexpr uint32_t kLoTmaSmem = kLoTmaTileBytes + 8 * kLoPlane * 4 + 2 * kLoTwBytes + 16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared (bytes a multiple of 16, both addresses 16-byte aligned), completing on `bar`.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ Fr lds_fr(const unsigned char* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  Fr r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
__device__ __forceinline__ Fr tw_sm(const unsigned char* tw, uint32_t j) { return lds_fr(tw + tw_pad_off(j)); }

// Stages sl and sl + 1 of the contiguous 2^10 tile (global bit = local bit), twiddles from the padded shared table:
// w^(imod * n / 2^(s+1)) = table[imod << (9 - s)].
template <bool DIT>
__device__ __forceinline__ void lo_stage4(uint32_t* sm, const unsigned char* tw, int sl) {
  for (uint32_t g = threadIdx.x; g < (kLoTmaTile >> 2); g += blockDim.x) {
    const uint32_t l00 = ((g >> sl) << (sl + 2)) | (g & ((1u << sl) - 1));
    const uint32_t l01 = l00 | (1u << sl), l10 = l00 | (2u << sl), l11 = l00 | (3u << sl);
    const uint32_t imod = l00 & ((1u << sl) - 1);
    const uint32_t j1 = imod << (9 - sl), j2 = imod << (8 - sl), j3 = j2 + (kLoTwEntries >> 1);
    Fr x0 = sm_load(sm, kLoPlane, l00), x1 = sm_load(sm, kLoPlane, l01);
    Fr x2 = sm_load(sm, kLoPlane, l10), x3 = sm_load(sm, kLoPlane, l11);
    if (DIT) {
      if (j1) {
        Fr w1 = tw_sm(tw, j1);
        x1 = fp_mul(x1, w1);
        x3 = fp_mul(x3, w1);
      }
      Fr s0 = fp_add(x0, x1), s1 = fp_sub(x0, x1), s2 = fp_add(x2, x3), s3 = fp_sub(x2, x3);
      if (j2) s2 = fp_mul(s2, tw_sm(tw, j2));
      s3 = fp_mul(s3, tw_sm(tw, j3));
      sm_store(sm, kLoPlane, l00, fp_add(s0, s2));
      sm_store(sm, kLoPlane, l10, fp_sub(s0, s2));
      sm_store(sm, kLoPlane, l01, fp_add(s1, s3));
      sm_store(sm, kLoPlane, l11, fp_sub(s1, s3));
    } else {
      Fr p0 = fp_add(x0, x2), p2 = fp_sub(x0, x2), p1 = fp_add(x1, x3), p3 = fp_sub(x1, x3);
      if (j2) p2 = fp_mul(p2, tw_sm(tw, j2));
      p3 = fp_mul(p3, tw_sm(tw, j3));
      Fr d0 = fp_sub(p0, p1), d1 = fp_sub(p2, p3);
      if (j1) {
        Fr w1 = tw_sm(tw, j1);
        d0 = fp_mul(d0, w1);
        d1 = fp_mul(d1, w1);
      }
      sm_store(sm, kLoPlane, l00, fp_add(p0, p1));
      sm_store(sm, kLoPlane, l01, d0);
      sm_store(sm, kLoPlane, l10, fp_add(p2, p3));
      sm_store(sm, kLoPlane, l11, d1);
    }
  }
}

__global__ void __launch_bounds__(kNttThreads, 2)
ntt_fused_lo_tma_kernel(Fr* __restrict__ data, const unsigned char* __restrict__ tw_inv_lo,
                        const unsigned char* __restrict__ tw_fwd_lo, const Fr* __restrict__ scale, int log_n, uint32_t n_tiles) {
  extern __shared__ __align__(128) unsigned char lo_smem[];
  unsigned char* stage = lo_smem;                                                     // 32 KB, bulk-copy destination
  uint32_t* sm = reinterpret_cast<uint32_t*>(lo_smem + kLoTmaTileBytes);             // limb-planar compute tile
  unsigned char* tw_inv = lo_smem + kLoTmaTileBytes + 8 * kLoPlane * 4;
  unsigned char* tw_fwd = tw_inv + kLoTwBytes;
  uint64_t* bar_tile = reinterpret_cast<uint64_t*>(tw_fwd + kLoTwBytes);
  uint64_t* bar_tw = bar_tile + 1;
  const uint32_t tile_bits = (uint32_t)(log_n - kLoTmaBits);                         // tiles per polynomial = 2^tile_bits
  auto tile_ptr = [&](uint32_t t) { return data + (((size_t)(t >> tile_bits)) << log_n) + ((size_t)(t & ((1u << tile_bits) - 1)) << kLoTmaBits); };
  uint32_t t = blockIdx.x;
  if (threadIdx.x == 0) {
    mbar_init(bar_tile, 1);
    mbar_init(bar_tw, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(bar_tw, 2 * kLoTwBytes);
    bulk_g2s(tw_inv, tw_inv_lo, kLoTwBytes, bar_tw);
    bulk_g2s(tw_fwd, tw_fwd_lo, kLoTwBytes, bar_tw);
    if (t < n_tiles) {
      mbar_expect_tx(bar_tile, kLoTmaTileBytes);
      bulk_g2s(stage, tile_ptr(t), kLoTmaTileBytes, bar_tile);
    }
  }
  __syncthreads();                 // barrier initialisation visible to every waiter
  mbar_wait(bar_tw, 0);
  uint32_t parity = 0;
  for (; t < n_tiles; t += gridDim.x) {
    mbar_wait(bar_tile, parity);
    parity ^= 1;
    for (uint32_t l = threadIdx.x; l < kLoTmaTile; l += blockDim.x) sm_store(sm, kLoPlane, l, lds_fr(stage + 32 * l));
    __syncthreads();               // staging buffer drained, compute tile complete
    const uint32_t tn = t + gridDim.x;
    if (threadIdx.x == 0 && tn < n_tiles) {   // next tile on its way while this one is transformed
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar_tile, kLoTmaTileBytes);
      bulk_g2s(stage, tile_ptr(tn), kLoTmaTileBytes, bar_tile);
    }
    for (int sl = kLoTmaBits - 2; sl >= 0; sl -= 2) {      // DIF: stages 9..0, two at a time
      lo_stage4<false>(sm, tw_inv, sl);
      __syncthreads();
    }
    Fr* x = tile_ptr(t);
    const Fr* sc = scale + ((size_t)(t & ((1u << tile_bits) - 1)) << kLoTmaBits);
    for (uint32_t l = threadIdx.x; l < kLoTmaTile; l += blockDim.x) {
      Fr v = sm_load(sm, kLoPlane, l);
      sm_store(sm, kLoPlane, l, fp_mul(v, g_load(sc + l)));
    }
    __syncthreads();
    for (int sl = 0; sl < kLoTmaBits; sl += 2) {           // DIT: stages 0..9
      lo_stage4<true>(sm, tw_fwd, sl);
      __syncthreads();
    }
    for (uint32_t l = threadIdx.x; l < kLoTmaTile; l += blockDim.x) g_store(x + l, sm_load(sm, kLoPlane, l));
    __syncthreads();               // compute tile free for the next repack
  }
}

__global__ void bitrev_permute_kernel(const Fr* __restrict__ in, Fr* __restrict__ out, int log_n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ((size_t)1 << log_n)) return;
  uint32_t j = log_n ? (__brev((uint32_t)i) >> (32 - log_n)) : 0;
  g_store(out + j, g_load(in + i));
}

__global__ void scale_const_kernel(Fr* __restrict__ data, const Fr* __restrict__ k, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  g_store(data + i, fp_mul(g_load(data + i), g_load(k)));
}

__global__ void join_abc_kernel(const Fr* __restrict__ a, const Fr* __restrict__ b, const Fr* __restrict__ c,
                                Fr* __restrict__ h, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr t = fp_sub(fp_mul(g_load(a + i), g_load(b + i)), g_load(c + i));
  g_store(h + i, fp_from_mont(t));
}

// ---------------------------------------------------------------------------------------------- host side
static Fr host_fr_from_u64(uint64_t x) {
  Fr t = Fr::zero();
  t.v[0] = (uint32_t)x;
  t.v[1] = (uint32_t)(x >> 32);
  return fp_to_mont(t);
}

// w[k]: primitive 2^k-th root of unity, ffjavascript convention (nqr = 5, w[28] = 5^((r-1)/2^28), w[k-1] = w[k]^2).
Fr host_fr_root(int k) {
  uint32_t e[8];
  for (int i = 0; i < 8; i++) e[i] = FrParams::mod(i);
  e[0] -= 1;
  // e >>= 28
  uint32_t t[8];
  for (int i = 0; i < 8; i++) {
    uint64_t lo = e[i] >> 28;
    uint64_t hi = (i + 1 < 8) ? ((uint64_t)e[i + 1] << 4) : 0;
    t[i] = (uint32_t)(lo | hi);
  }
  Fr w = fp_pow(host_fr_from_u64(5), t);
  for (int i = 28; i > k; i--) w = fp_sqr(w);
  return w;
}

static size_t pass_smem_bytes(int ns, int cb) {
  size_t tile = (size_t)1 << (ns + cb);
  return 8 * (tile + (tile >> 5) + 1) * sizeof(uint32_t);
}

// Function attributes are per device: called from ntt_domain_create, i.e. once per domain per device.
static void ensure_smem_attrs() {
  int mx = (int)pass_smem_bytes(kMaxPassBits, 1);
  NZCP_CUDA(cudaFuncSetAttribute(ntt_pass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
  NZCP_CUDA(cudaFuncSetAttribute(ntt_pass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
  NZCP_CUDA(cudaFuncSetAttribute(ntt_fused_lo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
  NZCP_CUDA(cudaFuncSetAttribute(ntt_fused_lo_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLoTmaSmem));
}

void ntt_domain_create(NttDomain* d, int log_n, cudaStream_t st) {
  if (log_n < 1 || log_n > 27) throw std::runtime_error("ntt: unsupported domain size");
  ensure_smem_attrs();
  d->log_n = log_n;
  size_t n = (size_t)1 << log_n;
  std::vector<Fr> fwd(n / 2), inv(n / 2), scale(n);
  Fr w = host_fr_root(log_n);
  Fr winv = fp_inv(w);
  Fr a = Fr::one(), b = Fr::one();
  for (size_t j = 0; j < n / 2; j++) {
    fwd[j] = a;
    inv[j] = b;
    a = fp_mul(a, w);
    b = fp_mul(b, winv);
  }
  Fr ninv = fp_inv(host_fr_from_u64(n));
  Fr inc = (log_n == 28) ? host_fr_from_u64(25) : host_fr_root(log_n + 1);  // snarkjs: Fr.shift when power == Fr.s
  Fr k = ninv;
  for (size_t j = 0; j < n; j++) {
    uint32_t p = 0;
    for (int bit = 0; bit < log_n; bit++) p |= ((j >> bit) & 1) << (log_n - 1 - bit);
    scale[p] = k;
    k = fp_mul(k, inc);
  }
  if (log_n >= kLoTmaBits) {   // compact, padded twiddle tables of the TMA-staged low pass: entry j = w^(+-j * n / 1024)
    std::vector<unsigned char> pf(kLoTwBytes, 0), pi(kLoTwBytes, 0);
    for (uint32_t j = 0; j < kLoTwEntries; j++) {
      memcpy(pf.data() + tw_pad_off(j), &fwd[(size_t)j << (log_n - kLoTmaBits)], sizeof(Fr));
      memcpy(pi.data() + tw_pad_off(j), &inv[(size_t)j << (log_n - kLoTmaBits)], sizeof(Fr));
    }
    d->tw_lo_fwd = d->res.device<unsigned char>(kLoTwBytes);
    d->tw_lo_inv = d->res.device<unsigned char>(kLoTwBytes);
    NZCP_CUDA(cudaMemcpy(d->tw_lo_fwd, pf.data(), kLoTwBytes, cudaMemcpyHostToDevice));
    NZCP_CUDA(cudaMemcpy(d->tw_lo_inv, pi.data(), kLoTwBytes, cudaMemcpyHostToDevice));
  }
  d->tw_fwd = d->res.device<Fr>(n / 2);
  d->tw_inv = d->res.device<Fr>(n / 2);
  d->coset_scale = d->res.device<Fr>(n);
  d->ninv_scale = d->res.device<Fr>(1);
  NZCP_CUDA(cudaMemcpyAsync(d->tw_fwd, fwd.data(), (n / 2) * sizeof(Fr), cudaMemcpyHostToDevice, st));
  NZCP_CUDA(cudaMemcpyAsync(d->tw_inv, inv.data(), (n / 2) * sizeof(Fr), cudaMemcpyHostToDevice, st));
  NZCP_CUDA(cudaMemcpyAsync(d->coset_scale, scale.data(), n * sizeof(Fr), cudaMemcpyHostToDevice, st));
  NZCP_CUDA(cudaMemcpyAsync(d->ninv_scale, &ninv, sizeof(Fr), cudaMemcpyHostToDevice, st));
  NZCP_CUDA(cudaStreamSynchronize(st));
}

// Split bits [lo_bits, log_n) into hi passes of <= kMaxPassBits stages each.
static std::vector<std::pair<int, int>> hi_passes(int log_n, int lo_bits) {
  std::vector<std::pair<int, int>> v;  // (lo, ns)
  int rem = log_n - lo_bits;
  if (rem <= 0) return v;
  int np = (rem + kMaxPassBits - 1) / kMaxPassBits;
  int lo = lo_bits;
  for (int i = 0; i < np; i++) {
    int ns = rem / np + (i < rem % np ? 1 : 0);
    v.push_back({lo, ns});
    lo += ns;
  }
  return v;
}

template <bool DIT>
static void launch_pass(Fr* data, const Fr* tw, int log_n, int lo, int ns, int batch, cudaStream_t st) {
  // adjacent columns per tile row: as many as keep the tile at 2^(kMaxPassBits+1) elements, so short passes (the split
  // of 11..19 high bits at 2^21..2^24) still fill the block and read 2^cb * 32 contiguous bytes per row
  int cb = kMaxPassBits + 1 - ns;
  if (cb > lo) cb = lo;
  if (cb < 0) cb = 0;
  dim3 grid(1u << (log_n - ns - cb), batch);
  ntt_pass_kernel<DIT><<<grid, kNttThreads, pass_smem_bytes(ns, cb), st>>>(data, tw, log_n, lo, ns, cb);
  NZCP_LAUNCH_CHECK();
}

void ntt_coset_pipeline(const NttDomain& d, Fr* data, int batch, cudaStream_t st) {
  int lo_bits = d.log_n < kMaxPassBits ? d.log_n : kMaxPassBits;
  auto hp = hi_passes(d.log_n, lo_bits);
  for (int i = (int)hp.size() - 1; i >= 0; i--)
    launch_pass<false>(data, d.tw_inv, d.log_n, hp[i].first, hp[i].second, batch, st);
  if (g_tune_ntt_tma.load() && lo_bits == kLoTmaBits && d.tw_lo_fwd) {
    const uint32_t n_tiles = (uint32_t)batch << (d.log_n - kLoTmaBits);
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const uint32_t grid_tma = n_tiles < (uint32_t)(2 * sms) ? n_tiles : (uint32_t)(2 * sms);   // persistent: two blocks per SM
    ntt_fused_lo_tma_kernel<<<grid_tma, kNttThreads, kLoTmaSmem, st>>>(data, d.tw_lo_inv, d.tw_lo_fwd, d.coset_scale, d.log_n,
                                                                       n_tiles);
  } else {
    dim3 grid(1u << (d.log_n - lo_bits), batch);
    ntt_fused_lo_kernel<<<grid, kNttThreads, pass_smem_bytes(lo_bits, 0), st>>>(data, d.tw_inv, d.tw_fwd, d.coset_scale,
                                                                                d.log_n, lo_bits);
  }
  NZCP_LAUNCH_CHECK();
  for (size_t i = 0; i < hp.size(); i++) launch_pass<true>(data, d.tw_fwd, d.log_n, hp[i].first, hp[i].second, batch, st);
}

static void ntt_natural(const NttDomain& d, Fr* data, Fr* tmp, const Fr* tw, cudaStream_t st) {
  size_t n = (size_t)1 << d.log_n;
  bitrev_permute_kernel<<<div_up(n, 256), 256, 0, st>>>(data, tmp, d.log_n);
  NZCP_LAUNCH_CHECK();
  int lo_bits = d.log_n < kMaxPassBits ? d.log_n : kMaxPassBits;
  launch_pass<true>(tmp, tw, d.log_n, 0, lo_bits, 1, st);
  auto hp = hi_passes(d.log_n, lo_bits);
  for (size_t i = 0; i < hp.size(); i++) launch_pass<true>(tmp, tw, d.log_n, hp[i].first, hp[i].second, 1, st);
  NZCP_CUDA(cudaMemcpyAsync(data, tmp, n * sizeof(Fr), cudaMemcpyDeviceToDevice, st));
}

void ntt_forward(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st) { ntt_natural(d, data, tmp, d.tw_fwd, st); }

void ntt_inverse(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st) {
  ntt_natural(d, data, tmp, d.tw_inv, st);
  size_t n = (size_t)1 << d.log_n;
  scale_const_kernel<<<div_up(n, 256), 256, 0, st>>>(data, d.ninv_scale, n);
  NZCP_LAUNCH_CHECK();
}

void ntt_join_abc(const Fr* a, const Fr* b, const Fr* c, Fr* h, size_t n, cudaStream_t st) {
  join_abc_kernel<<<div_up(n, 256), 256, 0, st>>>(a, b, c, h, n);
  NZCP_LAUNCH_CHECK();
}

}  // namespace nzcp
