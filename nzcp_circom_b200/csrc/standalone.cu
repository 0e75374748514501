// Stand-alone entry points: NTT / MSM sweeps (BASELINE.json config 4) and the device self-tests the parity suite uses.
// Each call allocates, runs, times with CUDA events on the launching stream, and frees -- they are measurement and
// test hooks, not the proving path (that is prover.cu, which keeps everything resident).
#include <memory>

#include "api_util.cuh"
#include "msm_pair.cuh"

namespace nzcp {

extern std::atomic<int> g_tune_rounds;                   // msm.cu
extern std::atomic<int> g_tune_pair_stage;
extern std::atomic<int> g_tune_pair_k[kMsmMaxRounds];
extern std::atomic<int> g_tune_rounds_w, g_tune_rounds_h;

struct DevBuf {
  void* p = nullptr;
  explicit DevBuf(size_t bytes) { NZCP_CUDA(cudaMalloc(&p, bytes ? bytes : 16)); }
  ~DevBuf() { cudaFree(p); }
  template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

struct Timer {
  cudaEvent_t a, b;
  cudaStream_t st;
  explicit Timer(cudaStream_t s) : st(s) {
    NZCP_CUDA(cudaEventCreate(&a));
    NZCP_CUDA(cudaEventCreate(&b));
    NZCP_CUDA(cudaEventRecord(a, st));
  }
  float stop() {
    float ms = 0;
    NZCP_CUDA(cudaEventRecord(b, st));
    NZCP_CUDA(cudaEventSynchronize(b));
    NZCP_CUDA(cudaEventElapsedTime(&ms, a, b));
    return ms;
  }
  ~Timer() {
    cudaEventDestroy(a);
    cudaEventDestroy(b);
  }
};

// ------------------------------------------------------------------------------------------------ self-test kernels
template <class P>
__global__ void field_op_kernel(int op, const Fp<P>* a, const Fp<P>* b, Fp<P>* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp<P> x = a[i], y = b[i], r;
  switch (op) {
    case 0: r = fp_mul(x, y); break;
    case 1: r = fp_add(x, y); break;
    case 2: r = fp_sub(x, y); break;
    case 3: r = fp_mul_portable(x, y); break;
    case 4: r = fp_add_portable(x, y); break;
    case 5: r = fp_sub_portable(x, y); break;
    case 6: r = fp_inv_fast(x); break;                       // safegcd (b ignored)
    default: r = x.is_zero() ? x : fp_inv(x); break;         // 7: Fermat ladder
  }
  out[i] = r;
}

// Exercises madd / add / dbl / to_affine on the device: out[i] = affine( (a_i + b_i) + 2*a_i - b_i ) = 3 * a_i.
template <class F>
__global__ void curve_op_kernel(const Affine<F>* a, const Affine<F>* b, Affine<F>* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  XYZZ<F> acc = XYZZ<F>::inf();
  xyzz_madd(acc, a[i], false);
  xyzz_madd(acc, b[i], false);
  XYZZ<F> d = xyzz_dbl(XYZZ<F>::from_affine(a[i]));
  xyzz_add(acc, d);
  xyzz_madd(acc, b[i], true);
  out[i] = xyzz_to_affine(acc);
}

// Record sizes (bytes) of nzcp_arith_op, per op: in, out.
static const int kArithIn[10] = {64, 64, 128, 128, 128, 128, 64, 64, 64, 256};
static const int kArithOut[10] = {64, 32, 32, 32, 64, 64, 64, 64, 64, 64};

// One case per thread through the exact device functions the kernels call (the lazy-reduction bodies, the non-inlined
// Fq2 product / square, the device inversions), so the suite can pin them limb for limb against a big-integer reference.
__global__ void arith_op_kernel(int op, const uint32_t* in, uint32_t* out, size_t n, int in_w, int out_w) {
#if defined(__CUDA_ARCH__)   // fp_mul_wide / fp_redc_wide exist only in the device pass
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* x = in + i * in_w;
  uint32_t* y = out + i * out_w;
  auto fq = [&](int k) { return *reinterpret_cast<const Fq*>(x + 8 * k); };
  auto fq2 = [&](int k) { return Fq2{fq(2 * k), fq(2 * k + 1)}; };
  Fq r1;
  Fq2 r2;
  switch (op) {
    case 0: fp_mul_wide(y, x, x + 8); return;
    case 1: fp_redc_wide<FqParams>(y, x); return;
    case 2: r1 = f_mulsub(fq(0), fq(1), fq(2), fq(3)); break;
    case 3: r1 = fp_sub(fp_mul(fq(0), fq(1)), fp_mul(fq(2), fq(3))); break;
    case 4: r2 = f_mul(fq2(0), fq2(1)); break;
    case 5: r2 = f2_mul_inline(fq2(0), fq2(1)); break;
    case 6: r2 = f_sqr(fq2(0)); break;
    case 7: r2 = f_inv(fq2(0)); break;
    case 8: r2 = f_inv_fast(fq2(0)); break;
    default: r2 = f_mulsub(fq2(0), fq2(1), fq2(2), fq2(3)); break;
  }
  if (op <= 3) {
    *reinterpret_cast<Fq*>(y) = r1;
  } else {
    *reinterpret_cast<Fq*>(y) = r2.c0;
    *reinterpret_cast<Fq*>(y + 8) = r2.c1;
  }
#endif
}

// XYZZ group law on records: 0 add(a, b), 1 madd(a, affine b), 2 madd(a, -affine b), 3 dbl(a), 4 to_affine(a).
template <class F>
__global__ void xyzz_op_kernel(int op, const XYZZ<F>* a, const void* b, void* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  XYZZ<F> acc = a[i];
  switch (op) {
    case 0: xyzz_add(acc, reinterpret_cast<const XYZZ<F>*>(b)[i]); break;
    case 1: xyzz_madd(acc, reinterpret_cast<const Affine<F>*>(b)[i], false); break;
    case 2: xyzz_madd(acc, reinterpret_cast<const Affine<F>*>(b)[i], true); break;
    case 3: acc = xyzz_dbl(acc); break;
    default: reinterpret_cast<Affine<F>*>(out)[i] = xyzz_to_affine(acc); return;
  }
  reinterpret_cast<XYZZ<F>*>(out)[i] = acc;
}

template <class F>
static void run_xyzz_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  const size_t xs = sizeof(XYZZ<F>), as = sizeof(Affine<F>);
  const size_t bs = op == 0 ? xs : (op <= 2 ? as : 0), os = op == 4 ? as : xs;
  DevBuf da(n * xs), db(n * bs), dout(n * os);
  NZCP_CUDA(cudaMemcpy(da.p, a, n * xs, cudaMemcpyHostToDevice));
  if (bs) NZCP_CUDA(cudaMemcpy(db.p, b, n * bs, cudaMemcpyHostToDevice));
  xyzz_op_kernel<F><<<div_up(n, 128), 128>>>(op, da.as<XYZZ<F>>(), db.p, dout.p, n);
  NZCP_LAUNCH_CHECK();
  NZCP_CUDA(cudaMemcpy(out, dout.p, n * os, cudaMemcpyDeviceToHost));
}

template <class P>
static uint32_t selftest_field(uint64_t seed, uint32_t n) {
  std::vector<Fp<P>> a(n), b(n);
  uint64_t s = seed * 0x9E3779B97F4A7C15ull + 99;
  auto next = [&]() {
    s += 0x9E3779B97F4A7C15ull;
    uint64_t z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  };
  for (uint32_t i = 0; i < n; i++) {
    for (int k = 0; k < 4; k++) {
      uint64_t u = next(), v = next();
      a[i].v[2 * k] = (uint32_t)u; a[i].v[2 * k + 1] = (uint32_t)(u >> 32);
      b[i].v[2 * k] = (uint32_t)v; b[i].v[2 * k + 1] = (uint32_t)(v >> 32);
    }
    a[i].v[7] &= 0x1fffffffu;
    b[i].v[7] &= 0x1fffffffu;
  }
  // edge values: 0, 1, p-1, R mod p
  if (n >= 8) {
    a[0] = Fp<P>::zero(); b[0] = Fp<P>::zero();
    a[1] = Fp<P>::one(); b[1] = Fp<P>::one();
    a[2] = fp_sub_portable(Fp<P>::zero(), Fp<P>::one()); b[2] = a[2];
    a[3] = a[2]; b[3] = Fp<P>::one();
    a[4] = Fp<P>::zero(); a[4].v[0] = 1; b[4] = a[2];
    a[5] = fp_sub_portable(Fp<P>::modulus(), a[4]); b[5] = a[5];  // p-1 (plain) twice
    a[6] = a[5]; b[6] = Fp<P>::zero();
    a[7] = Fp<P>::zero(); b[7] = a[5];
  }
  DevBuf da(n * 32), db(n * 32), dout(n * 32);
  NZCP_CUDA(cudaMemcpy(da.p, a.data(), n * 32, cudaMemcpyHostToDevice));
  NZCP_CUDA(cudaMemcpy(db.p, b.data(), n * 32, cudaMemcpyHostToDevice));
  uint32_t bad = 0;
  std::vector<Fp<P>> out(n);
  for (int op = 0; op < 6; op++) {
    field_op_kernel<P><<<div_up(n, 128), 128>>>(op, da.as<Fp<P>>(), db.as<Fp<P>>(), dout.as<Fp<P>>(), n);
    NZCP_LAUNCH_CHECK();
    NZCP_CUDA(cudaMemcpy(out.data(), dout.p, n * 32, cudaMemcpyDeviceToHost));
    for (uint32_t i = 0; i < n; i++) {
      Fp<P> e = (op % 3 == 0) ? fp_mul_portable(a[i], b[i]) : (op % 3 == 1) ? fp_add_portable(a[i], b[i]) : fp_sub_portable(a[i], b[i]);
      if (e != out[i]) bad++;
    }
  }
  return bad;
}

template <class F>
static uint32_t selftest_curve(const Affine<F>& gen, uint64_t seed, uint32_t n) {
  std::vector<Affine<F>> a(n), b(n), out(n);
  XYZZ<F> g = XYZZ<F>::from_affine(gen);
  XYZZ<F> p = g, q = xyzz_dbl(g);
  for (uint32_t k = 0; k < (seed & 7); k++) xyzz_add(p, g);
  for (uint32_t i = 0; i < n; i++) {
    xyzz_add(p, q);  // distinct multiples of g
    q = xyzz_dbl(q);
    a[i] = xyzz_to_affine(p);
    b[i] = xyzz_to_affine(q);
  }
  if (n >= 4) {
    b[0] = a[0];                                   // madd hits the doubling branch
    b[1] = Affine<F>{a[1].x, f_neg(a[1].y)};       // madd hits the cancellation branch
  }
  DevBuf da(n * sizeof(Affine<F>)), db(n * sizeof(Affine<F>)), dout(n * sizeof(Affine<F>));
  NZCP_CUDA(cudaMemcpy(da.p, a.data(), n * sizeof(Affine<F>), cudaMemcpyHostToDevice));
  NZCP_CUDA(cudaMemcpy(db.p, b.data(), n * sizeof(Affine<F>), cudaMemcpyHostToDevice));
  curve_op_kernel<F><<<div_up(n, 64), 64>>>(da.as<Affine<F>>(), db.as<Affine<F>>(), dout.as<Affine<F>>(), n);
  NZCP_LAUNCH_CHECK();
  NZCP_CUDA(cudaMemcpy(out.data(), dout.p, n * sizeof(Affine<F>), cudaMemcpyDeviceToHost));
  uint32_t bad = 0;
  for (uint32_t i = 0; i < n; i++) {
    XYZZ<F> e = XYZZ<F>::from_affine(a[i]);
    XYZZ<F> d = xyzz_dbl(e);
    xyzz_add(e, d);  // 3a
    Affine<F> ea = xyzz_to_affine(e);
    if (!(ea.x == out[i].x) || !(ea.y == out[i].y)) bad++;
  }
  return bad;
}


// ------------------------------------------------------------------------------------------------ integer-pipe peak
// Microbenchmarks behind the MSM / NTT roofline denominator (MEASURED_PEAKS.json has no integer-pipe figure):
//   mode 0: mad.wide.u32 with loop-invariant multiplicands -- ptxas strength-reduces it to IADD3/IADD3.X pairs, so this
//           measures the 64-bit add rate, NOT the multiplier (kept as a warning; the IMAD.WIDE rate is modes 3..5)
//   mode 1: independent mad.lo.u32 chains (IMAD)
//   mode 2: fp_mul<Fq> chains, 2 independent products per thread (what a kernel that did nothing else would reach)
template <int mode>
__global__ void __launch_bounds__(256) intpipe_kernel(int iters, uint32_t seed, uint32_t* sink) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 0) {
    unsigned long long a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7;
    uint32_t x = seed | 1, y = seed + t;
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        asm volatile("mad.wide.u32 %0, %8, %9, %0;\n\tmad.wide.u32 %1, %8, %9, %1;\n\tmad.wide.u32 %2, %8, %9, %2;\n\t"
                     "mad.wide.u32 %3, %8, %9, %3;\n\tmad.wide.u32 %4, %8, %9, %4;\n\tmad.wide.u32 %5, %8, %9, %5;\n\t"
                     "mad.wide.u32 %6, %8, %9, %6;\n\tmad.wide.u32 %7, %8, %9, %7;"
                     : "+l"(a0), "+l"(a1), "+l"(a2), "+l"(a3), "+l"(a4), "+l"(a5), "+l"(a6), "+l"(a7)
                     : "r"(x), "r"(y));
      }
    }
    unsigned long long s = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
    if (s == 0x123456789ull) sink[0] = (uint32_t)s;
  } else if (mode == 1) {
    uint32_t a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7;
    uint32_t x = seed | 1, y = seed + t;
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        asm volatile("mad.lo.u32 %0, %8, %9, %0;\n\tmad.lo.u32 %1, %8, %9, %1;\n\tmad.lo.u32 %2, %8, %9, %2;\n\t"
                     "mad.lo.u32 %3, %8, %9, %3;\n\tmad.lo.u32 %4, %8, %9, %4;\n\tmad.lo.u32 %5, %8, %9, %5;\n\t"
                     "mad.lo.u32 %6, %8, %9, %6;\n\tmad.lo.u32 %7, %8, %9, %7;"
                     : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                     : "r"(x), "r"(y));
      }
    }
    uint32_t s = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
    if (s == 0x12345678u) sink[0] = s;
  } else if (mode >= 3 && mode <= 8) {
    // carry-chain variants: which form of IMAD.WIDE pays the half-rate penalty?
    //   3: 2-long chains  mad.lo.cc / madc.hi           (IMAD.WIDE with no external carry)
    //   4: 4-long chains  lo.cc hi.cc lo.cc hi          (1 carry-out + 1 carry-in)
    //   5: 8-long chains                                (1 carry-out + 2 in/out + 1 carry-in)
    //   6: mode 0 plus an independent add.cc/addc chain per IMAD (do the fma and alu pipes overlap?)
    uint32_t a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7;
    uint32_t c0 = t, c1 = t, c2 = t, c3 = t, c4 = t, c5 = t, c6 = t, c7 = t;
    uint32_t x = seed | 1, y = seed + t;
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        if (mode == 3) {
          asm volatile("mad.lo.cc.u32 %0, %8, %9, %0;\n\tmadc.hi.u32 %1, %8, %9, %1;\n\t"
                       "mad.lo.cc.u32 %2, %8, %9, %2;\n\tmadc.hi.u32 %3, %8, %9, %3;\n\t"
                       "mad.lo.cc.u32 %4, %8, %9, %4;\n\tmadc.hi.u32 %5, %8, %9, %5;\n\t"
                       "mad.lo.cc.u32 %6, %8, %9, %6;\n\tmadc.hi.u32 %7, %8, %9, %7;"
                       : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                       : "r"(x), "r"(y));
        } else if (mode == 4) {
          asm volatile("mad.lo.cc.u32 %0, %8, %9, %0;\n\tmadc.hi.cc.u32 %1, %8, %9, %1;\n\t"
                       "madc.lo.cc.u32 %2, %8, %9, %2;\n\tmadc.hi.u32 %3, %8, %9, %3;\n\t"
                       "mad.lo.cc.u32 %4, %8, %9, %4;\n\tmadc.hi.cc.u32 %5, %8, %9, %5;\n\t"
                       "madc.lo.cc.u32 %6, %8, %9, %6;\n\tmadc.hi.u32 %7, %8, %9, %7;"
                       : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                       : "r"(x), "r"(y));
        } else if (mode == 5) {
          asm volatile("mad.lo.cc.u32 %0, %8, %9, %0;\n\tmadc.hi.cc.u32 %1, %8, %9, %1;\n\t"
                       "madc.lo.cc.u32 %2, %8, %9, %2;\n\tmadc.hi.cc.u32 %3, %8, %9, %3;\n\t"
                       "madc.lo.cc.u32 %4, %8, %9, %4;\n\tmadc.hi.cc.u32 %5, %8, %9, %5;\n\t"
                       "madc.lo.cc.u32 %6, %8, %9, %6;\n\tmadc.hi.u32 %7, %8, %9, %7;"
                       : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                       : "r"(x), "r"(y));
        } else if (mode == 7) {   // 8 add-with-carry instructions per step, no multiplies
          asm volatile("add.cc.u32 %0, %0, %8;\n\taddc.cc.u32 %1, %1, %8;\n\taddc.cc.u32 %2, %2, %8;\n\taddc.u32 %3, %3, %8;\n\t"
                       "add.cc.u32 %4, %4, %8;\n\taddc.cc.u32 %5, %5, %8;\n\taddc.cc.u32 %6, %6, %8;\n\taddc.u32 %7, %7, %8;"
                       : "+r"(c0), "+r"(c1), "+r"(c2), "+r"(c3), "+r"(c4), "+r"(c5), "+r"(c6), "+r"(c7)
                       : "r"(y));
        } else if (mode == 8) {   // 4 plain mad.wide + 8 add-with-carry
          unsigned long long w0 = ((unsigned long long)a1 << 32) | a0, w1 = ((unsigned long long)a3 << 32) | a2;
          unsigned long long w2 = ((unsigned long long)a5 << 32) | a4, w3 = ((unsigned long long)a7 << 32) | a6;
          asm volatile("mad.wide.u32 %0, %4, %5, %0;\n\tmad.wide.u32 %1, %4, %5, %1;\n\t"
                       "mad.wide.u32 %2, %4, %5, %2;\n\tmad.wide.u32 %3, %4, %5, %3;"
                       : "+l"(w0), "+l"(w1), "+l"(w2), "+l"(w3) : "r"(c0), "r"(c4));
          a0 = (uint32_t)w0; a1 = (uint32_t)(w0 >> 32); a2 = (uint32_t)w1; a3 = (uint32_t)(w1 >> 32);
          a4 = (uint32_t)w2; a5 = (uint32_t)(w2 >> 32); a6 = (uint32_t)w3; a7 = (uint32_t)(w3 >> 32);
          asm volatile("add.cc.u32 %0, %0, %8;\n\taddc.cc.u32 %1, %1, %8;\n\taddc.cc.u32 %2, %2, %8;\n\taddc.u32 %3, %3, %8;\n\t"
                       "add.cc.u32 %4, %4, %8;\n\taddc.cc.u32 %5, %5, %8;\n\taddc.cc.u32 %6, %6, %8;\n\taddc.u32 %7, %7, %8;"
                       : "+r"(c0), "+r"(c1), "+r"(c2), "+r"(c3), "+r"(c4), "+r"(c5), "+r"(c6), "+r"(c7)
                       : "r"(y));
        } else {
          asm volatile("mad.lo.cc.u32 %0, %8, %9, %0;\n\tmadc.hi.u32 %1, %8, %9, %1;\n\t"
                       "mad.lo.cc.u32 %2, %8, %9, %2;\n\tmadc.hi.u32 %3, %8, %9, %3;\n\t"
                       "mad.lo.cc.u32 %4, %8, %9, %4;\n\tmadc.hi.u32 %5, %8, %9, %5;\n\t"
                       "mad.lo.cc.u32 %6, %8, %9, %6;\n\tmadc.hi.u32 %7, %8, %9, %7;"
                       : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                       : "r"(x), "r"(y));
          asm volatile("add.cc.u32 %0, %0, %8;\n\taddc.cc.u32 %1, %1, %8;\n\taddc.cc.u32 %2, %2, %8;\n\taddc.u32 %3, %3, %8;\n\t"
                       "add.cc.u32 %4, %4, %8;\n\taddc.cc.u32 %5, %5, %8;\n\taddc.cc.u32 %6, %6, %8;\n\taddc.u32 %7, %7, %8;"
                       : "+r"(c0), "+r"(c1), "+r"(c2), "+r"(c3), "+r"(c4), "+r"(c5), "+r"(c6), "+r"(c7)
                       : "r"(y));
        }
      }
    }
    uint32_t sx = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7 ^ c0 ^ c1 ^ c2 ^ c3 ^ c4 ^ c5 ^ c6 ^ c7;
    if (sx == 0x12345678u) sink[0] = sx;
  } else {
    Fq a = Fq::one(), b = Fq::r2(), c = Fq::one();
    a.v[0] ^= t & 0xffff;
    c.v[1] ^= (seed + t) & 0xffff;
    for (int i = 0; i < iters; i++) {
      a = fp_mul(a, b);
      c = fp_mul(c, b);
    }
    if ((a.v[0] ^ c.v[0]) == 0x12345678u) sink[0] = a.v[1];
  }
}

// Pipe-overlap probes behind DESIGN.md's cost model of the multiplier (which instructions issue "for free" next to
// IMAD.WIDE, and whether the FP64 pipe is a second multiplier worth building a 52-bit-limb product on):
//   0: fma.rn.f64, 8 independent chains                 -> DFMA/s
//   1: 4 IMAD.WIDE (2-long carry chains) + 4 DFMA        -> IMAD.WIDE/s with the FP64 pipe busy beside it
//   2: 4 IMAD.WIDE + 8 lop3 (majority)                      -> IMAD.WIDE/s next to plain ALU work
//   3: 4 IMAD.WIDE + 8 add.u32 (no carry)                -> IMAD.WIDE/s next to carry-free adds
template <int mode>
__global__ void __launch_bounds__(256) pipeprobe_kernel(int iters, uint32_t seed, uint32_t* sink) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7;
  uint32_t c0 = t, c1 = t ^ 1, c2 = t ^ 2, c3 = t ^ 3, c4 = t ^ 4, c5 = t ^ 5, c6 = t ^ 6, c7 = t ^ 7;
  double d0 = t, d1 = t + 0.5, d2 = t + 1.5, d3 = t + 2.5, d4 = t + 3.5, d5 = t + 4.5, d6 = t + 5.5, d7 = t + 6.5;
  const double fx = 1.0 + 1e-9 * (seed & 3), fy = 1e-3 * (1 + (t & 1));
  uint32_t x = seed | 1, y = seed + t;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (mode == 0) {
        asm volatile("fma.rn.f64 %0, %0, %8, %9;\n\tfma.rn.f64 %1, %1, %8, %9;\n\tfma.rn.f64 %2, %2, %8, %9;\n\t"
                     "fma.rn.f64 %3, %3, %8, %9;\n\tfma.rn.f64 %4, %4, %8, %9;\n\tfma.rn.f64 %5, %5, %8, %9;\n\t"
                     "fma.rn.f64 %6, %6, %8, %9;\n\tfma.rn.f64 %7, %7, %8, %9;"
                     : "+d"(d0), "+d"(d1), "+d"(d2), "+d"(d3), "+d"(d4), "+d"(d5), "+d"(d6), "+d"(d7)
                     : "d"(fx), "d"(fy));
      } else {
        asm volatile("mad.lo.cc.u32 %0, %8, %9, %0;\n\tmadc.hi.u32 %1, %8, %9, %1;\n\t"
                     "mad.lo.cc.u32 %2, %8, %9, %2;\n\tmadc.hi.u32 %3, %8, %9, %3;\n\t"
                     "mad.lo.cc.u32 %4, %8, %9, %4;\n\tmadc.hi.u32 %5, %8, %9, %5;\n\t"
                     "mad.lo.cc.u32 %6, %8, %9, %6;\n\tmadc.hi.u32 %7, %8, %9, %7;"
                     : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
                     : "r"(x), "r"(y));
        if (mode == 1) {
          asm volatile("fma.rn.f64 %0, %0, %4, %5;\n\tfma.rn.f64 %1, %1, %4, %5;\n\tfma.rn.f64 %2, %2, %4, %5;\n\t"
                       "fma.rn.f64 %3, %3, %4, %5;"
                       : "+d"(d0), "+d"(d1), "+d"(d2), "+d"(d3) : "d"(fx), "d"(fy));
        } else if (mode == 2) {
          // majority(c_k, c_k+1, y): a non-linear 3-input LUT ptxas cannot fold across the ring
          asm volatile("lop3.b32 %0, %0, %1, %8, 0xE8;\n\tlop3.b32 %1, %1, %2, %8, 0xE8;\n\t"
                       "lop3.b32 %2, %2, %3, %8, 0xE8;\n\tlop3.b32 %3, %3, %4, %8, 0xE8;\n\t"
                       "lop3.b32 %4, %4, %5, %8, 0xE8;\n\tlop3.b32 %5, %5, %6, %8, 0xE8;\n\t"
                       "lop3.b32 %6, %6, %7, %8, 0xE8;\n\tlop3.b32 %7, %7, %0, %8, 0xE8;"
                       : "+r"(c0), "+r"(c1), "+r"(c2), "+r"(c3), "+r"(c4), "+r"(c5), "+r"(c6), "+r"(c7) : "r"(y));
        } else {
          asm volatile("add.u32 %0, %0, %1;\n\tadd.u32 %1, %1, %2;\n\tadd.u32 %2, %2, %3;\n\tadd.u32 %3, %3, %4;\n\t"
                       "add.u32 %4, %4, %5;\n\tadd.u32 %5, %5, %6;\n\tadd.u32 %6, %6, %7;\n\tadd.u32 %7, %7, %0;"
                       : "+r"(c0), "+r"(c1), "+r"(c2), "+r"(c3), "+r"(c4), "+r"(c5), "+r"(c6), "+r"(c7));
        }
      }
    }
  }
  uint32_t sx = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7 ^ c0 ^ c1 ^ c2 ^ c3 ^ c4 ^ c5 ^ c6 ^ c7;
  double sd = d0 + d1 + d2 + d3 + d4 + d5 + d6 + d7;
  if (sx == 0x12345678u || sd == 0.123456) sink[0] = sx;
}


// ------------------------------------------------------------------------------------------------ host simulation
// The MSM data path with the pair rounds, run on the CPU with the SAME __host__ __device__ code the kernels execute
// (msm_pair.cuh forward / invert / backward bodies, the signed-digit rule of msm_digits_*_kernel, the round plan of
// msm_round_plan_kernel restated as plain loops).  Test-only: it lets the no-GPU suite pin the index arithmetic and the
// special-pair handling of the batched-affine rounds against the oracle; nothing in the product calls it.
template <class F, int K>
static void sim_round(bool from_table, const std::vector<Affine<F>>& src, const std::vector<uint32_t>& entries,
                      const std::vector<uint32_t>& off_in, const std::vector<uint32_t>& off_out, uint32_t nb,
                      std::vector<Affine<F>>& dst, bool stage_ops) {
  const uint32_t n_out = off_out[nb];
  const uint32_t threads = pair_n_prod<K>(n_out) + 3;   // a few surplus threads, as the over-sized device grid has
  std::vector<F> scratch((size_t)threads * K), prod(threads + 40, F::one());
  std::vector<Affine<F>> ops(from_table && stage_ops ? (size_t)threads * K * 2 : 0);   // round 1: staged operands, as on the device
  Affine<F>* opsp = ops.empty() ? nullptr : ops.data();
  dst.assign(n_out ? n_out : 1, Affine<F>::inf());
  const uint32_t n_prod = pair_n_prod<K>(n_out);
  for (int phase = 0; phase < 3; phase++) {
    if (phase == 1) {
      for (uint32_t g = 0; g * 32 < n_prod + 64; g++) msm_pair_invert_body<F, 32>(g, prod.data(), n_prod);
      continue;
    }
    for (uint32_t t = 0; t < threads; t++) {
      if (from_table) {
        PairSource<F, true> ps{src.data(), entries.data(), 0};
        if (phase == 0) msm_pair_forward_body<F, true, K>(t, threads, ps, off_in.data(), off_out.data(), nb, scratch.data(), prod.data(), opsp);
        else msm_pair_backward_body<F, true, K>(t, threads, ps, off_in.data(), off_out.data(), nb, dst.data(), scratch.data(), prod.data(), opsp);
      } else {
        PairSource<F, false> ps{src.data(), nullptr, 0};
        if (phase == 0) msm_pair_forward_body<F, false, K>(t, threads, ps, off_in.data(), off_out.data(), nb, scratch.data(), prod.data());
        else msm_pair_backward_body<F, false, K>(t, threads, ps, off_in.data(), off_out.data(), nb, dst.data(), scratch.data(), prod.data());
      }
    }
  }
}

template <class F>
static XYZZ<F> host_msm_sim(const uint8_t* bases, const uint8_t* scalars, size_t n, int c, int rounds, int k) {
  const int n_windows = msm_num_windows(c);
  const uint32_t nb = 1u << (c - 1);
  std::vector<Affine<F>> table((size_t)n_windows * n + 1);
  for (size_t i = 0; i < n; i++) {
    Affine<F> p;
    memcpy(&p, bases + i * sizeof(Affine<F>), sizeof(Affine<F>));
    table[i] = p;
    for (int w = 1; w < n_windows; w++) {
      if (!p.is_inf()) {
        XYZZ<F> acc = xyzz_dbl_affine(p);
        for (int j = 1; j < c; j++) acc = xyzz_dbl(acc);
        p = xyzz_to_affine(acc);
      }
      table[(size_t)w * n + i] = p;
    }
  }
  std::vector<std::vector<uint32_t>> lists(nb);
  for (size_t i = 0; i < n; i++) {
    uint32_t sc[8];
    memcpy(sc, scalars + 32 * i, 32);
    if (fp_geq_mod<FrParams>(sc)) throw ApiError(NZCP_E_RANGE, "witness/scalar value is not a canonical field element (>= r)");
    uint32_t carry = 0;
    for (int w = 0; w < n_windows; w++) {
      const int pos = w * c;
      uint32_t d = carry;
      if (pos < 256) {
        const int idx = pos >> 5, sh = pos & 31;
        uint64_t lo = sc[idx], hi = idx + 1 < 8 ? sc[idx + 1] : 0;
        d += (uint32_t)((lo | (hi << 32)) >> sh) & ((1u << c) - 1);
      }
      uint32_t neg = 0;
      if (d > nb) {
        d = (1u << c) - d;
        neg = 1;
        carry = 1;
      } else {
        carry = 0;
      }
      if (d) lists[d - 1].push_back(((uint32_t)w * (uint32_t)n + (uint32_t)i) | (neg << 31));
    }
  }
  std::vector<uint32_t> entries;
  std::vector<std::vector<uint32_t>> off(rounds + 1, std::vector<uint32_t>(nb + 1, 0));
  for (uint32_t b = 0; b < nb; b++) {
    uint32_t len = (uint32_t)lists[b].size();
    entries.insert(entries.end(), lists[b].begin(), lists[b].end());
    for (int r = 0; r <= rounds; r++) {
      off[r][b + 1] = off[r][b] + len;
      len = (len + 1) >> 1;
    }
  }
  entries.push_back(0);
  std::vector<Affine<F>> cur, nxt;
  const bool stage = g_tune_pair_stage.load() != 0;   // "pair_stage" knob, as the device path reads it
  for (int r = 1; r <= rounds; r++) {
    const std::vector<Affine<F>>& src = r == 1 ? table : cur;
    switch (k) {
      case 4: sim_round<F, 4>(r == 1, src, entries, off[r - 1], off[r], nb, nxt, stage); break;
      case 16: sim_round<F, 16>(r == 1, src, entries, off[r - 1], off[r], nb, nxt, stage); break;
      case 32: sim_round<F, 32>(r == 1, src, entries, off[r - 1], off[r], nb, nxt, stage); break;
      case 8: sim_round<F, 8>(r == 1, src, entries, off[r - 1], off[r], nb, nxt, stage); break;
      default: throw ApiError(NZCP_E_ARG, "additions per thread must be 4, 8, 16 or 32");
    }
    cur.swap(nxt);
  }
  // XYZZ tail per bucket, then sum_v v * B_v by the running-sum rule
  XYZZ<F> run = XYZZ<F>::inf(), tot = XYZZ<F>::inf();
  for (uint32_t b = nb; b-- > 0;) {
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t j = off[rounds][b]; j < off[rounds][b + 1]; j++) {
      Affine<F> q;
      bool neg = false;
      if (rounds == 0) {
        q = table[entries[j] & 0x7fffffffu];
        neg = (entries[j] >> 31) != 0;
      } else {
        q = cur[j];
      }
      if (!q.is_inf()) xyzz_madd(acc, q, neg);
    }
    xyzz_add(run, acc);
    xyzz_add(tot, run);
  }
  return tot;
}

}  // namespace nzcp

using namespace nzcp;

static void launch_intpipe(int mode, int blocks, int threads, int it, uint32_t seed, uint32_t* sink) {
  switch (mode) {
    case 0: intpipe_kernel<0><<<blocks, threads>>>(it, seed, sink); break;
    case 1: intpipe_kernel<1><<<blocks, threads>>>(it, seed, sink); break;
    case 2: intpipe_kernel<2><<<blocks, threads>>>(it, seed, sink); break;
    case 3: intpipe_kernel<3><<<blocks, threads>>>(it, seed, sink); break;
    case 4: intpipe_kernel<4><<<blocks, threads>>>(it, seed, sink); break;
    case 5: intpipe_kernel<5><<<blocks, threads>>>(it, seed, sink); break;
    case 6: intpipe_kernel<6><<<blocks, threads>>>(it, seed, sink); break;
    case 7: intpipe_kernel<7><<<blocks, threads>>>(it, seed, sink); break;
    default: intpipe_kernel<8><<<blocks, threads>>>(it, seed, sink); break;
  }
}

extern "C" {

// Per-mode raw rates for modes 0..8 -- diagnostic.  out[m] = per-second count of: mads (0, 1), Fq products (2),
// 32x32 products (3..6), add-with-carry instructions (7), mad.wide (8: each accompanied by two add-with-carry).
int nzcp_intpipe_modes(int device, int iters, double out[10]) {
  return api_guard([&] {
    if (!out || iters < 1) throw ApiError(NZCP_E_ARG, "bad argument");
    use_device(device);
    cudaDeviceProp prop;
    NZCP_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf sink(64);
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    for (int mode = 0; mode < 9; mode++) {
      int it = mode == 2 ? (iters / 16 > 0 ? iters / 16 : 1) : iters;
      float best = 1e30f;
      for (int rep = 0; rep < 4; rep++) {
        Timer t(0);
        launch_intpipe(mode, blocks, threads, it, 12345u + rep, sink.as<uint32_t>());
        NZCP_LAUNCH_CHECK();
        float ms = t.stop();
        if (rep && ms < best) best = ms;
      }
      // modes 0,1: 64 mads per iteration; modes 3..6: 64 mad.lo/hi halves = 32 wide products per iteration
      double per_thread = mode == 2 ? 2.0 * it : (mode <= 1 || mode == 7 ? 64.0 * it : 32.0 * it);
      out[mode] = per_thread * (double)blocks * threads / (best * 1e-3);
    }
    out[9] = (double)prop.multiProcessorCount;
  });
}

/* Diagnostic: pipe-overlap probes (csrc/standalone.cu pipeprobe_kernel).  out[0] = DFMA/s alone; out[1..3] =
 * IMAD.WIDE/s with DFMA (1:1), xor (1:2), carry-free add (1:2) beside it; out[4] = DFMA/s inside probe 1. */
int nzcp_pipe_probe(int device, int iters, double out[5]) {
  return api_guard([&] {
    if (!out || iters < 1) throw ApiError(NZCP_E_ARG, "bad argument");
    use_device(device);
    cudaDeviceProp prop;
    NZCP_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf sink(64);
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    for (int mode = 0; mode < 4; mode++) {
      float best = 1e30f;
      for (int rep = 0; rep < 4; rep++) {
        Timer t(0);
        switch (mode) {
          case 0: pipeprobe_kernel<0><<<blocks, threads>>>(iters, 777u + rep, sink.as<uint32_t>()); break;
          case 1: pipeprobe_kernel<1><<<blocks, threads>>>(iters, 777u + rep, sink.as<uint32_t>()); break;
          case 2: pipeprobe_kernel<2><<<blocks, threads>>>(iters, 777u + rep, sink.as<uint32_t>()); break;
          default: pipeprobe_kernel<3><<<blocks, threads>>>(iters, 777u + rep, sink.as<uint32_t>()); break;
        }
        NZCP_LAUNCH_CHECK();
        float ms = t.stop();
        if (rep && ms < best) best = ms;
      }
      // per iteration and thread: mode 0 = 64 DFMA; modes 1..3 = 32 IMAD.WIDE (+ 32 DFMA in mode 1)
      double per_thread = (mode == 0 ? 64.0 : 32.0) * iters;
      out[mode] = per_thread * (double)blocks * threads / (best * 1e-3);
    }
    out[4] = out[1];
  });
}

int nzcp_intpipe_bench(int device, int iters, double out[4]) {
  return api_guard([&] {
    if (!out || iters < 1) throw ApiError(NZCP_E_ARG, "bad argument");
    double m[10];
    int rc = nzcp_intpipe_modes(device, iters, m);
    if (rc != NZCP_OK) throw ApiError(rc, nzcp_last_error());
    out[0] = m[3];  // IMAD.WIDE.U32 (independent 2-long carry chains; the .X forms run at the same rate)
    out[1] = m[1];  // IMAD (32-bit)
    out[2] = m[2];  // Fq Montgomery products, dependent chains
    out[3] = m[9];
  });
}

int nzcp_ntt(uint8_t* data, int log_n, int inverse, int device, float* kernel_ms) {
  return api_guard([&] {
    if (!data) throw ApiError(NZCP_E_ARG, "null argument");
    if (log_n < 1 || log_n > 27) throw ApiError(NZCP_E_ARG, "log_n out of range [1, 27]");
    use_device(device);
    size_t n = (size_t)1 << log_n;
    NttDomain dom;
    ntt_domain_create(&dom, log_n, 0);
    struct Guard { NttDomain* d; ~Guard() { ntt_domain_destroy(d); } } g{&dom};
    DevBuf d(n * 32), tmp(n * 32);
    NZCP_CUDA(cudaMemcpy(d.p, data, n * 32, cudaMemcpyHostToDevice));
    Timer t(0);
    if (inverse) ntt_inverse(dom, d.as<Fr>(), tmp.as<Fr>(), 0); else ntt_forward(dom, d.as<Fr>(), tmp.as<Fr>(), 0);
    float ms = t.stop();
    if (kernel_ms) *kernel_ms = ms;
    NZCP_CUDA(cudaMemcpy(data, d.p, n * 32, cudaMemcpyDeviceToHost));
  });
}

int nzcp_ntt_coset(uint8_t* data, int log_n, int batch, int device, float* kernel_ms) {
  return api_guard([&] {
    if (!data || batch < 1) throw ApiError(NZCP_E_ARG, "bad argument");
    if (log_n < 1 || log_n > 27) throw ApiError(NZCP_E_ARG, "log_n out of range [1, 27]");
    use_device(device);
    size_t n = (size_t)1 << log_n;
    NttDomain dom;
    ntt_domain_create(&dom, log_n, 0);
    struct Guard { NttDomain* d; ~Guard() { ntt_domain_destroy(d); } } g{&dom};
    DevBuf d(n * 32 * batch);
    NZCP_CUDA(cudaMemcpy(d.p, data, n * 32 * batch, cudaMemcpyHostToDevice));
    Timer t(0);
    ntt_coset_pipeline(dom, d.as<Fr>(), batch, 0);
    float ms = t.stop();
    if (kernel_ms) *kernel_ms = ms;
    NZCP_CUDA(cudaMemcpy(data, d.p, n * 32 * batch, cudaMemcpyDeviceToHost));
  });
}

int nzcp_msm(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int device,
             uint8_t* out, float* kernel_ms) {
  return api_guard([&] {
    if (!out || (n_points && (!bases || !scalars))) throw ApiError(NZCP_E_ARG, "null argument");
    use_device(device);
    size_t bsz = g2 ? 128 : 64;
    int c = window_bits > 0 ? window_bits : msm_pick_window(n_points ? n_points : 1);
    DevBuf db(n_points * bsz), ds(n_points * 32);
    if (n_points) {
      NZCP_CUDA(cudaMemcpy(db.p, bases, n_points * bsz, cudaMemcpyHostToDevice));
      NZCP_CUDA(cudaMemcpy(ds.p, scalars, n_points * 32, cudaMemcpyHostToDevice));
    }
    MsmTable tab;
    MsmSort sort;
    MsmRun run;
    struct Guard {
      MsmTable* t; MsmSort* s; MsmRun* r;
      ~Guard() { msm_run_destroy(r); msm_sort_destroy(s); msm_table_destroy(t); }
    } gd{&tab, &sort, &run};
    // one-time per base set (the prover does this at zkey load); not part of kernel_ms
    msm_table_create(&tab, db.p, n_points, 0, g2 != 0, c, 0);
    msm_sort_create(&sort, n_points, c);
    msm_run_create(&run, &sort, g2 != 0);
    NZCP_CUDA(cudaDeviceSynchronize());
    Timer t(0);
    msm_sort_launch(&sort, ds.as<Fr>(), n_points, 0);
    msm_run_launch(&run, &sort, &tab, 0);
    float ms = t.stop();
    NZCP_CUDA(cudaDeviceSynchronize());
    if (kernel_ms) *kernel_ms = ms;
    try {
      msm_sort_check(&sort);
    } catch (const std::runtime_error& e) {
      throw ApiError(NZCP_E_RANGE, e.what());
    }
    if (g2) g2_to_plain_bytes(msm_run_finish_g2(&run), out); else g1_to_plain_bytes(msm_run_finish_g1(&run), out);
  });
}

int nzcp_selftest(int device, uint64_t seed, uint32_t n_cases, uint32_t* n_bad) {
  return api_guard([&] {
    if (!n_bad || n_cases == 0) throw ApiError(NZCP_E_ARG, "bad argument");
    use_device(device);
    uint32_t bad = 0;
    bad += selftest_field<FrParams>(seed, n_cases);
    bad += selftest_field<FqParams>(seed + 1, n_cases);
    uint32_t nc = n_cases > 64 ? 64 : n_cases;
    bad += selftest_curve<Fq>(g1_generator(), seed, nc);
    bad += selftest_curve<Fq2>(g2_generator(), seed, nc);
    *n_bad = bad;
  });
}

int nzcp_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int device) {
  return api_guard([&] {
    if (!a || !b || !out) throw ApiError(NZCP_E_ARG, "null argument");
    if (op < 0 || op > 7 || field < 0 || field > 1) throw ApiError(NZCP_E_ARG, "bad op/field");
    use_device(device);
    DevBuf da(n * 32), db(n * 32), dout(n * 32);
    NZCP_CUDA(cudaMemcpy(da.p, a, n * 32, cudaMemcpyHostToDevice));
    NZCP_CUDA(cudaMemcpy(db.p, b, n * 32, cudaMemcpyHostToDevice));
    if (field == 0)
      field_op_kernel<FrParams><<<div_up(n, 128), 128>>>(op, da.as<Fr>(), db.as<Fr>(), dout.as<Fr>(), n);
    else
      field_op_kernel<FqParams><<<div_up(n, 128), 128>>>(op, da.as<Fq>(), db.as<Fq>(), dout.as<Fq>(), n);
    NZCP_LAUNCH_CHECK();
    NZCP_CUDA(cudaMemcpy(out, dout.p, n * 32, cudaMemcpyDeviceToHost));
  });
}

int nzcp_arith_op(int op, const uint8_t* in, uint8_t* out, size_t n, int device) {
  return api_guard([&] {
    if (!in || !out) throw ApiError(NZCP_E_ARG, "null argument");
    if (op < 0 || op > 9) throw ApiError(NZCP_E_ARG, "bad op");
    // ops 0 and 1 take raw integers: keep them inside the bounds their carry chains assume
    for (size_t i = 0; i < n && op <= 1; i++) {
      const uint32_t* w = reinterpret_cast<const uint32_t*>(in + 64 * i);
      if (op == 0 && ((w[7] | w[15]) >> 31)) throw ApiError(NZCP_E_ARG, "fp_mul_wide operand >= 2^255");
      if (op == 1 && fp_geq_mod<FqParams>(w + 8)) throw ApiError(NZCP_E_ARG, "fp_redc_wide input >= q * 2^256");
    }
    use_device(device);
    if (!n) return;
    const int iw = kArithIn[op], ow = kArithOut[op];
    DevBuf din(n * iw), dout(n * ow);
    NZCP_CUDA(cudaMemcpy(din.p, in, n * iw, cudaMemcpyHostToDevice));
    arith_op_kernel<<<div_up(n, 128), 128>>>(op, din.as<uint32_t>(), dout.as<uint32_t>(), n, iw / 4, ow / 4);
    NZCP_LAUNCH_CHECK();
    NZCP_CUDA(cudaMemcpy(out, dout.p, n * ow, cudaMemcpyDeviceToHost));
  });
}

int nzcp_curve_op(int g2, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int device) {
  return api_guard([&] {
    if (!a || !out || (op <= 2 && !b)) throw ApiError(NZCP_E_ARG, "null argument");
    if (op < 0 || op > 4 || g2 < 0 || g2 > 1) throw ApiError(NZCP_E_ARG, "bad op/group");
    // xyzz_madd's contract: the affine operand is never the point at infinity (0, 0)
    const size_t as = g2 ? sizeof(G2Affine) : sizeof(G1Affine);
    for (size_t i = 0; i < n && (op == 1 || op == 2); i++) {
      const uint8_t* p = b + as * i;
      bool zero = true;
      for (size_t k = 0; k < as && zero; k++) zero = p[k] == 0;
      if (zero) throw ApiError(NZCP_E_ARG, "madd operand is the point at infinity");
    }
    use_device(device);
    if (!n) return;
    if (g2) run_xyzz_op<Fq2>(op, a, b, out, n); else run_xyzz_op<Fq>(op, a, b, out, n);
  });
}

// ---- host-side hooks: the same __host__ __device__ arithmetic compiled for the CPU.  Used by the no-GPU tests to pin
// the code the O(1) host glue (finalisation, twiddle tables, synthetic setup) runs, against the Python oracle.
int nzcp_host_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
  return api_guard([&] {
    if (!a || !b || !out) throw ApiError(NZCP_E_ARG, "null argument");
    if (op < 0 || op > 4 || field < 0 || field > 1) throw ApiError(NZCP_E_ARG, "bad op/field");
    for (size_t i = 0; i < n; i++) {
      if (field == 0) {
        Fr x = fp_from_bytes_plain<FrParams>(a + 32 * i), y = fp_from_bytes_plain<FrParams>(b + 32 * i);
        Fr r = op == 0 ? fp_mul(x, y) : op == 1 ? fp_add(x, y) : op == 2 ? fp_sub(x, y) : op == 3 ? fp_inv_fast(x)
               : (x.is_zero() ? x : fp_inv(x));
        fp_to_bytes(r, out + 32 * i);
      } else {
        Fq x = fp_from_bytes_plain<FqParams>(a + 32 * i), y = fp_from_bytes_plain<FqParams>(b + 32 * i);
        Fq r = op == 0 ? fp_mul(x, y) : op == 1 ? fp_add(x, y) : op == 2 ? fp_sub(x, y) : op == 3 ? fp_inv_fast(x)
               : (x.is_zero() ? x : fp_inv(x));
        fp_to_bytes(r, out + 32 * i);
      }
    }
  });
}

int nzcp_host_scalar_mul(int g2, const uint8_t* base_mont, const uint8_t* scalar, uint8_t* out_plain) {
  return api_guard([&] {
    if (!scalar || !out_plain) throw ApiError(NZCP_E_ARG, "null argument");
    Fr k = fp_from_bytes_plain<FrParams>(scalar);
    if (g2) {
      G2Affine b = g2_generator();
      if (base_mont) memcpy(&b, base_mont, 128);
      g2_to_plain_bytes(xyzz_mul(G2XYZZ::from_affine(b), k.v), out_plain);
    } else {
      G1Affine b = g1_generator();
      if (base_mont) memcpy(&b, base_mont, 64);
      g1_to_plain_bytes(xyzz_mul(G1XYZZ::from_affine(b), k.v), out_plain);
    }
  });
}

int nzcp_host_msm_sim(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int rounds,
                      int adds_per_thread, uint8_t* out) {
  return api_guard([&] {
    if (!out || (n_points && (!bases || !scalars))) throw ApiError(NZCP_E_ARG, "null argument");
    if (window_bits < 2 || window_bits > 16 || rounds < 0 || rounds > kMsmMaxRounds) throw ApiError(NZCP_E_ARG, "bad window / rounds");
    if (g2) g2_to_plain_bytes(host_msm_sim<Fq2>(bases, scalars, n_points, window_bits, rounds, adds_per_thread), out);
    else g1_to_plain_bytes(host_msm_sim<Fq>(bases, scalars, n_points, window_bits, rounds, adds_per_thread), out);
  });
}

int nzcp_host_root_of_unity(int k, uint8_t* out_plain) {
  return api_guard([&] {
    if (!out_plain || k < 0 || k > 28) throw ApiError(NZCP_E_ARG, "bad argument");
    fp_to_bytes(fp_from_mont(host_fr_root(k)), out_plain);
  });
}

}  // extern "C"
