// Synthetic circuits of the NZCP shape + Groth16 setup from explicit toxic waste.
//
// Why this exists: the reference's circuit cannot be compiled here (no circom; sha256-var-circom is fetched at build
// time by /root/reference/Makefile:14-19) and snarkjs cannot run (no node), so BASELINE.json's workloads are defined
// on *synthetic* R1CS instances with the derived shape of nzcp_exampleTest / nzcp_liveTest
// (/root/reference/circuits/nzcp_exampleTest.circom:4, nzcp_liveTest.circom:4; SURVEY.md section 8d).
// The setup below restates snarkjs 0.4.12 src/zkey_new.js with the ptau file replaced by a known tau: every point it
// would read from ptau sections 12-15 is scalar * generator, computed on the GPU by a fixed-base window kernel.
// Output is a byte-exact snarkjs-format .zkey (SURVEY.md 8b), plus .r1cs (iden3 r1csfile) and .wtns images.
#include <memory>

#include "api_util.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ PRNG
struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed * 0x9E3779B97F4A7C15ull + 0x1234567ull) {}
  uint64_t next() {  // splitmix64
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  uint32_t below(uint32_t n) { return (uint32_t)(next() % n); }
  Fr fr_plain() {  // uniform below 2^253 (< r)
    Fr x;
    for (int i = 0; i < 4; i++) {
      uint64_t v = next();
      x.v[2 * i] = (uint32_t)v;
      x.v[2 * i + 1] = (uint32_t)(v >> 32);
    }
    x.v[7] &= 0x1fffffffu;
    return x;
  }
};

static Fr fr_small(uint64_t v) {
  Fr t = Fr::zero();
  t.v[0] = (uint32_t)v;
  t.v[1] = (uint32_t)(v >> 32);
  return fp_to_mont(t);
}

struct Term {
  uint32_t wire;
  Fr coef;  // Montgomery form
};

struct LC {
  std::vector<Term> t;
  void add(uint32_t wire, const Fr& c) {
    for (auto& x : t)
      if (x.wire == wire) {
        x.coef = fp_add(x.coef, c);
        return;
      }
    t.push_back(Term{wire, c});
  }
};

enum WireClass : uint8_t { kBit = 0, kByte = 1, kFull = 2 };

}  // namespace nzcp

using namespace nzcp;

struct nzcp_synth {
  uint64_t seed = 0;
  uint32_t n_constraints = 0, n_public = 0, n_free = 0, n_vars = 0, domain_size = 0, power = 0;
  // CSR over constraints, three matrices
  std::vector<uint32_t> ptr[3];
  std::vector<Term> terms[3];
  std::vector<uint32_t> defines;   // wire fixed by constraint j
  std::vector<Fr> c_out_inv;       // inverse of the coefficient of `defines[j]` in C_j (Montgomery)
  std::vector<uint8_t> wire_class;
  uint64_t n_coefs = 0;            // section-4 records: A + B terms + nPublic + 1
};

namespace nzcp {

static WireClass draw_class(Rng& g) {
  uint32_t x = g.below(100);
  return x < 55 ? kBit : x < 80 ? kByte : kFull;
}

static nzcp_synth* synth_create_impl(uint64_t seed, uint32_t nc, uint32_t npub, uint32_t nfree) {
  if (nc < npub || nfree < 16 || nc == 0) throw ApiError(NZCP_E_ARG, "synth: need n_constraints >= n_public and n_free >= 16");
  std::unique_ptr<nzcp_synth> c(new nzcp_synth());
  c->seed = seed;
  c->n_constraints = nc;
  c->n_public = npub;
  c->n_free = nfree;
  c->n_vars = 1 + nfree + nc;
  uint64_t need = (uint64_t)nc + npub + 1;
  c->power = 1;  // snarkjs: cirPower = log2(nConstraints + nPublic + 1 - 1) + 1; domain at least 2
  while (((uint64_t)1 << c->power) < need) c->power++;
  c->domain_size = 1u << c->power;
  c->wire_class.assign(c->n_vars, kFull);
  Rng g(seed);
  const uint32_t first_free = 1 + npub, first_int = 1 + npub + nfree;
  std::vector<uint32_t> known, known_bits;
  known.reserve(c->n_vars);
  known_bits.reserve(c->n_vars);
  c->wire_class[0] = kBit;  // the constant 1
  for (uint32_t i = 0; i < nfree; i++) {
    uint32_t w = first_free + i;
    WireClass k = i < 8 ? kBit : draw_class(g);
    c->wire_class[w] = k;
    known.push_back(w);
    if (k == kBit) known_bits.push_back(w);
  }
  const Fr one = Fr::one(), two = fr_small(2), minus1 = fp_neg(one);
  for (int k = 0; k < 3; k++) c->ptr[k].push_back(0);
  const uint32_t n_int = nc - npub;
  for (uint32_t j = 0; j < nc; j++) {
    uint32_t out = j < n_int ? first_int + j : 1 + (j - n_int);
    WireClass cls = j < n_int ? draw_class(g) : ((j - n_int) + 1 == npub ? kFull : kBit);  // NZCP: 512 hash bits + exp
    LC A, B, C;
    Fr out_coef = one;
    auto pick_bit = [&]() { return known_bits[g.below((uint32_t)known_bits.size())]; };
    auto pick_any = [&]() { return known[g.below((uint32_t)known.size())]; };
    if (cls == kBit) {
      uint32_t x = pick_bit(), y = pick_bit(), sel = pick_bit();
      switch (g.below(3)) {
        case 0:  // AND: x*y = out
          A.add(x, one); B.add(y, one); C.add(out, one);
          break;
        case 1:  // XOR: 2x*y = x + y - out
          A.add(x, two); B.add(y, one); C.add(x, one); C.add(y, one); C.add(out, minus1);
          out_coef = minus1;
          break;
        default:  // MUX: sel*(x - y) = out - y
          A.add(sel, one); B.add(x, one); B.add(y, minus1); C.add(out, one); C.add(y, minus1);
          break;
      }
      // C may have merged `out`-free duplicates (x == y); the coefficient of `out` is still out_coef
    } else if (cls == kByte) {  // out = sum 2^k b_k  (times the constant 1)
      for (int k = 0; k < 8; k++) A.add(pick_bit(), fr_small(1u << k));
      B.add(0, one);
      C.add(out, one);
    } else {
      auto rand_lc = [&](LC& lc) {
        int k = 2 + (int)g.below(7);
        for (int i = 0; i < k; i++) {
          uint32_t kind = g.below(4);
          Fr coef = kind < 2 ? one : kind == 2 ? fr_small(1 + g.below(65535)) : fp_to_mont(g.fr_plain());
          lc.add(pick_any(), coef);
        }
      };
      rand_lc(A);
      rand_lc(B);
      C.add(out, one);
    }
    LC* lcs[3] = {&A, &B, &C};
    for (int k = 0; k < 3; k++) {
      for (auto& t : lcs[k]->t)
        if (!t.coef.is_zero()) c->terms[k].push_back(t);
      c->ptr[k].push_back((uint32_t)c->terms[k].size());
    }
    c->defines.push_back(out);
    c->c_out_inv.push_back(out_coef);  // +-1 is its own inverse
    c->wire_class[out] = cls;
    known.push_back(out);
    if (cls == kBit) known_bits.push_back(out);
  }
  c->n_coefs = c->terms[0].size() + c->terms[1].size() + npub + 1;
  return c.release();
}

// Satisfying witness in Montgomery form.
static std::vector<Fr> synth_witness(const nzcp_synth* c, uint64_t wseed) {
  std::vector<Fr> w(c->n_vars, Fr::zero());
  w[0] = Fr::one();
  Rng g(wseed ^ 0xA5A5A5A55A5A5A5Aull);
  const uint32_t first_free = 1 + c->n_public;
  for (uint32_t i = 0; i < c->n_free; i++) {
    uint32_t wi = first_free + i;
    switch (c->wire_class[wi]) {
      case kBit: w[wi] = fr_small(g.next() & 1); break;
      case kByte: w[wi] = fr_small(g.next() & 0xff); break;
      default: w[wi] = fp_to_mont(g.fr_plain()); break;
    }
  }
  auto dot = [&](int k, uint32_t j, uint32_t skip, bool use_skip) {
    Fr acc = Fr::zero();
    for (uint32_t t = c->ptr[k][j]; t < c->ptr[k][j + 1]; t++) {
      const Term& tm = c->terms[k][t];
      if (use_skip && tm.wire == skip) continue;
      acc = fp_add(acc, fp_mul(tm.coef, w[tm.wire]));
    }
    return acc;
  };
  for (uint32_t j = 0; j < c->n_constraints; j++) {
    Fr a = dot(0, j, 0, false), b = dot(1, j, 0, false);
    Fr rest = dot(2, j, c->defines[j], true);
    w[c->defines[j]] = fp_mul(fp_sub(fp_mul(a, b), rest), c->c_out_inv[j]);
  }
  return w;
}

// ------------------------------------------------------------------------------------------------ container writer
struct Writer {
  uint8_t* p;
  size_t cap, pos = 0;
  Writer(uint8_t* b, size_t c) : p(b), cap(c) {}
  void need(size_t n) {
    if (pos + n > cap) throw ApiError(NZCP_E_ARG, "output buffer too small");
  }
  void u32(uint32_t v) { need(4); memcpy(p + pos, &v, 4); pos += 4; }
  void u64(uint64_t v) { need(8); memcpy(p + pos, &v, 8); pos += 8; }
  void raw(const void* s, size_t n) { need(n); memcpy(p + pos, s, n); pos += n; }
  void zeros(size_t n) { need(n); memset(p + pos, 0, n); pos += n; }
  void section(uint32_t id, uint64_t len) { u32(id); u64(len); }
};

static const uint32_t kG1GenX[8] = {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
static const uint32_t kG1GenY[8] = {0x8b1e1b3au, 0xa6ba871bu, 0xeb8e167bu, 0x14f1d651u, 0xf0f28c58u, 0xccdd46deu, 0x340fbe5eu, 0x1c14ef83u};
static const uint32_t kG2GenX0[8] = {0x02bc2026u, 0x8e83b5d1u, 0x497b0172u, 0xdceb1935u, 0x97811adfu, 0xfbb82647u, 0xaf96503bu, 0x19573841u};
static const uint32_t kG2GenX1[8] = {0xa84c6140u, 0xafb4737du, 0x5802d8c4u, 0x6043dd5au, 0x52a02f86u, 0x09e950fcu, 0x3aea7b6bu, 0x14fef083u};
static const uint32_t kG2GenY0[8] = {0x886be9f6u, 0x619dfa9du, 0xf59e9b78u, 0xfe7fd297u, 0x231b7dfeu, 0xff9e1a62u, 0xae9e4206u, 0x28fd7eebu};
static const uint32_t kG2GenY1[8] = {0xc71856eeu, 0x64095b56u, 0x327d3cbbu, 0xdc57f922u, 0x33351076u, 0x55f935beu, 0x93fd6482u, 0x0da4a0e6u};

static Fq fq_limbs(const uint32_t* l) {
  Fq x;
  memcpy(x.v, l, 32);
  return x;
}
G1Affine g1_generator() { return G1Affine{fq_limbs(kG1GenX), fq_limbs(kG1GenY)}; }
G2Affine g2_generator() {
  return G2Affine{Fq2{fq_limbs(kG2GenX0), fq_limbs(kG2GenX1)}, Fq2{fq_limbs(kG2GenY0), fq_limbs(kG2GenY1)}};
}

// ------------------------------------------------------------------------------------------------ fixed-base kernel
static constexpr int kFbWindow = 8;
static constexpr int kFbWindows = 32;
static constexpr int kFbRow = 255;

// table[w][d-1] = d * 2^(8w) * G  (affine, Montgomery)
template <class F>
static std::vector<Affine<F>> fixed_base_table(const Affine<F>& gen) {
  std::vector<XYZZ<F>> pts((size_t)kFbWindows * kFbRow);
  XYZZ<F> base = XYZZ<F>::from_affine(gen);
  for (int w = 0; w < kFbWindows; w++) {
    XYZZ<F> acc = XYZZ<F>::inf();
    for (int d = 0; d < kFbRow; d++) {
      xyzz_add(acc, base);
      pts[(size_t)w * kFbRow + d] = acc;
    }
    for (int k = 0; k < kFbWindow; k++) base = xyzz_dbl(base);
  }
  std::vector<Affine<F>> out(pts.size());
  for (size_t i = 0; i < pts.size(); i++) out[i] = xyzz_to_affine(pts[i]);
  return out;
}

template <class F>
__global__ void __launch_bounds__(128)
fixed_base_mul_kernel(const Affine<F>* __restrict__ table, const Fr* __restrict__ scalars, Affine<F>* __restrict__ out,
                      size_t count) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  Fr s = scalars[i];
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int w = 0; w < kFbWindows; w++) {
    uint32_t d = (s.v[w >> 2] >> ((w & 3) * 8)) & 0xff;
    if (d) xyzz_madd(acc, table[w * kFbRow + (d - 1)], false);
  }
  out[i] = xyzz_to_affine(acc);
}

// scalars: plain Fr (host).  dst: host buffer receiving count affine Montgomery points in zkey byte order.
template <class F>
static void fixed_base_batch(const Affine<F>* d_table, const std::vector<Fr>& scalars, uint8_t* dst) {
  size_t count = scalars.size();
  if (!count) return;
  CudaResources res;
  Fr* d_s = res.device<Fr>(count);
  Affine<F>* d_o = res.device<Affine<F>>(count);
  NZCP_CUDA(cudaMemcpy(d_s, scalars.data(), count * sizeof(Fr), cudaMemcpyHostToDevice));
  fixed_base_mul_kernel<F><<<div_up(count, 128), 128>>>(d_table, d_s, d_o, count);
  NZCP_LAUNCH_CHECK();
  NZCP_CUDA(cudaMemcpy(dst, d_o, count * sizeof(Affine<F>), cudaMemcpyDeviceToHost));
}

// In-place batch inversion (Montgomery trick); zero entries are left untouched.
static void batch_inverse(std::vector<Fr>& v) {
  std::vector<Fr> pre(v.size());
  Fr acc = Fr::one();
  for (size_t i = 0; i < v.size(); i++) {
    pre[i] = acc;
    if (!v[i].is_zero()) acc = fp_mul(acc, v[i]);
  }
  Fr inv = fp_inv(acc);
  for (size_t i = v.size(); i-- > 0;) {
    if (v[i].is_zero()) continue;
    Fr t = fp_mul(inv, pre[i]);
    inv = fp_mul(inv, v[i]);
    v[i] = t;
  }
}

// L_j(tau) for the size-2^log_n domain, j = first, first+step, ... (count values).  Montgomery form.
static std::vector<Fr> lagrange_at(const Fr& tau, int log_n, size_t first, size_t step, size_t count) {
  size_t n = (size_t)1 << log_n;
  Fr w = host_fr_root(log_n);
  Fr tn = tau;
  for (int i = 0; i < log_n; i++) tn = fp_sqr(tn);
  Fr zt = fp_sub(tn, Fr::one());
  Fr k = fp_mul(zt, fp_inv(fr_small(n)));
  Fr wstep = Fr::one(), wfirst = Fr::one();
  {  // w^step, w^first by square-and-multiply on small exponents
    auto pw = [&](size_t e) {
      Fr r = Fr::one(), b = w;
      while (e) {
        if (e & 1) r = fp_mul(r, b);
        b = fp_sqr(b);
        e >>= 1;
      }
      return r;
    };
    wstep = pw(step);
    wfirst = pw(first);
  }
  std::vector<Fr> wj(count), den(count);
  Fr cur = wfirst;
  for (size_t i = 0; i < count; i++) {
    wj[i] = cur;
    den[i] = fp_sub(tau, cur);
    cur = fp_mul(cur, wstep);
  }
  batch_inverse(den);
  std::vector<Fr> out(count);
  for (size_t i = 0; i < count; i++) out[i] = fp_mul(fp_mul(k, wj[i]), den[i]);
  return out;
}

static size_t zkey_size(const nzcp_synth* c) {
  size_t m = c->n_vars, n = c->domain_size, np = c->n_public;
  size_t hdr = 4 + 32 + 4 + 32 + 12 + 64 + 64 + 128 + 128 + 64 + 128;
  size_t body = 4 + hdr + (np + 1) * 64 + (4 + c->n_coefs * 44) + m * 64 + m * 64 + m * 128 + (m - np - 1) * 64 + n * 64 + (64 + 4);
  return 12 + 10 * 12 + body;
}

static void synth_write_zkey_impl(const nzcp_synth* c, const uint8_t toxic[160], int device, uint8_t* out, size_t cap) {
  use_device(device);
  const size_t m = c->n_vars, n = c->domain_size, np = c->n_public, nc = c->n_constraints;
  Fr tx[5];
  for (int i = 0; i < 5; i++) {
    if (!fr_bytes_canonical(toxic + 32 * i)) throw ApiError(NZCP_E_ARG, "toxic value not < r");
    tx[i] = fp_to_mont(fp_from_bytes_plain<FrParams>(toxic + 32 * i));
    if (tx[i].is_zero()) throw ApiError(NZCP_E_ARG, "toxic value is zero");
  }
  const Fr tau = tx[0], alpha = tx[1], beta = tx[2], gamma = tx[3], delta = tx[4];
  const Fr ginv = fp_inv(gamma), dinv = fp_inv(delta);
  // polynomial evaluations at tau
  std::vector<Fr> L = lagrange_at(tau, (int)c->power, 0, 1, n);
  std::vector<Fr> ev[3];
  for (int k = 0; k < 3; k++) {
    ev[k].assign(m, Fr::zero());
    for (size_t j = 0; j < nc; j++)
      for (uint32_t t = c->ptr[k][j]; t < c->ptr[k][j + 1]; t++) {
        const Term& tm = c->terms[k][t];
        ev[k][tm.wire] = fp_add(ev[k][tm.wire], fp_mul(tm.coef, L[j]));
      }
  }
  for (size_t i = 0; i <= np; i++) ev[0][i] = fp_add(ev[0][i], L[nc + i]);  // appended rows A[nc+i][i] = 1
  std::vector<Fr> L2odd = lagrange_at(tau, (int)c->power + 1, 1, 2, n);
  L.clear();
  L.shrink_to_fit();
  // scalar vectors (plain) for the fixed-base kernel
  auto plain = [](const Fr& x) { return fp_from_mont(x); };
  std::vector<Fr> sA(m), sB(m), sIC(np + 1), sC(m - np - 1), sH(n);
  for (size_t i = 0; i < m; i++) {
    sA[i] = plain(ev[0][i]);
    sB[i] = plain(ev[1][i]);
    Fr comb = fp_add(fp_add(fp_mul(beta, ev[0][i]), fp_mul(alpha, ev[1][i])), ev[2][i]);
    if (i <= np)
      sIC[i] = plain(fp_mul(comb, ginv));
    else
      sC[i - np - 1] = plain(fp_mul(comb, dinv));
  }
  for (size_t i = 0; i < n; i++) sH[i] = plain(fp_mul(L2odd[i], dinv));
  // device tables
  std::vector<G1Affine> t1 = fixed_base_table<Fq>(g1_generator());
  std::vector<G2Affine> t2 = fixed_base_table<Fq2>(g2_generator());
  CudaResources res;
  G1Affine* d_t1 = res.device<G1Affine>(t1.size());
  G2Affine* d_t2 = res.device<G2Affine>(t2.size());
  NZCP_CUDA(cudaMemcpy(d_t1, t1.data(), t1.size() * sizeof(G1Affine), cudaMemcpyHostToDevice));
  NZCP_CUDA(cudaMemcpy(d_t2, t2.data(), t2.size() * sizeof(G2Affine), cudaMemcpyHostToDevice));

  Writer w(out, cap);
  w.raw("zkey", 4);
  w.u32(1);
  w.u32(10);
  w.section(1, 4);
  w.u32(1);
  const size_t hdr = 4 + 32 + 4 + 32 + 12 + 64 + 64 + 128 + 128 + 64 + 128;
  w.section(2, hdr);
  w.u32(32);
  w.raw(kQBytes, 32);
  w.u32(32);
  w.raw(kRBytes, 32);
  w.u32((uint32_t)m);
  w.u32((uint32_t)np);
  w.u32((uint32_t)n);
  {
    std::vector<Fr> s1 = {plain(alpha), plain(beta), plain(delta)};
    std::vector<Fr> s2 = {plain(beta), plain(gamma), plain(delta)};
    uint8_t p1[3 * 64], p2[3 * 128];
    fixed_base_batch<Fq>(d_t1, s1, p1);
    fixed_base_batch<Fq2>(d_t2, s2, p2);
    w.raw(p1, 64);          // alpha1
    w.raw(p1 + 64, 64);     // beta1
    w.raw(p2, 128);         // beta2
    w.raw(p2 + 128, 128);   // gamma2
    w.raw(p1 + 128, 64);    // delta1
    w.raw(p2 + 256, 128);   // delta2
  }
  w.section(3, (np + 1) * 64);
  w.need((np + 1) * 64);
  fixed_base_batch<Fq>(d_t1, sIC, w.p + w.pos);
  w.pos += (np + 1) * 64;
  w.section(4, 4 + c->n_coefs * 44);
  w.u32((uint32_t)c->n_coefs);
  for (size_t j = 0; j < nc; j++)
    for (int k = 0; k < 2; k++)
      for (uint32_t t = c->ptr[k][j]; t < c->ptr[k][j + 1]; t++) {
        const Term& tm = c->terms[k][t];
        w.u32((uint32_t)k);
        w.u32((uint32_t)j);
        w.u32(tm.wire);
        Fr stored = fp_to_mont(tm.coef);  // coef * R^2 mod r (zkey_new.js), SURVEY F7
        w.raw(stored.v, 32);
      }
  {
    Fr stored = Fr::r2();  // 1 * R^2
    for (size_t i = 0; i <= np; i++) {
      w.u32(0);
      w.u32((uint32_t)(nc + i));
      w.u32((uint32_t)i);
      w.raw(stored.v, 32);
    }
  }
  w.section(5, m * 64);
  w.need(m * 64);
  fixed_base_batch<Fq>(d_t1, sA, w.p + w.pos);
  w.pos += m * 64;
  w.section(6, m * 64);
  w.need(m * 64);
  fixed_base_batch<Fq>(d_t1, sB, w.p + w.pos);
  w.pos += m * 64;
  w.section(7, m * 128);
  w.need(m * 128);
  fixed_base_batch<Fq2>(d_t2, sB, w.p + w.pos);
  w.pos += m * 128;
  w.section(8, (m - np - 1) * 64);
  w.need((m - np - 1) * 64);
  fixed_base_batch<Fq>(d_t1, sC, w.p + w.pos);
  w.pos += (m - np - 1) * 64;
  w.section(9, n * 64);
  w.need(n * 64);
  fixed_base_batch<Fq>(d_t1, sH, w.p + w.pos);
  w.pos += n * 64;
  w.section(10, 64 + 4);
  w.zeros(64);
  w.u32(0);
  if (w.pos != zkey_size(c)) throw ApiError(NZCP_E_INTERNAL, "synth: zkey size accounting is off");
}

static size_t r1cs_size(const nzcp_synth* c) {
  size_t hdr = 4 + 32 + 4 * 4 + 8 + 4;
  size_t nterms = c->terms[0].size() + c->terms[1].size() + c->terms[2].size();
  size_t body = (size_t)c->n_constraints * 12 + nterms * 36;
  return 12 + 3 * 12 + hdr + body + (size_t)c->n_vars * 8;
}

static void synth_write_r1cs_impl(const nzcp_synth* c, uint8_t* out, size_t cap) {
  Writer w(out, cap);
  w.raw("r1cs", 4);
  w.u32(1);
  w.u32(3);
  w.section(1, 4 + 32 + 16 + 8 + 4);
  w.u32(32);
  w.raw(kRBytes, 32);
  w.u32(c->n_vars);
  w.u32(c->n_public);  // nPubOut
  w.u32(0);            // nPubIn
  w.u32(c->n_free);    // nPrvIn
  w.u64(c->n_vars);    // nLabels
  w.u32(c->n_constraints);
  size_t nterms = c->terms[0].size() + c->terms[1].size() + c->terms[2].size();
  w.section(2, (size_t)c->n_constraints * 12 + nterms * 36);
  for (uint32_t j = 0; j < c->n_constraints; j++)
    for (int k = 0; k < 3; k++) {
      w.u32(c->ptr[k][j + 1] - c->ptr[k][j]);
      for (uint32_t t = c->ptr[k][j]; t < c->ptr[k][j + 1]; t++) {
        w.u32(c->terms[k][t].wire);
        Fr pl = fp_from_mont(c->terms[k][t].coef);
        w.raw(pl.v, 32);
      }
    }
  w.section(3, (size_t)c->n_vars * 8);
  for (uint32_t i = 0; i < c->n_vars; i++) w.u64(i);
  if (w.pos != r1cs_size(c)) throw ApiError(NZCP_E_INTERNAL, "synth: r1cs size accounting is off");
}

static size_t wtns_size(const nzcp_synth* c) { return 12 + 2 * 12 + 40 + (size_t)c->n_vars * 32; }

static void synth_write_wtns_impl(const nzcp_synth* c, uint64_t wseed, uint8_t* out, size_t cap) {
  std::vector<Fr> wm = synth_witness(c, wseed);
  Writer w(out, cap);
  w.raw("wtns", 4);
  w.u32(2);
  w.u32(2);
  w.section(1, 40);
  w.u32(32);
  w.raw(kRBytes, 32);
  w.u32(c->n_vars);
  w.section(2, (size_t)c->n_vars * 32);
  w.need((size_t)c->n_vars * 32);
  for (uint32_t i = 0; i < c->n_vars; i++) {
    Fr pl = fp_from_mont(wm[i]);
    memcpy(w.p + w.pos, pl.v, 32);
    w.pos += 32;
  }
}

}  // namespace nzcp

namespace nzcp {
// n pseudo-random points k_i * G (k_i from splitmix64(seed)), Montgomery affine, written to a HOST buffer.
template <class F>
static void synth_points_impl(const Affine<F>& gen, uint64_t seed, size_t n, uint8_t* out) {
  std::vector<Affine<F>> tab = fixed_base_table<F>(gen);
  CudaResources res;
  Affine<F>* d_tab = res.device<Affine<F>>(tab.size());
  NZCP_CUDA(cudaMemcpy(d_tab, tab.data(), tab.size() * sizeof(Affine<F>), cudaMemcpyHostToDevice));
  Rng g(seed);
  const size_t chunk = (size_t)1 << 20;
  std::vector<Fr> sc;
  for (size_t done = 0; done < n; done += chunk) {
    size_t cnt = n - done < chunk ? n - done : chunk;
    sc.resize(cnt);
    for (size_t i = 0; i < cnt; i++) {
      sc[i] = g.fr_plain();
      if (sc[i].is_zero()) sc[i].v[0] = 1;
    }
    fixed_base_batch<F>(d_tab, sc, out + done * sizeof(Affine<F>));
  }
}
}  // namespace nzcp

extern "C" {

int nzcp_synth_points(uint64_t seed, size_t n_points, int g2, int device, uint8_t* out) {
  return api_guard([&] {
    if (!out && n_points) throw ApiError(NZCP_E_ARG, "null argument");
    use_device(device);
    if (g2) synth_points_impl<Fq2>(g2_generator(), seed, n_points, out);
    else synth_points_impl<Fq>(g1_generator(), seed, n_points, out);
  });
}

int nzcp_synth_create(uint64_t seed, uint32_t n_constraints, uint32_t n_public, uint32_t n_free, nzcp_synth** out) {
  return api_guard([&] {
    if (!out) throw ApiError(NZCP_E_ARG, "null argument");
    *out = nullptr;
    *out = synth_create_impl(seed, n_constraints, n_public, n_free);
  });
}

void nzcp_synth_free(nzcp_synth* c) { delete c; }

int nzcp_synth_dims(const nzcp_synth* c, uint32_t* n_vars, uint32_t* n_constraints, uint32_t* n_public,
                    uint32_t* domain_size, uint64_t* n_coefs) {
  return api_guard([&] {
    if (!c) throw ApiError(NZCP_E_ARG, "null argument");
    if (n_vars) *n_vars = c->n_vars;
    if (n_constraints) *n_constraints = c->n_constraints;
    if (n_public) *n_public = c->n_public;
    if (domain_size) *domain_size = c->domain_size;
    if (n_coefs) *n_coefs = c->n_coefs;
  });
}

size_t nzcp_synth_zkey_size(const nzcp_synth* c) { return c ? zkey_size(c) : 0; }
size_t nzcp_synth_r1cs_size(const nzcp_synth* c) { return c ? r1cs_size(c) : 0; }
size_t nzcp_synth_wtns_size(const nzcp_synth* c) { return c ? wtns_size(c) : 0; }

int nzcp_synth_write_zkey(const nzcp_synth* c, const uint8_t toxic[160], int device, uint8_t* out, size_t cap) {
  return api_guard([&] {
    if (!c || !toxic || !out) throw ApiError(NZCP_E_ARG, "null argument");
    synth_write_zkey_impl(c, toxic, device, out, cap);
  });
}

int nzcp_synth_write_r1cs(const nzcp_synth* c, uint8_t* out, size_t cap) {
  return api_guard([&] {
    if (!c || !out) throw ApiError(NZCP_E_ARG, "null argument");
    synth_write_r1cs_impl(c, out, cap);
  });
}

int nzcp_synth_write_wtns(const nzcp_synth* c, uint64_t witness_seed, uint8_t* out, size_t cap) {
  return api_guard([&] {
    if (!c || !out) throw ApiError(NZCP_E_ARG, "null argument");
    synth_write_wtns_impl(c, witness_seed, out, cap);
  });
}

}  // extern "C"
