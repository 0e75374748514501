// `zkey new` on the GPU: the circuit-specific Groth16 proving key from an .r1cs and a PREPARED powers-of-tau file.
//
// Replaces snarkjs 0.4.12 src/zkey_new.js newZKey(r1csName, ptauName, zkeyName) (upstream, not vendored: package.json:12,
// yarn.lock:987-999) -- the step that makes the `nzcp_exampleTest_final.zkey` the proving path loads; the reference names
// its inputs at /root/reference/Makefile:5-9 (`circom ... --r1cs`) and Makefile:31 (`powersOfTau28_hez_final_22.ptau`).
// SURVEY.md 8f row 4.  "Parity unpinned": neither snarkjs nor a real .ptau is available here; the layout below is the
// published one (binfileutils containers; ptau sections 1-7 and the Lagrange-basis sections 12-15 that `powersoftau
// prepare phase2` adds), pinned in the tests by the toxic-waste identity: with a ptau written from a known tau the output
// must equal the closed-form key (oracle/setup.py make_zkey with gamma = delta = 1) section by section.
//
// What zkey_new computes, restated:
//   cirPower = floor(log2(nConstraints + nPublic)) + 1, domainSize = 2^cirPower, nPublic = nOutputs + nPubInputs
//   section 2   alpha1 = ptau[4][0], beta1 = ptau[5][0], beta2 = ptau[6][0]; gamma2 = delta2 = G2, delta1 = G1
//   section 4   per A / B term of constraint c: (matrix, c, signal, coef * R^2 mod r); then nPublic+1 rows (0, nC+s, s, R^2)
//   with L_c = Lagrange basis point c of the size-domainSize level of ptau section 12 (tauG1), 13 (tauG2), 14 (alphaTauG1),
//   15 (betaTauG1):
//   A[s]  = sum over A terms (c, s, k) of k * tauG1_L[c]            (+ tauG1_L[nC+s] for s <= nPublic)
//   B1[s] / B2[s] = sum over B terms of k * tauG1_L[c] / k * tauG2_L[c]
//   K[s]  = sum_A k * betaTauG1_L[c] + sum_B k * alphaTauG1_L[c] + sum_C k * tauG1_L[c]   (+ betaTauG1_L[nC+s], s <= nPublic)
//   section 3 (IC) = K[0..nPublic], section 8 (C) = K[nPublic+1..]   (gamma = delta = 1 at `zkey new` time)
//   section 9   H[i] = tauG1 Lagrange level cirPower+1, entry 2i+1
//   section 10  csHash + 0 contributions.  The circuit hash (BLAKE2b-512 over an uncompressed-point transcript) is NOT
//               computed here: the section is written zero-filled.  `groth16 prove`, `zkey export verificationkey` and
//               `zkey contribute` do not check it; `zkey verify` refuses such a key.  verify.cu computes it from this
//               output and the ptau (nzcp_zkey_circuit_hash; api.zkey_new(..., circuit_hash=True) stamps it).
// Sections are written in zkey_new.js's own order: 1, 2, 4, 3, 9, 8, 5, 6, 7, 10.
//
// B200 design: the four sparse point combinations are one kernel each, one thread per wire walking its term list
// (CSR by wire built on the host): k * P over signed 4-bit windows of k (ec.cuh scalar_mul_accumulate), with k > r/2
// folded to (r - k) * (-P) so the -1 / small-negative coefficients circom emits cost one addition, not 254 doublings.
// One-time work per circuit.
#include <memory>

#include "binfile.cuh"

namespace nzcp {

R1cs parse_r1cs(const uint8_t* b, size_t len) {
  Sect s[4];
  parse_bin(b, len, "r1cs", s, 3);
  if (!s[1].p || !s[2].p || s[1].len < 4 + 32 + 4 * 4 + 8 + 4) throw ApiError(NZCP_E_FORMAT, "r1cs: missing or short section");
  R1cs r;
  const uint8_t* h = s[1].p;
  if (rd32u(h) != 32 || memcmp(h + 4, kRBytes, 32) != 0)
    throw ApiError(NZCP_E_CURVE, "r1cs curve does not match powers of tau ceremony curve");
  r.n_wires = rd32u(h + 36);
  r.n_pub_out = rd32u(h + 40);
  r.n_pub_in = rd32u(h + 44);
  r.n_prv_in = rd32u(h + 48);
  r.n_constraints = rd32u(h + 60);
  r.n_public = r.n_pub_out + r.n_pub_in;
  if (r.n_public + 1 > r.n_wires) throw ApiError(NZCP_E_FORMAT, "r1cs: more public signals than wires");
  r.cons = s[2].p;
  r.cons_len = s[2].len;
  // one validating pass: term counts, bounds
  uint64_t pos = 0;
  for (uint32_t c = 0; c < r.n_constraints; c++) {
    for (int m = 0; m < 3; m++) {
      if (pos + 4 > r.cons_len) throw ApiError(NZCP_E_FORMAT, "r1cs: truncated constraint section");
      const uint32_t cnt = rd32u(r.cons + pos);
      pos += 4;
      if ((uint64_t)cnt * 36 > r.cons_len - pos) throw ApiError(NZCP_E_FORMAT, "r1cs: truncated constraint section");
      for (uint32_t t = 0; t < cnt; t++, pos += 36) {
        if (rd32u(r.cons + pos) >= r.n_wires) throw ApiError(NZCP_E_FORMAT, "r1cs: wire index out of range");
        if (!fr_bytes_canonical(r.cons + pos + 4)) throw ApiError(NZCP_E_RANGE, "r1cs: coefficient is not a canonical field element");
      }
      r.n_terms[m] += cnt;
    }
  }
  return r;
}

Ptau parse_ptau(const uint8_t* b, size_t len) {
  Ptau p = read_ptau(b, len);
  need_sections(p.s, 2, 6);
  if (!p.s[12].p || !p.s[13].p || !p.s[14].p || !p.s[15].p) throw ApiError(NZCP_E_FORMAT, "Powers of tau is not prepared.");
  const uint64_t n = (uint64_t)1 << p.power;
  // Lagrange sections: levels 0..power back to back (2^(power+1) - 1 points); tauG1 carries one more level (power + 1)
  if (p.s[12].len != (4 * n - 1) * 64 || p.s[13].len != (2 * n - 1) * 128 || p.s[14].len != (2 * n - 1) * 64 ||
      p.s[15].len != (2 * n - 1) * 64 || p.s[4].len < 64 || p.s[5].len < 64 || p.s[6].len < 128)
    throw ApiError(NZCP_E_FORMAT, "ptau: section size does not match the header power");
  return p;
}

uint32_t circuit_power(const R1cs& r) {
  uint64_t v = (uint64_t)r.n_constraints + r.n_public;
  uint32_t lg = 0;
  while (v >> (lg + 1)) lg++;      // floor(log2(v)); snarkjs log2(0) = 0
  return lg + 1;
}

namespace {

struct Term {
  uint32_t point;   // Lagrange point index (constraint number) | source << 30
  uint32_t coef;    // index into the coefficient pool
};

struct Combo {      // one sparse point combination: CSR by wire
  std::vector<uint32_t> row_ptr;
  std::vector<Term> terms;
};

}  // namespace

template <class F>
__global__ void __launch_bounds__(128)
setup_combine_kernel(const uint32_t* __restrict__ row_ptr, const Term* __restrict__ terms, const Fr* __restrict__ coefs,
                     const Affine<F>* __restrict__ src0, const Affine<F>* __restrict__ src1, const Affine<F>* __restrict__ src2,
                     Affine<F>* __restrict__ out, uint32_t n_wires) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_wires) return;
  XYZZ<F> acc = XYZZ<F>::inf();
  for (uint32_t t = row_ptr[s]; t < row_ptr[s + 1]; t++) {
    const Term tm = terms[t];
    const uint32_t which = tm.point >> 30, idx = tm.point & 0x3fffffffu;
    const Affine<F>* src = which == 0 ? src0 : which == 1 ? src1 : src2;
    scalar_mul_accumulate(acc, src[idx], coefs[tm.coef]);
  }
  out[s] = xyzz_to_affine(acc);
}

namespace {

template <class F>
void run_combo(const Combo& cb, const Fr* d_coefs, const void* d_src0, const void* d_src1, const void* d_src2, uint32_t n_wires,
               uint8_t* host_out) {
  CudaResources res;
  uint32_t* d_rp = res.device<uint32_t>(cb.row_ptr.size());
  Term* d_terms = res.device<Term>(cb.terms.size() ? cb.terms.size() : 1);
  Affine<F>* d_out = res.device<Affine<F>>(n_wires ? n_wires : 1);
  NZCP_CUDA(cudaMemcpy(d_rp, cb.row_ptr.data(), cb.row_ptr.size() * 4, cudaMemcpyHostToDevice));
  if (!cb.terms.empty()) NZCP_CUDA(cudaMemcpy(d_terms, cb.terms.data(), cb.terms.size() * sizeof(Term), cudaMemcpyHostToDevice));
  if (n_wires) {
    setup_combine_kernel<F><<<div_up(n_wires, 128), 128>>>(d_rp, d_terms, d_coefs, reinterpret_cast<const Affine<F>*>(d_src0),
                                                          reinterpret_cast<const Affine<F>*>(d_src1),
                                                          reinterpret_cast<const Affine<F>*>(d_src2), d_out, n_wires);
    NZCP_LAUNCH_CHECK();
    NZCP_CUDA(cudaMemcpy(host_out, d_out, (size_t)n_wires * sizeof(Affine<F>), cudaMemcpyDeviceToHost));
  }
}

}  // namespace

size_t zkey_new_size(const R1cs& r, uint32_t cir_power) {
  const uint64_t n = (uint64_t)1 << cir_power, m = r.n_wires, np = r.n_public;
  const uint64_t n_coefs = r.n_terms[0] + r.n_terms[1] + np + 1;
  return 12 + 10 * 12 + 4 + kZkeyHeaderLen + (4 + n_coefs * 44) + (np + 1) * 64 + n * 64 + (m - np - 1) * 64 + m * 64 + m * 64 +
         m * 128 + 68;
}

void zkey_new_impl(const uint8_t* r1cs_b, size_t r1cs_len, const uint8_t* ptau_b, size_t ptau_len, int device, uint8_t* out,
                   size_t cap, size_t* written) {
  const R1cs r = parse_r1cs(r1cs_b, r1cs_len);
  const Ptau pt = parse_ptau(ptau_b, ptau_len);
  const uint32_t cir_power = circuit_power(r);
  if (cir_power > pt.power)
    throw ApiError(NZCP_E_ARG, "circuit too big for this power of tau ceremony. " + std::to_string(r.n_constraints) + "*2 > 2**" +
                                   std::to_string(pt.power));
  const uint64_t n = (uint64_t)1 << cir_power;
  const uint32_t m = r.n_wires, np = r.n_public, nc = r.n_constraints;
  if (n >= ((uint64_t)1 << 30)) throw ApiError(NZCP_E_ARG, "circuit too big");
  const size_t total = zkey_new_size(r, cir_power);
  if (cap < total) throw ApiError(NZCP_E_ARG, "output buffer too small");
  use_device(device);

  // ---- term lists: coefficient pool = the r1cs terms in file order, plus "1" for the appended public rows
  const uint64_t n_pool = r.n_terms[0] + r.n_terms[1] + r.n_terms[2] + 1;
  if (n_pool >= ((uint64_t)1 << 32)) throw ApiError(NZCP_E_ARG, "circuit too big");
  std::vector<Fr> pool(n_pool);
  const uint32_t one_idx = (uint32_t)(n_pool - 1);
  pool[one_idx] = Fr::zero();
  pool[one_idx].v[0] = 1;                                   // plain 1
  // sources: 0 = tauG1_L, 1 = alphaTauG1_L (G2 combo: 0 = tauG2_L), 2 = betaTauG1_L
  Combo A, B, K;                                            // B serves B1 (G1) and B2 (G2): same terms, source 0
  for (Combo* c : {&A, &B, &K}) c->row_ptr.assign((size_t)m + 1, 0);
  auto walk = [&](auto&& on_term) {
    uint64_t pos = 0;
    uint32_t ci = 0;
    for (uint32_t c = 0; c < nc; c++)
      for (int mtx = 0; mtx < 3; mtx++) {
        const uint32_t cnt = rd32u(r.cons + pos);
        pos += 4;
        for (uint32_t t = 0; t < cnt; t++, pos += 36, ci++) on_term(mtx, c, rd32u(r.cons + pos), r.cons + pos + 4, ci);
      }
  };
  walk([&](int mtx, uint32_t, uint32_t s, const uint8_t* coef, uint32_t ci) {
    memcpy(pool[ci].v, coef, 32);
    if (mtx == 0) A.row_ptr[s + 1]++;
    if (mtx == 1) B.row_ptr[s + 1]++;
    K.row_ptr[s + 1]++;
  });
  for (uint32_t s = 0; s <= np; s++) {
    A.row_ptr[s + 1]++;
    K.row_ptr[s + 1]++;
  }
  for (Combo* c : {&A, &B, &K}) {
    for (size_t i = 0; i < m; i++) c->row_ptr[i + 1] += c->row_ptr[i];
    c->terms.resize(c->row_ptr[m]);
  }
  {
    std::vector<uint32_t> fa(A.row_ptr.begin(), A.row_ptr.end() - 1), fb(B.row_ptr.begin(), B.row_ptr.end() - 1),
        fk(K.row_ptr.begin(), K.row_ptr.end() - 1);
    walk([&](int mtx, uint32_t c, uint32_t s, const uint8_t*, uint32_t ci) {
      if (mtx == 0) {
        A.terms[fa[s]++] = Term{c, ci};
        K.terms[fk[s]++] = Term{c | (2u << 30), ci};        // beta * A
      } else if (mtx == 1) {
        B.terms[fb[s]++] = Term{c, ci};
        K.terms[fk[s]++] = Term{c | (1u << 30), ci};        // alpha * B
      } else {
        K.terms[fk[s]++] = Term{c, ci};                     // C
      }
    });
    for (uint32_t s = 0; s <= np; s++) {
      A.terms[fa[s]++] = Term{nc + s, one_idx};
      K.terms[fk[s]++] = Term{(nc + s) | (2u << 30), one_idx};
    }
  }

  // ---- device: the four Lagrange levels of size n, the coefficient pool
  const uint64_t lvl = n - 1;   // points before level cir_power in a Lagrange section
  CudaResources res;
  auto up = [&](const uint8_t* src, size_t bytes) {
    void* d = res.device<unsigned char>(bytes);
    NZCP_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
    return d;
  };
  void* d_tau1 = up(pt.s[12].p + lvl * 64, n * 64);
  void* d_tau2 = up(pt.s[13].p + lvl * 128, n * 128);
  void* d_alpha = up(pt.s[14].p + lvl * 64, n * 64);
  void* d_beta = up(pt.s[15].p + lvl * 64, n * 64);
  const Fr* d_coefs = static_cast<const Fr*>(up(reinterpret_cast<const uint8_t*>(pool.data()), pool.size() * sizeof(Fr)));

  // ---- write the file in zkey_new.js's order
  Writer w(out, cap);
  w.raw("zkey", 4);
  w.u32(1);
  w.u32(10);
  w.section(1, 4);
  w.u32(1);                                                  // groth16
  w.section(2, kZkeyHeaderLen);
  w.u32(32); w.raw(kQBytes, 32);
  w.u32(32); w.raw(kRBytes, 32);
  w.u32(m); w.u32(np); w.u32((uint32_t)n);
  w.raw(pt.s[4].p, 64);                                      // alpha1 = alphaTauG1[0]
  w.raw(pt.s[5].p, 64);                                      // beta1  = betaTauG1[0]
  w.raw(pt.s[6].p, 128);                                     // beta2
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  w.raw(&g2, 128);                                           // gamma2
  w.raw(&g1, 64);                                            // delta1
  w.raw(&g2, 128);                                           // delta2
  // section 4: coef * R^2 mod r (Montgomery form of the Montgomery form), A and B terms in file order, then the public rows
  const uint64_t n_coefs = r.n_terms[0] + r.n_terms[1] + np + 1;
  w.section(4, 4 + n_coefs * 44);
  w.u32((uint32_t)n_coefs);
  walk([&](int mtx, uint32_t c, uint32_t s, const uint8_t* coef, uint32_t) {
    if (mtx == 2) return;
    w.u32((uint32_t)mtx); w.u32(c); w.u32(s);
    Fr k;
    memcpy(k.v, coef, 32);
    k = fp_to_mont(fp_to_mont(k));
    w.raw(k.v, 32);
  });
  for (uint32_t s = 0; s <= np; s++) {
    w.u32(0); w.u32(nc + s); w.u32(s);
    w.raw(Fr::r2().v, 32);
  }
  // K = beta*A + alpha*B + C per wire -> IC (section 3) and C (section 8)
  std::vector<uint8_t> kbuf((size_t)m * 64);
  run_combo<Fq>(K, d_coefs, d_tau1, d_alpha, d_beta, m, kbuf.data());
  w.section(3, (uint64_t)(np + 1) * 64);
  w.raw(kbuf.data(), (size_t)(np + 1) * 64);
  // section 9: odd entries of the size-2n Lagrange level of tauG1
  w.section(9, n * 64);
  {
    const uint8_t* lv = pt.s[12].p + (2 * n - 1) * 64;
    uint8_t* dst = w.reserve(n * 64);
    for (uint64_t i = 0; i < n; i++) memcpy(dst + i * 64, lv + (2 * i + 1) * 64, 64);
  }
  w.section(8, (uint64_t)(m - np - 1) * 64);
  w.raw(kbuf.data() + (size_t)(np + 1) * 64, (size_t)(m - np - 1) * 64);
  w.section(5, (uint64_t)m * 64);
  run_combo<Fq>(A, d_coefs, d_tau1, nullptr, nullptr, m, w.reserve((size_t)m * 64));
  w.section(6, (uint64_t)m * 64);
  run_combo<Fq>(B, d_coefs, d_tau1, nullptr, nullptr, m, w.reserve((size_t)m * 64));
  w.section(7, (uint64_t)m * 128);
  run_combo<Fq2>(B, d_coefs, d_tau2, nullptr, nullptr, m, w.reserve((size_t)m * 128));
  w.section(10, 68);
  w.zeros(64);                                               // csHash: not computed (see the header of this file)
  w.u32(0);                                                  // no contributions
  if (w.pos != total) throw ApiError(NZCP_E_INTERNAL, "zkey new: size accounting error");
  if (written) *written = w.pos;
}

}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_zkey_new_size(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, size_t* out_size) {
  return api_guard([&] {
    if (!r1cs || !ptau || !out_size) throw ApiError(NZCP_E_ARG, "null argument");
    const R1cs r = parse_r1cs(r1cs, r1cs_len);
    const Ptau pt = parse_ptau(ptau, ptau_len);
    const uint32_t cp = circuit_power(r);
    if (cp > pt.power)
      throw ApiError(NZCP_E_ARG, "circuit too big for this power of tau ceremony. " + std::to_string(r.n_constraints) + "*2 > 2**" +
                                     std::to_string(pt.power));
    *out_size = zkey_new_size(r, cp);
  });
}

int nzcp_zkey_new(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, int device, uint8_t* out, size_t cap,
                  size_t* written) {
  return api_guard([&] {
    if (!r1cs || !ptau || !out) throw ApiError(NZCP_E_ARG, "null argument");
    zkey_new_impl(r1cs, r1cs_len, ptau, ptau_len, device, out, cap, written);
  });
}

}  // extern "C"
