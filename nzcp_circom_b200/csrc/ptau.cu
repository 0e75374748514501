// `powersoftau prepare phase2` on the GPU: the Lagrange-basis sections 12-15 of a powers-of-tau file, computed from its
// monomial sections 2-5 by an inverse FFT whose elements are curve points.
//
// Replaces snarkjs 0.4.12 src/powersoftau_preparephase2.js preparePhase2(oldPtauFilename, newPTauFilename) (upstream, not
// vendored: package.json:12, yarn.lock:987-999).  What it computes, restated:
//   header     section 1 rewritten by writePTauHeader(curve, power): n8, q, power, ceremonyPower = power
//   copied     sections 2, 3, 4, 5, 6, 7 verbatim; sections 12-15 of the input, if any, are ignored and recomputed
//   section 12 from 2 (tauG1), levels p = 0 .. power+1; 13 from 3 (tauG2), 14 from 4 (alphaTauG1), 15 from 5 (betaTauG1),
//              levels p = 0 .. power.  Level p = the 2^p affine points L_i = (1/N) sum_j w^(-ij) P_j, N = 2^p,
//              w = ffjavascript Fr.w[p], natural order, written back to back (level p starts at point 2^p - 1).
//   The top tauG1 level reads the 2^(power+1) - 1 points section 2 holds and, like snarkjs, puts the point at infinity
//   in the last slot: it is L_i(tau) - w^i tau^(N-1) / N, not the exact Lagrange basis.  `zkey new` reads it only for
//   section 9 (H) at cirPower == power; proofs are unaffected (the coefficient of x^(N-1) of A*B - C is zero).
//   Output container: 11 sections in the order 1-7, 12-15.
// Every affine point has one Montgomery encoding, so any correct algorithm gives these exact bytes.
//
// B200 design.  Per output section: one buffer holding all its levels in the output layout; the points stay AFFINE
// between launches (one division-step inversion per point written, ~2 % of a butterfly) so the buffer is the output
// itself and a tauG1 section at power 27 (2^29 points) takes 34 GB instead of 68 GB as XYZZ.
//   load   slot i of level p = (1/2^p) * P[bitrev_p(i)]  (the 1/N of the iFFT folded into the gather)
//   stage  radix-2 DIT stage s over EVERY level p > s of the section in one launch: 2^T - 2^s butterflies for a section
//          of top level T, so no launch has fewer than 2^(T-1) of them.  Butterfly: t = w^(-k) * b (signed 4-bit
//          windows, ec.cuh scalar_mul_accumulate), (a + t, a - t) by mixed additions.  ~3 300 Fq products per G1
//          butterfly against 256 bytes moved: integer-multiplier bound, no shared-memory tiling.  The stage-s twiddle is a root of order
//          2^(s+1) whatever the level, so one table w_top^(-k), k < 2^power, serves every level of every section.
// Sections are computed one after the other (their times are reported apart); all of them are validated on the host
// first: container, sizes, canonical coordinates and curve membership of every input point.

#include "binfile.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ shared host/device code
// tw[k] = w^k, plain form, for a Montgomery-form w
HD Fr pow_u32_plain(Fr w, uint32_t e) {
  Fr r = Fr::one();
  for (; e; e >>= 1) {
    if (e & 1) r = fp_mul(r, w);
    w = fp_sqr(w);
  }
  return fp_from_mont(r);
}

// Slot i (< 2^(T+1) - 1) of a section: level p = floor(log2(i + 1)), position j = i + 1 - 2^p.  src holds n_src points;
// an index past them reads as infinity (the pad of the top tauG1 level).  ninv[p] = 2^-p (plain).
template <class F>
HD Affine<F> prep_load(const Affine<F>* src, uint64_t n_src, const Fr* ninv, uint64_t i) {
  const int p = ilog2_u64(i + 1);
  const uint64_t j = bitrev_bits(i + 1 - ((uint64_t)1 << p), p);
  XYZZ<F> acc = XYZZ<F>::inf();
  if (j < n_src) scalar_mul_accumulate(acc, src[j], ninv[p]);
  return to_affine_fast(acc);
}

template <class F>
HD XYZZ<F> add_affine(XYZZ<F> t, const Affine<F>& a) {
  if (!a.is_inf()) xyzz_madd(t, a, false);
  return t;
}

// Butterfly u (< 2^T - 2^s) of DIT stage s over the levels p = s+1 .. T of a section laid out as prep_load writes it.
// Levels before p contribute 2^(p-1) - 2^s butterflies, so v = u + 2^s lies in [2^(p-1), 2^p).  tw[k] = w^(-k) with
// w = Fr.w[t_log], k < 2^(t_log - 1); the stage needs the root of order 2^(s+1): tw[k << (t_log - 1 - s)].
template <class F>
HD void prep_butterfly(Affine<F>* x, const Fr* tw, int t_log, int s, uint64_t u) {
  const uint64_t half = (uint64_t)1 << s;
  const uint64_t v = u + half;
  const int p = ilog2_u64(v) + 1;
  const uint64_t b = v - ((uint64_t)1 << (p - 1));
  const uint64_t k = b & (half - 1);
  const uint64_t i0 = ((uint64_t)1 << p) - 1 + ((b >> s) << (s + 1)) + k, i1 = i0 + half;
  const Affine<F> a = x[i0];
  XYZZ<F> t = XYZZ<F>::inf();
  scalar_mul_accumulate(t, x[i1], tw[k << (t_log - 1 - s)]);
  x[i0] = to_affine_fast(add_affine(t, a));
  x[i1] = to_affine_fast(add_affine(xyzz_neg(t), a));
}

// ------------------------------------------------------------------------------------------------ Exec ops
struct PtauTwiddle {
  Fr* tw;
  Fr w;
  HD void operator()(uint64_t k) const { tw[k] = pow_u32_plain(w, (uint32_t)k); }
};

template <class F>
struct PtauLoad {
  const Affine<F>* src;
  uint64_t n_src;
  const Fr* ninv;
  Affine<F>* x;
  HD void operator()(uint64_t i) const { x[i] = prep_load(src, n_src, ninv, i); }
};

template <class F>
struct PtauStage {
  Affine<F>* x;
  const Fr* tw;
  int t_log, s;
  HD void operator()(uint64_t u) const { prep_butterfly(x, tw, t_log, s, u); }
};

// ------------------------------------------------------------------------------------------------ host side
namespace {

constexpr uint32_t kHostMaxPower = 4;

// Everything preparePhase2 needs from its input, validated before any device work.
Ptau parse_prepare_in(const uint8_t* b, size_t len) {
  const Ptau p = read_ptau(b, len);
  if (p.power == kPtauMaxPower) throw ApiError(NZCP_E_ARG, kPtauPower28Phase2);
  check_ptau_sections(p);
  return p;
}

// One output section: its source section, group and top level.
struct OutSect {
  uint32_t id, src;
  bool g2;
  uint32_t top;
};

void out_sects(uint32_t power, OutSect o[4]) {
  o[0] = {12, 2, false, power + 1};
  o[1] = {13, 3, true, power};
  o[2] = {14, 4, false, power};
  o[3] = {15, 5, false, power};
}

uint64_t level_points(uint32_t top) { return ((uint64_t)2 << top) - 1; }   // levels 0 .. top back to back

size_t prepare_size(const Ptau& p) {
  size_t total = 12 + 11 * 12 + kPtauHeaderLen;
  for (int id = 2; id <= 7; id++) total += p.s[id].len;
  OutSect o[4];
  out_sects(p.power, o);
  for (const OutSect& s : o) total += level_points(s.top) * (s.g2 ? 128 : 64);
  return total;
}

// 2^-p for p = 0 .. top (plain)
std::vector<Fr> ninv_table(uint32_t top) {
  Fr two = Fr::zero();
  two.v[0] = 2;
  const Fr half = fp_inv(fp_to_mont(two));
  std::vector<Fr> t(top + 1);
  Fr acc = Fr::one();
  for (uint32_t p = 0; p <= top; p++) {
    t[p] = fp_from_mont(acc);
    acc = fp_mul(acc, half);
  }
  return t;
}

// One output section: load, then every stage; returns their device ms.  Its buffers are freed when it is written.
template <class F>
float run_section(bool host, const uint8_t* src, uint64_t n_src, uint32_t top, const Fr* ninv, const Fr* tw, int t_log,
                  uint8_t* out) {
  const uint64_t n = level_points(top);
  Exec ex(host);
  Affine<F>* in = ex.alloc<Affine<F>>(n_src);   // n_src, n > 0
  Affine<F>* x = ex.alloc<Affine<F>>(n);
  ex.upload(in, src, n_src * sizeof(Affine<F>));
  Timer t = ex.timer();
  ex.run<128>(n, PtauLoad<F>{in, n_src, ninv, x});
  for (uint32_t s = 0; s < top; s++) ex.run<128>(((uint64_t)1 << top) - ((uint64_t)1 << s), PtauStage<F>{x, tw, t_log, (int)s});
  const float ms = t.stop();
  ex.download(out, x, n * sizeof(Affine<F>));
  return ms;
}

// device < 0: the host hook.
void prepare_impl(const uint8_t* b, size_t len, int device, uint8_t* out, size_t cap, size_t* written, float* section_ms) {
  const Ptau p = parse_prepare_in(b, len);
  const size_t total = prepare_size(p);
  if (cap < total) throw ApiError(NZCP_E_ARG, "output buffer too small");
  const bool host = device < 0;
  if (host && p.power > kHostMaxPower) throw ApiError(NZCP_E_ARG, "ptau: the host run is limited to power 4");
  if (!host) use_device(device);

  OutSect os[4];
  out_sects(p.power, os);
  const int t_log = (int)p.power + 1;                       // twiddle table: w^(-k), w = Fr.w[power + 1], k < 2^power
  const uint64_t n_tw = (uint64_t)1 << p.power;
  const Fr w_inv = fp_inv(host_fr_root(t_log));
  const std::vector<Fr> ninv_h = ninv_table(p.power + 1);
  Exec ex(host);
  Fr* tw = ex.alloc<Fr>(n_tw);
  Fr* ninv = ex.alloc<Fr>(ninv_h.size());
  ex.upload(ninv, ninv_h.data(), ninv_h.size() * sizeof(Fr));
  ex.run<256>(n_tw, PtauTwiddle{tw, w_inv});

  Writer w(out, cap);
  write_ptau_header(w, p.power, 11);
  for (int id = 2; id <= 7; id++) {
    w.section(id, p.s[id].len);
    w.raw(p.s[id].p, p.s[id].len);
  }
  for (int k = 0; k < 4; k++) {
    const OutSect& o = os[k];
    const uint64_t n = level_points(o.top);
    const size_t psz = o.g2 ? 128 : 64;
    w.section(o.id, n * psz);
    uint8_t* dst = w.reserve(n * psz);
    const uint64_t n_src = p.s[o.src].len / psz;           // 2^top, or 2^top - 1 for tauG1 (the top level's pad)
    const float ms = o.g2 ? run_section<Fq2>(host, p.s[o.src].p, n_src, o.top, ninv, tw, t_log, dst)
                          : run_section<Fq>(host, p.s[o.src].p, n_src, o.top, ninv, tw, t_log, dst);
    if (section_ms) section_ms[k] = ms;
  }
  if (w.pos != total) throw ApiError(NZCP_E_INTERNAL, "ptau prepare: size accounting error");
  if (written) *written = w.pos;
}

}  // namespace
}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_ptau_prepare_size(const uint8_t* ptau, size_t len, size_t* out_size) {
  return api_guard([&] {
    if (!ptau || !out_size) throw ApiError(NZCP_E_ARG, "null argument");
    *out_size = prepare_size(parse_prepare_in(ptau, len));
  });
}

int nzcp_ptau_prepare(const uint8_t* ptau, size_t len, int device, uint8_t* out, size_t cap, size_t* written,
                      float section_ms[4]) {
  return api_guard([&] {
    if (!ptau || !out) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    prepare_impl(ptau, len, device, out, cap, written, section_ms);
  });
}

int nzcp_host_ptau_prepare(const uint8_t* ptau, size_t len, uint8_t* out, size_t cap, size_t* written) {
  return api_guard([&] {
    if (!ptau || !out) throw ApiError(NZCP_E_ARG, "null argument");
    prepare_impl(ptau, len, -1, out, cap, written, nullptr);
  });
}

}  // extern "C"
