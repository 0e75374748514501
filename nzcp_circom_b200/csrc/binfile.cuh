// binfileutils containers (snarkjs .r1cs / .wtns / .ptau / .zkey) and the Groth16 .zkey and .ptau headers: the only code
// that knows their byte layout.  The section-table reader, the .zkey and .ptau header readers with the checks every entry
// shares, the .ptau section geometry, the output writer and the point check; and the .r1cs / prepared .ptau readers and
// `zkey new` of setup.cu.
#pragma once
#include <algorithm>
#include <thread>

#include "api_util.cuh"

namespace nzcp {

static inline uint32_t rd32u(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline uint64_t rd64u(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

struct Sect { const uint8_t* p = nullptr; uint64_t len = 0; };

// binfileutils readBinFile: magic, version, nSections, then (u32 id, u64 len, payload)*.  secs[id] = first section with
// that id, for id <= max_id; later duplicates are ignored.
static inline void parse_bin(const uint8_t* b, size_t len, const char* magic, Sect* secs, int max_id,
                             uint32_t max_version = 1) {
  if (len < 12 || memcmp(b, magic, 4) != 0) throw ApiError(NZCP_E_FORMAT, std::string(magic) + " file: Invalid File format");
  if (rd32u(b + 4) > max_version) throw ApiError(NZCP_E_FORMAT, "Version not supported");
  size_t pos = 12;
  for (uint32_t i = 0, n = rd32u(b + 8); i < n; i++) {
    if (pos + 12 > len) throw ApiError(NZCP_E_FORMAT, "truncated section table");
    const uint32_t id = rd32u(b + pos);
    const uint64_t sl = rd64u(b + pos + 4);
    pos += 12;
    if (sl > len - pos) throw ApiError(NZCP_E_FORMAT, "section exceeds file size");
    // unsigned compare: a section id >= 2^31 must not index backwards
    if (id <= (uint32_t)max_id && !secs[id].p) { secs[id].p = b + pos; secs[id].len = sl; }
    pos += sl;
  }
}

inline void need_sections(const Sect* secs, int first, int last) {
  for (int id = first; id <= last; id++)
    if (!secs[id].p) throw ApiError(NZCP_E_FORMAT, "Missing section " + std::to_string(id));
}

struct Writer {
  uint8_t* p;
  size_t cap, pos = 0;
  Writer(uint8_t* b, size_t c) : p(b), cap(c) {}
  void need(size_t n) { if (pos + n > cap) throw ApiError(NZCP_E_ARG, "output buffer too small"); }
  void u32(uint32_t v) { need(4); memcpy(p + pos, &v, 4); pos += 4; }
  void u64(uint64_t v) { need(8); memcpy(p + pos, &v, 8); pos += 8; }
  void raw(const void* s, size_t n) { need(n); memcpy(p + pos, s, n); pos += n; }
  void zeros(size_t n) { need(n); memset(p + pos, 0, n); pos += n; }
  uint8_t* reserve(size_t n) { need(n); uint8_t* q = p + pos; pos += n; return q; }
  void section(uint32_t id, uint64_t len) { u32(id); u64(len); }
};

// Every point of a section of n affine points must be the (0,0) marker or have canonical coordinates and lie on the curve
// y^2 = x^3 + b.  Scanned by all host threads; throws NZCP_E_RANGE naming the first offending point ("<what>: section
// <sec> point <i> ...").
template <class F>
void check_points(const char* what, const uint8_t* p, uint64_t n, int sec, const F& b) {
  // first offending point of each thread's chunk; 1 = coordinate >= q, 2 = off the curve
  const unsigned nt = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
  const uint64_t chunk = (n + nt - 1) / nt;
  std::vector<uint64_t> first(nt, UINT64_MAX);
  std::vector<int> kind(nt, 0);
  auto scan = [&](unsigned t) {
    for (uint64_t i = t * chunk; i < std::min(n, (t + 1) * chunk); i++) {
      Affine<F> a;
      memcpy(&a, p + i * sizeof(Affine<F>), sizeof(Affine<F>));
      bool inf;
      if (a.is_inf()) continue;
      const int k = !(CoordCanon<F>::ok(a.x) && CoordCanon<F>::ok(a.y)) ? 1 : !point_ok(a, b, &inf) ? 2 : 0;
      if (k) { first[t] = i; kind[t] = k; return; }
    }
  };
  if (n < 4096) {
    for (unsigned t = 0; t < nt; t++) scan(t);
  } else {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++) th.emplace_back(scan, t);
    for (auto& t : th) t.join();
  }
  for (unsigned t = 0; t < nt; t++)
    if (kind[t])
      throw ApiError(NZCP_E_RANGE, std::string(what) + ": section " + std::to_string(sec) + " point " + std::to_string(first[t]) +
                                       (kind[t] == 1 ? " has a coordinate >= q" : " is not on the curve"));
}

// ------------------------------------------------------------------------------------------------ .zkey (Groth16)
// zkey_utils.js readHeader / readHeaderGroth16.  Section 1: u32 protocol (1 = groth16).  Section 2: u32 n8q, q, u32 n8r,
// r, u32 nVars, nPublic, domainSize, then alpha1, beta1 (G1), beta2, gamma2 (G2), delta1 (G1), delta2 (G2) as Montgomery
// affine points.  Sections 3-9 hold IC, the coefficients, A, B1, B2, C (the private wires) and H; 10 the MPC parameters.
constexpr size_t kZkeyNVarsOff = 72, kZkeyNPublicOff = 76, kZkeyDomainOff = 80;
constexpr size_t kZkeyAlpha1Off = 84, kZkeyBeta1Off = 148, kZkeyBeta2Off = 212, kZkeyGamma2Off = 340, kZkeyDelta1Off = 468,
                 kZkeyDelta2Off = 532;
constexpr size_t kZkeyHeaderLen = 660;

struct Zkey {
  Sect s[11];
  uint32_t n_vars = 0, n_public = 0, domain_size = 0;
  uint64_t n_l() const { return (uint64_t)n_vars - n_public - 1; }   // points of section 8
};

// The checks every .zkey entry shares: a Groth16 key over bn128 whose header holds nPublic + 1 <= nVars.  Sections 3-10
// and the header's points are left to the entry that reads them.
inline Zkey read_zkey(const uint8_t* b, size_t len) {
  Zkey z;
  parse_bin(b, len, "zkey", z.s, 10);
  if (!z.s[1].p || z.s[1].len < 4) throw ApiError(NZCP_E_FORMAT, "zkey: missing header");
  if (rd32u(z.s[1].p) != 1) throw ApiError(NZCP_E_NOT_GROTH16, "zkey file is not groth16");
  need_sections(z.s, 2, 2);
  const uint8_t* h = z.s[2].p;
  if (z.s[2].len < kZkeyHeaderLen) throw ApiError(NZCP_E_FORMAT, "zkey: header section 2 is not 660 bytes");
  if (rd32u(h) != 32 || memcmp(h + 4, kQBytes, 32) != 0 || rd32u(h + 36) != 32 || memcmp(h + 40, kRBytes, 32) != 0)
    throw ApiError(NZCP_E_CURVE, "zkey: curve is not bn128");
  z.n_vars = rd32u(h + kZkeyNVarsOff);
  z.n_public = rd32u(h + kZkeyNPublicOff);
  z.domain_size = rd32u(h + kZkeyDomainOff);
  if ((uint64_t)z.n_public + 1 > z.n_vars) throw ApiError(NZCP_E_FORMAT, "zkey: more public signals than variables");
  return z;
}

// log2 of domainSize, which must be a power of two >= 2 wherever the key's polynomials are transformed.
inline uint32_t zkey_domain_power(const Zkey& z) {
  const uint32_t n = z.domain_size;
  if (n < 2 || (n & (n - 1))) throw ApiError(NZCP_E_FORMAT, "zkey: domainSize is not a power of two >= 2");
  uint32_t p = 0;
  while ((1u << p) < n) p++;
  return p;
}

// ------------------------------------------------------------------------------------------------ .ptau
// powersoftau_utils.js readPTauHeader: section 1 = u32 n8, q, u32 power, u32 ceremonyPower.  Sections 2-6 hold tauG1,
// tauG2, alphaTauG1, betaTauG1 and betaG2 (Montgomery affine), 7 the contributions, 12-15 the Lagrange basis of a
// prepared file.
constexpr size_t kPtauHeaderLen = 4 + 32 + 4 + 4;
constexpr uint32_t kPtauMaxPower = 28;
// Why no Lagrange sections exist at the top power (`prepare phase2` and `powersoftau verify` reject such files).
constexpr const char* kPtauPower28Phase2 = "ptau: power 28 is not supported: its top tauG1 level has 2^29 points, more "
                                           "than the 2^28 roots of unity of Fr, and needs the coset branch of snarkjs's "
                                           "lagrangeEvaluations";

struct Ptau {
  Sect s[16];
  uint32_t power = 0, ceremony_power = 0;
};

// The checks every .ptau entry shares: a bn128 file of power 1..28.
inline Ptau read_ptau(const uint8_t* b, size_t len) {
  Ptau p;
  parse_bin(b, len, "ptau", p.s, 15);
  const uint8_t* h = p.s[1].p;
  if (!h || p.s[1].len < kPtauHeaderLen) throw ApiError(NZCP_E_FORMAT, "ptau: missing header");
  if (rd32u(h) != 32 || memcmp(h + 4, kQBytes, 32) != 0) throw ApiError(NZCP_E_CURVE, "ptau: curve is not bn128");
  p.power = rd32u(h + 36);
  p.ceremony_power = rd32u(h + 40);
  if (p.power < 1 || p.power > kPtauMaxPower) throw ApiError(NZCP_E_FORMAT, "ptau: power out of range [1, 28]");
  return p;
}

// Section id (2..6) of a file of 2^power: 2^(power+1) - 1 tauG1 points, 2^power each of tauG2 / alphaTauG1 / betaTauG1,
// one betaG2.
inline uint64_t sect_points(uint32_t power, int id) {
  const uint64_t n = (uint64_t)1 << power;
  return id == 2 ? 2 * n - 1 : id == 6 ? 1 : n;
}
inline bool sect_g2(int id) { return id == 3 || id == 6; }
inline size_t sect_bytes(uint32_t power, int id) { return sect_points(power, id) * (sect_g2(id) ? 128 : 64); }

// The accumulator of a full (not reduced) file: sections 2-7 present, 2-6 sized for the power, every point of 2-6
// canonical and on its curve.
inline void check_ptau_sections(const Ptau& p) {
  need_sections(p.s, 2, 7);
  for (int id = 2; id <= 6; id++)
    if (p.s[id].len != sect_bytes(p.power, id))
      throw ApiError(NZCP_E_FORMAT, "ptau: section " + std::to_string(id) + " size does not match the header power");
  const Fq b1 = curve_b(g1_generator());
  const Fq2 b2 = curve_b(g2_generator());
  for (int id = 2; id <= 6; id++) {
    if (sect_g2(id)) check_points<Fq2>("ptau", p.s[id].p, sect_points(p.power, id), id, b2);
    else check_points<Fq>("ptau", p.s[id].p, sect_points(p.power, id), id, b1);
  }
}

// writePTauHeader: the container head for n_sections sections, then section 1 with ceremonyPower = power.
inline void write_ptau_header(Writer& w, uint32_t power, uint32_t n_sections) {
  w.raw("ptau", 4);
  w.u32(1);
  w.u32(n_sections);
  w.section(1, kPtauHeaderLen);
  w.u32(32);
  w.raw(kQBytes, 32);
  w.u32(power);
  w.u32(power);
}

// ------------------------------------------------------------------------------------------------ setup.cu
struct R1cs {
  uint32_t n_wires = 0, n_pub_out = 0, n_pub_in = 0, n_prv_in = 0, n_constraints = 0, n_public = 0;
  const uint8_t* cons = nullptr;
  uint64_t cons_len = 0;
  uint64_t n_terms[3] = {0, 0, 0};   // A, B, C terms in total
};

R1cs parse_r1cs(const uint8_t* b, size_t len);
Ptau parse_ptau(const uint8_t* b, size_t len);   // a prepared file: read_ptau, then sections 2-6 and 12-15
uint32_t circuit_power(const R1cs& r);
size_t zkey_new_size(const R1cs& r, uint32_t cir_power);
// snarkjs `zkey new` into out[0 .. cap); section 10 holds a zero circuit hash.
void zkey_new_impl(const uint8_t* r1cs_b, size_t r1cs_len, const uint8_t* ptau_b, size_t ptau_len, int device, uint8_t* out,
                   size_t cap, size_t* written);

}  // namespace nzcp
