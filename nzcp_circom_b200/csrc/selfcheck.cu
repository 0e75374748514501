// Format self-checks on a proving key (SURVEY.md 8c-3): the facts a snarkjs-made Groth16 .zkey must satisfy, checked
// without any reference implementation at hand -- so that the first REAL nzcp_exampleTest_final.zkey this library meets
// (the files ignored at /root/reference/.gitignore:2-4, produced by the CLI steps of /root/reference/Makefile:30-33) is
// validated before a proof is attempted against it:
//   * header: protocol = groth16, q and r are the BN254 moduli, domainSize a power of two >= nConstraints + nPublic + 1
//   * section 4: every coefficient value is canonical (< r); the LAST nPublic+1 records are the rows snarkjs zkey_new.js
//     appends for the public inputs -- (matrix A, constraint nConstraints+i, signal i, value R^2 mod r), i.e. the
//     Montgomery form of the Montgomery form of 1 (SURVEY.md F7) -- which pins the "coef * R^2" convention buildABC1 relies on
//   * sections 5-9 and the six header points: every point is the (0,0) infinity marker or satisfies the curve equation
//     (y^2 = x^3 + 3 on G1, y^2 = x^3 + 3/(9+u) on the twist) in Montgomery form, with canonical coordinates
// The point checks run on the GPU (one thread per point); the rest is a host scan.
#include <memory>

#include "api_util.cuh"

namespace nzcp {

G1Affine g1_generator();  // synth.cu
G2Affine g2_generator();

// counts[0] += points off the curve (or with a non-canonical coordinate), counts[1] += infinity markers
template <class F>
__global__ void __launch_bounds__(128) curve_check_kernel(const Affine<F>* __restrict__ pts, size_t n, F b, unsigned long long* counts) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false, inf = false;
  if (i < n) bad = !point_ok(pts[i], b, &inf);
  const unsigned bad_mask = __ballot_sync(0xffffffffu, bad), inf_mask = __ballot_sync(0xffffffffu, inf);
  if ((threadIdx.x & 31) == 0) {
    if (bad_mask) atomicAdd(&counts[0], (unsigned long long)__popc(bad_mask));
    if (inf_mask) atomicAdd(&counts[1], (unsigned long long)__popc(inf_mask));
  }
}

template <class F>
static void check_section(const uint8_t* host, size_t n_points, const F& b, uint64_t* off_curve, uint64_t* infinity) {
  *off_curve = 0;
  *infinity = 0;
  if (!n_points) return;
  const size_t bytes = n_points * sizeof(Affine<F>);
  void* d = nullptr;
  unsigned long long* d_counts = nullptr;
  NZCP_CUDA(cudaMalloc(&d, bytes));
  struct Guard { void* a; void* b; ~Guard() { cudaFree(a); cudaFree(b); } } gd{d, nullptr};
  NZCP_CUDA(cudaMalloc((void**)&d_counts, 2 * sizeof(unsigned long long)));
  gd.b = d_counts;
  NZCP_CUDA(cudaMemset(d_counts, 0, 2 * sizeof(unsigned long long)));
  NZCP_CUDA(cudaMemcpy(d, host, bytes, cudaMemcpyHostToDevice));
  curve_check_kernel<F><<<div_up(n_points, 128), 128>>>(reinterpret_cast<const Affine<F>*>(d), n_points, b, d_counts);
  NZCP_LAUNCH_CHECK();
  unsigned long long c[2];
  NZCP_CUDA(cudaMemcpy(c, d_counts, sizeof c, cudaMemcpyDeviceToHost));
  *off_curve = c[0];
  *infinity = c[1];
}

static uint32_t rd32s(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static uint64_t rd64s(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

static void selfcheck_impl(const uint8_t* b, size_t len, int device, nzcp_zkey_check* rep) {
  memset(rep, 0, sizeof *rep);
  // container (binfileutils): magic, version, nSections, (u32 id, u64 len, payload)*
  if (len < 12 || memcmp(b, "zkey", 4) != 0) throw ApiError(NZCP_E_FORMAT, "zkey file: Invalid File format");
  struct Sec { const uint8_t* p = nullptr; uint64_t len = 0; } s[11];
  size_t pos = 12;
  for (uint32_t i = 0, nsec = rd32s(b + 8); i < nsec; i++) {
    if (pos + 12 > len) throw ApiError(NZCP_E_FORMAT, "truncated section table");
    const uint32_t id = rd32s(b + pos);
    const uint64_t sl = rd64s(b + pos + 4);
    pos += 12;
    if (sl > len - pos) throw ApiError(NZCP_E_FORMAT, "section exceeds file size");
    if (id <= 10 && !s[id].p) { s[id].p = b + pos; s[id].len = sl; }
    pos += sl;
  }
  for (int id = 1; id <= 9; id++)
    if (!s[id].p) throw ApiError(NZCP_E_FORMAT, "zkey: missing section " + std::to_string(id));
  if (s[1].len < 4 || rd32s(s[1].p) != 1) throw ApiError(NZCP_E_NOT_GROTH16, "zkey file is not groth16");
  const uint8_t* h = s[2].p;
  const size_t hdr_len = 4 + 32 + 4 + 32 + 12 + 64 + 64 + 128 + 128 + 64 + 128;
  if (s[2].len < hdr_len) throw ApiError(NZCP_E_FORMAT, "zkey: short header");
  rep->header_moduli_ok = rd32s(h) == 32 && rd32s(h + 36) == 32 && memcmp(h + 4, kQBytes, 32) == 0 && memcmp(h + 40, kRBytes, 32) == 0;
  if (!rep->header_moduli_ok) throw ApiError(NZCP_E_CURVE, "zkey: curve is not bn128");
  rep->n_vars = rd32s(h + 72);
  rep->n_public = rd32s(h + 76);
  rep->domain_size = rd32s(h + 80);
  const uint64_t m = rep->n_vars, npub = rep->n_public, n = rep->domain_size;
  if (n < 2 || (n & (n - 1)) != 0 || npub + 1 > m) throw ApiError(NZCP_E_FORMAT, "zkey: inconsistent header dimensions");
  if (s[3].len != (npub + 1) * 64 || s[5].len != m * 64 || s[6].len != m * 64 || s[7].len != m * 128 ||
      s[8].len != (m - npub - 1) * 64 || s[9].len != n * 64)
    throw ApiError(NZCP_E_FORMAT, "zkey: point section size does not match header");
  if (s[4].len < 4) throw ApiError(NZCP_E_FORMAT, "zkey: short coefficient section");
  const uint64_t nc = rd32s(s[4].p);
  if (s[4].len != 4 + nc * 44) throw ApiError(NZCP_E_FORMAT, "zkey: coefficient section size mismatch");
  rep->n_coefs = nc;
  // section 4 scan
  const uint8_t* cp = s[4].p + 4;
  uint64_t bad_val = 0, bad_idx = 0;
  for (uint64_t i = 0; i < nc; i++) {
    const uint8_t* rec = cp + i * 44;
    if (rd32s(rec) > 1 || rd32s(rec + 4) >= n || rd32s(rec + 8) >= m) bad_idx++;
    if (!fr_bytes_canonical(rec + 12)) bad_val++;
  }
  rep->bad_coef_values = bad_val;
  rep->bad_coef_indices = bad_idx;
  // the appended public-input rows: last nPublic+1 records = (0, nConstraints + i, i, R^2 mod r)
  uint8_t r2b[32];
  fp_to_bytes(Fr::r2(), r2b);      // R^2 mod r
  rep->public_rows_ok = nc >= npub + 1;
  if (rep->public_rows_ok) {
    const uint8_t* tail = cp + (nc - npub - 1) * 44;
    const uint32_t c0 = rd32s(tail + 4);
    rep->n_constraints = c0;
    for (uint64_t i = 0; i <= npub; i++) {
      const uint8_t* rec = tail + i * 44;
      if (rd32s(rec) != 0 || rd32s(rec + 4) != c0 + i || rd32s(rec + 8) != i || memcmp(rec + 12, r2b, 32) != 0) rep->public_rows_ok = 0;
    }
    if ((uint64_t)c0 + npub + 1 > n) rep->public_rows_ok = 0;
  }
  // points
  use_device(device);
  const Fq b1 = curve_b(g1_generator());
  const Fq2 b2 = curve_b(g2_generator());
  check_section<Fq>(s[5].p, m, b1, &rep->off_curve[0], &rep->infinity[0]);
  check_section<Fq>(s[6].p, m, b1, &rep->off_curve[1], &rep->infinity[1]);
  check_section<Fq2>(s[7].p, m, b2, &rep->off_curve[2], &rep->infinity[2]);
  check_section<Fq>(s[8].p, m - npub - 1, b1, &rep->off_curve[3], &rep->infinity[3]);
  check_section<Fq>(s[9].p, n, b1, &rep->off_curve[4], &rep->infinity[4]);
  check_section<Fq>(s[3].p, npub + 1, b1, &rep->off_curve[5], &rep->infinity[5]);
  // header points (host): alpha1, beta1, beta2, gamma2, delta1, delta2 -- on the curve and not infinity
  const uint8_t* pp = h + 84;
  bool inf = false, ok = true;
  G1Affine g1p;
  G2Affine g2p;
  memcpy(&g1p, pp, 64); ok = ok && point_ok(g1p, b1, &inf) && !inf; pp += 64;       // alpha1
  memcpy(&g1p, pp, 64); ok = ok && point_ok(g1p, b1, &inf) && !inf; pp += 64;       // beta1
  memcpy(&g2p, pp, 128); ok = ok && point_ok(g2p, b2, &inf) && !inf; pp += 128;     // beta2
  memcpy(&g2p, pp, 128); ok = ok && point_ok(g2p, b2, &inf) && !inf; pp += 128;     // gamma2
  memcpy(&g1p, pp, 64); ok = ok && point_ok(g1p, b1, &inf) && !inf; pp += 64;       // delta1
  memcpy(&g2p, pp, 128); ok = ok && point_ok(g2p, b2, &inf) && !inf;                // delta2
  rep->header_points_ok = ok;
  uint64_t off = 0;
  for (int k = 0; k < 6; k++) off += rep->off_curve[k];
  rep->ok = rep->header_moduli_ok && rep->header_points_ok && rep->public_rows_ok && off == 0 && bad_val == 0 && bad_idx == 0;
}

}  // namespace nzcp

using namespace nzcp;

extern "C" int nzcp_zkey_selfcheck(const uint8_t* bytes, size_t len, int device, nzcp_zkey_check* report) {
  return api_guard([&] {
    if (!bytes || !report) throw ApiError(NZCP_E_ARG, "null argument");
    selfcheck_impl(bytes, len, device, report);
  });
}
