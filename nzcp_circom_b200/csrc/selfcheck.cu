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

#include "binfile.cuh"

namespace nzcp {

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
  CudaResources res;
  void* d = res.device<unsigned char>(bytes);
  unsigned long long* d_counts = res.device<unsigned long long>(2);
  NZCP_CUDA(cudaMemset(d_counts, 0, 2 * sizeof(unsigned long long)));
  NZCP_CUDA(cudaMemcpy(d, host, bytes, cudaMemcpyHostToDevice));
  curve_check_kernel<F><<<div_up(n_points, 128), 128>>>(reinterpret_cast<const Affine<F>*>(d), n_points, b, d_counts);
  NZCP_LAUNCH_CHECK();
  unsigned long long c[2];
  NZCP_CUDA(cudaMemcpy(c, d_counts, sizeof c, cudaMemcpyDeviceToHost));
  *off_curve = c[0];
  *infinity = c[1];
}

static void selfcheck_impl(const uint8_t* b, size_t len, int device, nzcp_zkey_check* rep) {
  memset(rep, 0, sizeof *rep);
  const Zkey z = read_zkey(b, len);
  const Sect* s = z.s;
  need_sections(s, 3, 9);
  zkey_domain_power(z);
  rep->header_moduli_ok = 1;   // read_zkey refuses any other
  rep->n_vars = z.n_vars;
  rep->n_public = z.n_public;
  rep->domain_size = z.domain_size;
  const uint64_t m = rep->n_vars, npub = rep->n_public, n = rep->domain_size;
  if (s[3].len != (npub + 1) * 64 || s[5].len != m * 64 || s[6].len != m * 64 || s[7].len != m * 128 ||
      s[8].len != z.n_l() * 64 || s[9].len != n * 64)
    throw ApiError(NZCP_E_FORMAT, "zkey: point section size does not match header");
  if (s[4].len < 4) throw ApiError(NZCP_E_FORMAT, "zkey: short coefficient section");
  const uint64_t nc = rd32u(s[4].p);
  if (s[4].len != 4 + nc * 44) throw ApiError(NZCP_E_FORMAT, "zkey: coefficient section size mismatch");
  rep->n_coefs = nc;
  // section 4 scan
  const uint8_t* cp = s[4].p + 4;
  uint64_t bad_val = 0, bad_idx = 0;
  for (uint64_t i = 0; i < nc; i++) {
    const uint8_t* rec = cp + i * 44;
    if (rd32u(rec) > 1 || rd32u(rec + 4) >= n || rd32u(rec + 8) >= m) bad_idx++;
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
    const uint32_t c0 = rd32u(tail + 4);
    rep->n_constraints = c0;
    for (uint64_t i = 0; i <= npub; i++) {
      const uint8_t* rec = tail + i * 44;
      if (rd32u(rec) != 0 || rd32u(rec + 4) != c0 + i || rd32u(rec + 8) != i || memcmp(rec + 12, r2b, 32) != 0) rep->public_rows_ok = 0;
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
  check_section<Fq>(s[8].p, z.n_l(), b1, &rep->off_curve[3], &rep->infinity[3]);
  check_section<Fq>(s[9].p, n, b1, &rep->off_curve[4], &rep->infinity[4]);
  check_section<Fq>(s[3].p, npub + 1, b1, &rep->off_curve[5], &rep->infinity[5]);
  // header points (host): alpha1, beta1, beta2, gamma2, delta1, delta2 -- on the curve and not infinity
  const uint8_t* h = s[2].p;
  G1Affine g1p;
  G2Affine g2p;
  bool inf = false;
  auto g1_ok = [&](size_t off) { memcpy(&g1p, h + off, 64); return point_ok(g1p, b1, &inf) && !inf; };
  auto g2_ok = [&](size_t off) { memcpy(&g2p, h + off, 128); return point_ok(g2p, b2, &inf) && !inf; };
  rep->header_points_ok = g1_ok(kZkeyAlpha1Off) && g1_ok(kZkeyBeta1Off) && g2_ok(kZkeyBeta2Off) && g2_ok(kZkeyGamma2Off) &&
                          g1_ok(kZkeyDelta1Off) && g2_ok(kZkeyDelta2Off);
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
