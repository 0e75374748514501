// `zkey verify` on the GPU: the circuit hash of a Groth16 key and the checks of a contributed key against its circuit.
//
// Replaces snarkjs 0.4.12 src/zkey_verify_fromr1cs.js verifyFromR1cs(r1cs, ptau, zkey) (build the initial key with
// newZKey in memory, then verifyFromInit) and src/zkey_verify_frominit.js verifyFromInit(init, ptau, zkey) (upstream, not
// vendored: package.json:12, yarn.lock:987-999), and the circuit hash (csHash) of src/zkey_new.js newZKey.  Restated:
//   csHash   BLAKE2b-512 over U(alpha1) U(beta1) U(beta2) U(G2) U(G1) U(G2) (gamma2, delta1, delta2 of a new key), then
//            hashU32(nPublic + 1) IC, hashU32(N - 1) H', hashU32(nVars - nPublic - 1) C, hashU32(nVars) A, B1, B2
//            (sections 3, 8, 5, 6, 7); hashU32 = big-endian u32, U = the uncompressed encoding of mpc.cuh hash_g1/g2.
//            H' are not section 9 but d_i = tauG1[i + N] - tauG1[i] from ptau section 2 (hashHPoints).  Its chunk loop
//            passes min(N - 1, 2^14) points per chunk for every i < N - 1 in steps of 2^14: N - 1 points for N <= 2^14,
//            N points above (the count written stays N - 1).  The last difference then reads tauG1[2N - 1], which section
//            2 (2^(power+1) - 1 points) lacks when cirPower = power and N > 2^14; snarkjs reads the next section's bytes
//            there, so that case is rejected (NZCP_E_ARG) rather than hashed with anything else.
//   verify   1. per record i of section 10, the accumulated hash starting from the key's csHash: the transcript must be
//               BLAKE2b(acc || U(g1_s) || U(g1_sx)); g2_sp = hashToG2(transcript); sameRatio(g1_s, g1_sx, g2_sp,
//               g2_spx); sameRatio(curDelta, deltaAfter, g2_sp, g2_spx); a beacon record's g1_s and k * g1_s are rebuilt
//               from its parameters; acc += hashPubKey(record); curDelta = deltaAfter (starting from G1).
//            2. the headers: nVars, nPublic, domainSize; alpha1, beta1, beta2, gamma2 equal to the initial key's; delta1 =
//               curDelta; sameRatio(G1, curDelta, G2, delta2).
//            3. csHash equal to the initial key's.  4. sections 3-7 byte-identical to the initial key's.
//            5. L: R1 = sum rho_i L_init[i], R2 = sum rho_i L[i]; sameRatio(R1, R2, delta2, delta2_init).
//            6. H: r_i random for i < N - 1, r_(N-1) = 0; R1 = sum r_i d_i; r' = Fr.fft(-2 w_2N^m r_m), w_2N = Fr.w[cirPower
//               + 1]; R2 = sum r'_j H[j]; sameRatio(R1, R2, delta2, delta2_init).  Since H[j] = L^(2N)_(2j+1)(tau) / delta,
//               sum_j r'_j L^(2N)_(2j+1)(x) = sum_m r_m (x^(m+N) - x^m) for every x (tests/verify_cases.py derives it); it is
//               linear in the points, and r_(N-1) = 0 drops the only term that would read tauG1[2N - 1], which is also the
//               term in which snarkjs's top tauG1 level (the point at infinity for the missing power) differs.
// sameRatio(a, b, c, d) claims e(a, d) = e(b, c).  The pairings are NOT computed here: every claim up to the first failed
// check this file decides itself is returned as a record (plain affine points), and the caller checks them in order
// (nzcp_circom_b200/verifier.py, as groth16.verify does).  The verdict is the first false claim, else this file's failure,
// else true; the C ABI alone does not give it.
// Deviations: the L scalars are full-width draws of a ChaCha seeded with 32 OS-random bytes (snarkjs: 32-bit scalars from
// crypto.randomFillSync, which bound a forged L section's chance at 2^-32); points of the key's header, records and
// sections 8 and 9 must be canonical and on their curve, delta2 and every g2_spx in the order-r subgroup (a Miller loop on
// other points is not a pairing; snarkjs checks none of this) -- a bad point is a false verdict naming it.  An input that
// cannot be parsed is an error code, raised before any device work; a key that parses but fails a check is a false
// verdict, never an error.  Both keys must be over bn128 (an error otherwise), so snarkjs's "Different curves" cannot
// arise, and the section 8 / 9 sizes follow from the header check.
//
// B200 design.  The bulk of the circuit hash is the uncompressed encoding of ~1.9 M points at the NZCP shape (~350 MB):
// one kernel forms the H differences (one thread per point: a mixed XYZZ addition of -P_i, then to_affine_fast) and keeps
// them resident as the bases of the H check; a second converts Montgomery affine points to the big-endian encoding in
// chunks, so the host BLAKE2b of chunk j (one sequential stream) overlaps the conversion and copy of chunk j + 1.  The L
// and H combinations are variable-base MSMs (msm.cu, table-free), the H scalars pass through the Fr NTT on the device.
#include <sys/random.h>

#include "mpc.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ shared host/device code
// d = hi - lo (hi = tauG1[i + N], lo = tauG1[i])
HD G1Affine h_diff_point(const G1Affine& hi, const G1Affine& lo) {
  G1XYZZ acc = G1XYZZ::from_affine(hi);
  if (!lo.is_inf()) xyzz_madd(acc, lo, true);
  return to_affine_fast(acc);
}

__global__ void __launch_bounds__(128) h_diff_kernel(const G1Affine* __restrict__ tau, uint64_t N, G1Affine* __restrict__ out,
                                                     uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = h_diff_point(tau[i + N], tau[i]);
}

// r[m] <- -2 w^m r[m]: plain r, Montgomery w and -2, plain result.
__global__ void __launch_bounds__(256) h_scalar_kernel(Fr* __restrict__ r, uint64_t n, Fr w, Fr neg2) {
  const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  Fr p = Fr::one(), b = w;
  for (uint64_t e = m; e; e >>= 1) {
    if (e & 1) p = fp_mul(p, b);
    b = fp_sqr(b);
  }
  r[m] = fp_mul(fp_mul(r[m], p), neg2);
}

namespace {

constexpr uint64_t kHashHChunk = 1u << 14;    // hashHPoints CHUNK_SIZE

// Points hashHPoints passes to the hasher for a domain of N (see the header of this file).
uint64_t h_hash_points(uint64_t N) { return N - 1 <= kHashHChunk ? N - 1 : (N - 1 + kHashHChunk - 1) / kHashHChunk * kHashHChunk; }

// ------------------------------------------------------------------------------------------------ inputs
// A ptau whose section 2 covers what the circuit hash of a domain of N reads.
void check_ptau_for(const Ptau& pt, uint32_t cir_power) {
  const uint64_t n_tau = ((uint64_t)2 << pt.power) - 1;
  if (pt.s[2].len != n_tau * 64) throw ApiError(NZCP_E_FORMAT, "ptau: section size does not match the header power");
  if (cir_power > pt.power)
    throw ApiError(NZCP_E_ARG, "circuit too big for this power of tau ceremony. 2**" + std::to_string(cir_power) + " > 2**" +
                                   std::to_string(pt.power));
  const uint64_t N = (uint64_t)1 << cir_power;
  if (N + h_hash_points(N) > n_tau)
    throw ApiError(NZCP_E_ARG, "zkey verify: at cirPower = power = " + std::to_string(pt.power) +
                                   " snarkjs's hashHPoints reads tauG1[2^" + std::to_string(cir_power + 1) +
                                   " - 1], past the end of ptau section 2; the circuit hash is not defined there");
  check_points<Fq>("ptau", pt.s[2].p, N + h_hash_points(N), 2, curve_b(g1_generator()));
}

// The initial key: the sections the circuit hash reads must have the sizes its header gives.
void check_init_sections(const ZkeyIn& z) {
  const uint64_t m = z.n_vars, np = z.n_public;
  const uint64_t want[8] = {0, 0, 0, (np + 1) * 64, 0, m * 64, m * 64, m * 128};
  for (int id : {3, 5, 6, 7})
    if (z.s[id].len != want[id])
      throw ApiError(NZCP_E_FORMAT, "zkey: section " + std::to_string(id) + " size does not match the header");
}

// ------------------------------------------------------------------------------------------------ circuit hash
struct HDiff {
  uint64_t n = 0;                   // h_hash_points(N)
  std::unique_ptr<DevMem> d;        // device run: the differences, resident for the H check
  std::vector<G1Affine> h;          // host run
};

// csHash of the initial key zi (zkey_new.js order); the H differences are left in `diff`.
void circuit_hash(const ZkeyIn& zi, const Ptau& pt, bool host, uint8_t out[64], HDiff& diff, float* kernel_ms, float* blake_ms) {
  const uint8_t* hd = zi.s[2].p;
  const uint64_t N = zi.domain_size, m = zi.n_vars, np = zi.n_public;
  Hasher hs(host);
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  hs.points_host(reinterpret_cast<const G1Affine*>(hd + kZkeyAlpha1Off), 2);   // alpha1, beta1
  hs.points_host(reinterpret_cast<const G2Affine*>(hd + kZkeyBeta2Off), 1);    // beta2
  hs.points_host(&g2, 1);                                                      // gamma2
  hs.points_host(&g1, 1);                                                      // delta1
  hs.points_host(&g2, 1);                                                      // delta2
  hs.u32be((uint32_t)(np + 1));
  hs.section<Fq>(zi.s[3].p, np + 1);
  hs.u32be((uint32_t)(N - 1));
  diff.n = h_hash_points(N);
  float diff_ms = 0;
  if (host) {
    diff.h.resize(diff.n);
    const G1Affine* tau = reinterpret_cast<const G1Affine*>(pt.s[2].p);
    for (uint64_t i = 0; i < diff.n; i++) {
      G1Affine a, b;
      memcpy(&a, tau + i + N, 64);
      memcpy(&b, tau + i, 64);
      diff.h[i] = h_diff_point(a, b);
    }
    hs.points_host(diff.h.data(), diff.n);
  } else {
    DevMem d_tau((N + diff.n) * 64);
    diff.d.reset(new DevMem(diff.n * 64));
    NZCP_CUDA(cudaMemcpy(d_tau.p, pt.s[2].p, (N + diff.n) * 64, cudaMemcpyHostToDevice));
    Events ev;
    NZCP_CUDA(cudaEventRecord(ev.a, 0));
    h_diff_kernel<<<div_up(diff.n, 128), 128>>>(static_cast<const G1Affine*>(d_tau.p), N, static_cast<G1Affine*>(diff.d->p), diff.n);
    NZCP_LAUNCH_CHECK();
    NZCP_CUDA(cudaEventRecord(ev.b, 0));
    NZCP_CUDA(cudaEventSynchronize(ev.b));
    NZCP_CUDA(cudaEventElapsedTime(&diff_ms, ev.a, ev.b));
    hs.points_device(static_cast<const G1Affine*>(diff.d->p), diff.n);
  }
  hs.u32be((uint32_t)(m - np - 1));
  hs.section<Fq>(zi.s[8].p, m - np - 1);
  for (int id : {5, 6}) {
    hs.u32be((uint32_t)m);
    hs.section<Fq>(zi.s[id].p, m);
  }
  hs.u32be((uint32_t)m);
  hs.section<Fq2>(zi.s[7].p, m);
  hs.h.final(out);
  if (kernel_ms) *kernel_ms = hs.kernel_ms + diff_ms;
  if (blake_ms) *blake_ms = hs.blake_ms;
}

// ------------------------------------------------------------------------------------------------ verification
struct Verdict {   // the first failed check this file decides
  int step, record;
  std::string msg;
};

struct Rec {
  const uint8_t* p;
  uint32_t type, exp = 0;
  const uint8_t *name = nullptr, *beacon = nullptr;
  size_t name_len = 0, beacon_len = 0;
};

Rec read_record(const uint8_t* r) {
  Rec c{r, rd32u(r + 384)};
  const uint8_t* q = r + kRecFixed;
  const uint8_t* end = q + rd32u(r + 388);
  while (q < end) {   // parse_mpc has checked the layout
    const int tag = *q++;
    if (tag == 2) {
      c.exp = *q++;
    } else {
      const size_t l = *q++;
      (tag == 1 ? c.name : c.beacon) = q;
      (tag == 1 ? c.name_len : c.beacon_len) = l;
      q += l;
    }
  }
  if (c.type == 1 && (!c.beacon || c.beacon_len == 0 || c.exp > 63))
    throw ApiError(NZCP_E_FORMAT, "zkey: beacon record without a beacon hash or with numIterationsExp > 63");
  return c;
}

template <class F>
Affine<F> load_pt(const uint8_t* p) {
  Affine<F> a;
  memcpy(&a, p, sizeof a);
  return a;
}

bool in_g2_subgroup(const G2Affine& p) {
  uint32_t r[8];
  for (int i = 0; i < 8; i++) r[i] = FrParams::mod(i);
  return xyzz_mul(G2XYZZ::from_affine(p), r).is_inf();
}

// The points of the key under verification: a bad one is a false verdict (step 1) naming it.
void check_key_points(const ZkeyIn& z, const std::vector<Rec>& recs) {
  const Fq b1 = curve_b(g1_generator());
  const Fq2 b2 = curve_b(g2_generator());
  bool inf;
  auto g1 = [&](const uint8_t* p, const std::string& what) {
    if (!point_ok(load_pt<Fq>(p), b1, &inf)) throw Verdict{1, -1, "zkey: " + what + " is not a canonical point of G1"};
  };
  auto g2 = [&](const uint8_t* p, const std::string& what, bool subgroup) {
    const G2Affine a = load_pt<Fq2>(p);
    if (!point_ok(a, b2, &inf)) throw Verdict{1, -1, "zkey: " + what + " is not a canonical point of the twist"};
    if (subgroup && !in_g2_subgroup(a)) throw Verdict{1, -1, "zkey: " + what + " is not in the order-r subgroup of G2"};
  };
  const uint8_t* h = z.s[2].p;
  g1(h + kZkeyAlpha1Off, "header alpha1");
  g1(h + kZkeyBeta1Off, "header beta1");
  g2(h + kZkeyBeta2Off, "header beta2", false);
  g2(h + kZkeyGamma2Off, "header gamma2", false);
  g1(h + kZkeyDelta1Off, "header delta1");
  g2(h + kZkeyDelta2Off, "header delta2", true);
  for (size_t i = 0; i < recs.size(); i++) {
    const std::string w = "section 10 record " + std::to_string(i) + " ";
    g1(recs[i].p, w + "deltaAfter");
    g1(recs[i].p + 64, w + "g1_s");
    g1(recs[i].p + 128, w + "g1_sx");
    g2(recs[i].p + 192, w + "g2_spx", true);
  }
  try {
    check_points<Fq>("zkey", z.s[8].p, z.n_l(), 8, b1);
    check_points<Fq>("zkey", z.s[9].p, z.domain_size, 9, b1);
  } catch (const ApiError& e) {
    throw Verdict{1, -1, e.what()};
  }
}

void plain_g1(const G1Affine& a, uint8_t* o) {
  fp_to_bytes(fp_from_mont(a.x), o);
  fp_to_bytes(fp_from_mont(a.y), o + 32);
}
void plain_g2(const G2Affine& a, uint8_t* o) {
  fp_to_bytes(fp_from_mont(a.x.c0), o);
  fp_to_bytes(fp_from_mont(a.x.c1), o + 32);
  fp_to_bytes(fp_from_mont(a.y.c0), o + 64);
  fp_to_bytes(fp_from_mont(a.y.c1), o + 96);
}

struct Claims {
  nzcp_zkey_verify_claim* out;
  size_t n = 0;
  void add(int step, int record, const G1Affine& a, const G1Affine& b, const G2Affine& c, const G2Affine& d) {
    nzcp_zkey_verify_claim& k = out[n++];
    k.step = step;
    k.record = record;
    plain_g1(a, k.a);
    plain_g1(b, k.b);
    plain_g2(c, k.c);
    plain_g2(d, k.d);
  }
};

// Sum s_i P_i over n device-resident G1 bases with device-resident plain scalars (the table-free MSM of msm_plan.cu).
G1Affine msm_g1(void* d_bases, const Fr* d_scalars, size_t n) {
  if (n == 0) return G1Affine::inf();
  const int c = msm_pick_window_free(n);
  MsmTable tab;
  MsmSort sort;
  MsmRun run;
  struct Guard {
    MsmTable* t; MsmSort* s; MsmRun* r;
    ~Guard() { msm_run_destroy(r); msm_sort_destroy(s); msm_table_destroy(t); }
  } g{&tab, &sort, &run};
  msm_table_view(&tab, d_bases, n, false, c);
  msm_sort_create(&sort, n, c, -1, true);
  msm_run_create(&run, &sort, false);
  msm_sort_launch(&sort, d_scalars, n, 0);
  msm_run_launch(&run, &sort, &tab, 0);
  NZCP_CUDA(cudaStreamSynchronize(0));
  msm_sort_check(&sort);
  return xyzz_to_affine(msm_run_finish_g1(&run));
}

struct Inputs {
  ZkeyIn key, init;
  std::vector<Rec> recs;
  Ptau pt;
  uint32_t cir_power = 0;
};

void fill_records(const Inputs& in, nzcp_zkey_contribution* out) {
  for (size_t i = 0; i < in.recs.size(); i++) {
    const Rec& c = in.recs[i];
    nzcp_zkey_contribution& o = out[i];
    memset(&o, 0, sizeof o);
    Blake2b512 h;
    hash_pub_key(h, c.p);
    h.final(o.hash);
    o.type = c.type;
    o.num_iterations_exp = c.exp;
    o.name_len = (uint32_t)c.name_len;
    if (c.name) memcpy(o.name, c.name, c.name_len);
    o.beacon_hash_len = (uint32_t)c.beacon_len;
    if (c.beacon) memcpy(o.beacon_hash, c.beacon, c.beacon_len);
  }
}

// Everything after parsing.  init_hash: the csHash the key must carry (the initial key's section 10, or the hash computed
// from it when verifyFromR1cs built it).  Throws Verdict at the first failed check.
void verify_checks(const Inputs& in, const uint8_t* init_hash, const uint8_t* seed, Claims& cl, HDiff& diff, float* ms) {
  const ZkeyIn &z = in.key, &zi = in.init;
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  check_key_points(z, in.recs);

  // 1. the contributions
  Blake2b512 acc;
  acc.update(z.s[10].p, 64);
  G1Affine cur = g1;
  for (size_t i = 0; i < in.recs.size(); i++) {
    const Rec& c = in.recs[i];
    const std::string pre = "INVALID(" + std::to_string(i) + "): ";
    Blake2b512 ours = acc;
    hash_g1(ours, c.p + 64);
    hash_g1(ours, c.p + 128);
    uint8_t t[64];
    ours.final(t);
    if (memcmp(t, c.p + 320, 64) != 0) throw Verdict{2, (int)i, pre + "Inconsistent transcript"};
    const G2Affine g2_sp = hash_to_g2(c.p + 320);
    const G1Affine g1_s = load_pt<Fq>(c.p + 64), g1_sx = load_pt<Fq>(c.p + 128), after = load_pt<Fq>(c.p);
    const G2Affine g2_spx = load_pt<Fq2>(c.p + 192);
    cl.add(3, (int)i, g1_s, g1_sx, g2_sp, g2_spx);
    cl.add(4, (int)i, cur, after, g2_sp, g2_spx);
    if (c.type == 1) {
      uint8_t s[32];
      beacon_seed(c.beacon, c.beacon_len, c.exp, s);
      ChaCha rng(s);
      const Fr k = fp_from_mont(fp_from_rng<FrParams>(rng));
      const G1Affine e_s = point_from_rng(rng, curve_b(g1), nullptr);
      const G1Affine e_sx = mul_plain(e_s, k.v);
      if (memcmp(&e_s, c.p + 64, 64) != 0) throw Verdict{5, (int)i, pre + "Key of the beacon does not match. g1_s"};
      if (memcmp(&e_sx, c.p + 128, 64) != 0) throw Verdict{5, (int)i, pre + "Key of the beacon does not match. g1_sx"};
    }
    hash_pub_key(acc, c.p);
    cur = after;
  }

  // 2. the headers
  if (z.n_vars != zi.n_vars || z.n_public != zi.n_public || z.domain_size != zi.domain_size)
    throw Verdict{6, -1, "Different circuit parameters"};
  const uint8_t *h = z.s[2].p, *hi = zi.s[2].p;
  const struct { size_t off, len; const char* msg; } same[] = {{kZkeyAlpha1Off, 64, "Invalid alpha1"},
                                                              {kZkeyBeta1Off, 64, "Invalid beta1"},
                                                              {kZkeyBeta2Off, 128, "Invalid beta2"},
                                                              {kZkeyGamma2Off, 128, "Invalid gamma2"}};
  for (const auto& s : same)
    if (memcmp(h + s.off, hi + s.off, s.len) != 0) throw Verdict{7, -1, s.msg};
  if (memcmp(h + kZkeyDelta1Off, &cur, 64) != 0) throw Verdict{7, -1, "Invalid delta1"};
  const G2Affine delta2 = load_pt<Fq2>(h + kZkeyDelta2Off), delta2_init = load_pt<Fq2>(hi + kZkeyDelta2Off);
  cl.add(8, -1, g1, cur, g2, delta2);

  // 3. the circuit, 4. the sections that no contribution changes
  if (memcmp(z.s[10].p, init_hash, 64) != 0) throw Verdict{9, -1, "Circuit does not match"};
  const char* names[8] = {nullptr, nullptr, nullptr, "IC", "Coeffs", "A", "B1", "B2"};
  for (int id = 3; id <= 7; id++)
    if (z.s[id].len != zi.s[id].len || memcmp(z.s[id].p, zi.s[id].p, z.s[id].len) != 0)
      throw Verdict{10, -1, std::string(names[id]) + " section is not identical"};

  // the random scalars: L first, then H
  uint8_t sd[32];
  if (seed) {
    memcpy(sd, seed, 32);
  } else {
    for (size_t got = 0; got < sizeof sd;) {
      const ssize_t r = getrandom(sd + got, sizeof sd - got, 0);
      if (r <= 0) throw ApiError(NZCP_E_INTERNAL, "zkey verify: no OS randomness");
      got += (size_t)r;
    }
  }
  ChaCha rng(sd);
  const uint64_t N = z.domain_size, n_l = z.n_l();
  std::vector<Fr> sc(std::max(n_l, N));
  Events ev;
  auto timed = [&](float& acc_ms, auto&& fn) {   // device time of fn's work on the default stream, added to acc_ms
    NZCP_CUDA(cudaEventRecord(ev.a, 0));
    const G1Affine r = fn();
    NZCP_CUDA(cudaEventRecord(ev.b, 0));
    NZCP_CUDA(cudaEventSynchronize(ev.b));
    float t = 0;
    NZCP_CUDA(cudaEventElapsedTime(&t, ev.a, ev.b));
    acc_ms += t;
    return r;
  };

  // 5. L: sum rho_i L_init[i] and sum rho_i L[i]
  if (n_l) {
    for (uint64_t i = 0; i < n_l; i++) sc[i] = fp_from_rng<FrParams>(rng);
    DevMem d_sc(n_l * sizeof(Fr)), d_b(n_l * 64);
    NZCP_CUDA(cudaMemcpy(d_sc.p, sc.data(), n_l * sizeof(Fr), cudaMemcpyHostToDevice));
    NZCP_CUDA(cudaMemcpy(d_b.p, zi.s[8].p, n_l * 64, cudaMemcpyHostToDevice));
    const G1Affine r1 = timed(ms[2], [&] { return msm_g1(d_b.p, static_cast<const Fr*>(d_sc.p), n_l); });
    NZCP_CUDA(cudaMemcpy(d_b.p, z.s[8].p, n_l * 64, cudaMemcpyHostToDevice));
    const G1Affine r2 = timed(ms[2], [&] { return msm_g1(d_b.p, static_cast<const Fr*>(d_sc.p), n_l); });
    cl.add(11, -1, r1, r2, delta2, delta2_init);
  }

  // 6. H: r_(N-1) = 0, R1 over the differences i <= N - 2, r' = Fr.fft(-2 w_2N^m r_m), R2 over section 9
  for (uint64_t i = 0; i + 1 < N; i++) sc[i] = fp_from_rng<FrParams>(rng);
  sc[N - 1] = Fr::zero();
  DevMem d_r(N * sizeof(Fr)), d_tmp(N * sizeof(Fr)), d_h(N * 64);
  NZCP_CUDA(cudaMemcpy(d_r.p, sc.data(), N * sizeof(Fr), cudaMemcpyHostToDevice));
  NZCP_CUDA(cudaMemcpy(d_h.p, z.s[9].p, N * 64, cudaMemcpyHostToDevice));
  NttDomain dom;
  ntt_domain_create(&dom, (int)in.cir_power, 0);
  struct DomGuard { NttDomain* d; ~DomGuard() { ntt_domain_destroy(d); } } dg{&dom};
  const G1Affine r1 = timed(ms[3], [&] { return msm_g1(diff.d->p, static_cast<const Fr*>(d_r.p), N - 1); });
  Fr two = Fr::zero();
  two.v[0] = 2;
  const G1Affine r2 = timed(ms[3], [&] {
    h_scalar_kernel<<<div_up(N, 256), 256>>>(static_cast<Fr*>(d_r.p), N, host_fr_root((int)in.cir_power + 1),
                                             fp_neg(fp_to_mont(two)));
    NZCP_LAUNCH_CHECK();
    ntt_forward(dom, static_cast<Fr*>(d_r.p), static_cast<Fr*>(d_tmp.p), 0);
    return msm_g1(d_h.p, static_cast<const Fr*>(d_r.p), N);
  });
  cl.add(12, -1, r1, r2, delta2, delta2_init);
}

struct Out {
  const uint8_t* seed;
  nzcp_zkey_verify_claim* claims;
  size_t claims_cap;
  nzcp_zkey_contribution* records;
  size_t records_cap;
  nzcp_zkey_verify_report* report;
  float* section_ms;
};

void check_out(const Out& o, size_t n_recs) {
  if (!o.report || (n_recs && !o.records) || !o.claims) throw ApiError(NZCP_E_ARG, "null argument");
  if (o.claims_cap < 2 * n_recs + 3 || o.records_cap < n_recs)
    throw ApiError(NZCP_E_ARG, "claims or records buffer too small (see nzcp_zkey_verify_size)");
}

// The key under verification: parsed, its points left to verify_checks.
void parse_key(Inputs& in, const uint8_t* key, size_t key_len) {
  in.key = parse_zkey_in(key, key_len, false);
  for (const uint8_t* r : in.key.recs) in.recs.push_back(read_record(r));
}

void run(Inputs& in, const uint8_t* init_hash_or_null, const Out& o) {
  nzcp_zkey_verify_report& rep = *o.report;
  memset(&rep, 0, sizeof rep);
  rep.failed_record = -1;
  rep.n_contributions = (uint32_t)in.recs.size();
  fill_records(in, o.records);
  float ms[4] = {0, 0, 0, 0};
  Claims cl{o.claims};
  HDiff diff;
  circuit_hash(in.init, in.pt, false, rep.cs_hash, diff, &ms[0], &ms[1]);
  try {
    verify_checks(in, init_hash_or_null ? init_hash_or_null : rep.cs_hash, o.seed, cl, diff, ms);
  } catch (const Verdict& v) {
    rep.failed_step = v.step;
    rep.failed_record = v.record;
    snprintf(rep.message, sizeof rep.message, "%s", v.msg.c_str());
  }
  rep.n_claims = (uint32_t)cl.n;
  if (o.section_ms) memcpy(o.section_ms, ms, sizeof ms);
}

}  // namespace
}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_zkey_circuit_hash(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, int device,
                           uint8_t hash[64], float ms[2]) {
  return api_guard([&] {
    if (!init || !ptau || !hash) throw ApiError(NZCP_E_ARG, "null argument");
    const ZkeyIn zi = parse_zkey_in(init, init_len);
    check_init_sections(zi);
    const Ptau pt = parse_ptau(ptau, ptau_len);
    check_ptau_for(pt, zkey_domain_power(zi));
    use_device(device);
    HDiff diff;
    circuit_hash(zi, pt, false, hash, diff, ms, ms ? ms + 1 : nullptr);
  });
}

int nzcp_host_zkey_circuit_hash(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, uint8_t hash[64]) {
  return api_guard([&] {
    if (!init || !ptau || !hash) throw ApiError(NZCP_E_ARG, "null argument");
    const ZkeyIn zi = parse_zkey_in(init, init_len);
    check_init_sections(zi);
    const Ptau pt = parse_ptau(ptau, ptau_len);
    check_ptau_for(pt, zkey_domain_power(zi));
    if (zi.domain_size > kHostMaxPoints) throw ApiError(NZCP_E_ARG, "zkey: the host run is limited to 4096 H points");
    HDiff diff;
    circuit_hash(zi, pt, true, hash, diff, nullptr, nullptr);
  });
}

int nzcp_zkey_verify_size(const uint8_t* zkey, size_t len, size_t* n_claims, size_t* n_records) {
  return api_guard([&] {
    if (!zkey || !n_claims || !n_records) throw ApiError(NZCP_E_ARG, "null argument");
    Inputs in;
    parse_key(in, zkey, len);
    *n_records = in.recs.size();
    *n_claims = 2 * in.recs.size() + 3;
  });
}

int nzcp_zkey_verify_from_init(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, const uint8_t* zkey,
                               size_t zkey_len, const uint8_t* seed, int device, nzcp_zkey_verify_claim* claims,
                               size_t claims_cap, nzcp_zkey_contribution* records, size_t records_cap,
                               nzcp_zkey_verify_report* report, float section_ms[4]) {
  return api_guard([&] {
    if (!init || !ptau || !zkey) throw ApiError(NZCP_E_ARG, "null argument");
    const Out o{seed, claims, claims_cap, records, records_cap, report, section_ms};
    Inputs in;
    parse_key(in, zkey, zkey_len);
    check_out(o, in.recs.size());
    in.init = parse_zkey_in(init, init_len);
    check_init_sections(in.init);
    in.pt = parse_ptau(ptau, ptau_len);
    in.cir_power = zkey_domain_power(in.init);
    check_ptau_for(in.pt, in.cir_power);
    use_device(device);
    run(in, in.init.s[10].p, o);
  });
}

int nzcp_zkey_verify_from_r1cs(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, const uint8_t* zkey,
                               size_t zkey_len, const uint8_t* seed, int device, nzcp_zkey_verify_claim* claims,
                               size_t claims_cap, nzcp_zkey_contribution* records, size_t records_cap,
                               nzcp_zkey_verify_report* report, float section_ms[4]) {
  return api_guard([&] {
    if (!r1cs || !ptau || !zkey) throw ApiError(NZCP_E_ARG, "null argument");
    const Out o{seed, claims, claims_cap, records, records_cap, report, section_ms};
    Inputs in;
    parse_key(in, zkey, zkey_len);
    check_out(o, in.recs.size());
    const R1cs r = parse_r1cs(r1cs, r1cs_len);
    in.pt = parse_ptau(ptau, ptau_len);
    in.cir_power = circuit_power(r);
    check_ptau_for(in.pt, in.cir_power);
    const size_t size = zkey_new_size(r, in.cir_power);
    std::vector<uint8_t> init(size);
    zkey_new_impl(r1cs, r1cs_len, ptau, ptau_len, device, init.data(), size, nullptr);
    in.init = parse_zkey_in(init.data(), size);
    run(in, nullptr, o);
  });
}

}  // extern "C"
