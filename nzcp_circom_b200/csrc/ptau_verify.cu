// `powersoftau verify` on the GPU: the checks of a phase-1 powers-of-tau file, its contributions and, when prepared, its
// Lagrange sections.
//
// Replaces snarkjs 0.4.12 src/powersoftau_verify.js verify(tauFilename) with the parts of src/powersoftau_utils.js and
// src/keypair.js it uses (upstream, not vendored: package.json:12, yarn.lock:987-999).  Restated:
//   records   section 7, laid out as ptau_contribute.cu writes them; id = index + 1.  responseHash = BLAKE2b-512 resumed
//             from the record's 216-byte partialHash, then U(pubkey) (toPtauPubKeyRpr, montgomery = false).  initial =
//             {tauG1 = alphaG1 = betaG1 = G1, tauG2 = betaG2 = G2, nextChallenge = calculateFirstChallengeHash(ceremonyPower)}.
//   1  (deviation) every point of sections 2-6, 12-15 and of the records canonical and on its curve; the records' g2_spx,
//      tauG2, betaG2 and the two tauG2-section sums below in the order-r subgroup of G2 (a Miller loop on other points is
//      not a pairing; snarkjs checks none of this)
//   2  no records: "This file has no contribution! It cannot be used in production"
//   verifyContribution(cur, prev): a beacon record's nine public-key points must equal keyFromBeacon(prev.nextChallenge)
//      (step 3); g2_sp[j] = hashToG2(BLAKE2b([j] || prev.nextChallenge || U(g1_s) || U(g1_sx))); claims 4-6 sameRatio(g1_s,
//      g1_sx, g2_sp, g2_spx) for tau, alpha, beta; 7 (prev.tauG1, cur.tauG1, tau.g2_sp, tau.g2_spx); 8 (tau.g1_s,
//      tau.g1_sx, prev.tauG2, cur.tauG2); 9 (prev.alphaG1, cur.alphaG1, alpha.g2_sp, alpha.g2_spx); 10 the same for beta;
//      11 (beta.g1_s, beta.g1_sx, prev.betaG2, cur.betaG2).
//   verifyContribution(last record, the one before or initial); then sections 2-6 in order: nextChallenge' =
//      BLAKE2b(last.responseHash || U(every point of 2, 3, 4, 5, 6)); for 2-5, R1 = sum_(i<N-1) r_i P_i, R2 = sum_(i<N-1)
//      r_i P_(i+1); claims 12 (R1, R2, G2, last.tauG2) tauG1, 13 (G1, last.tauG1, R1, R2) tauG2, 14 / 15 (R1, R2, G2,
//      last.tauG2) alphaTauG1 / betaTauG1; after each claim the section's first points (step 16): tauG1[0] = G1, tauG1[1]
//      = last.tauG1, tauG2[0] = G2, tauG2[1] = last.tauG2, alphaTauG1[0] = last.alphaG1, betaTauG1[0] = last.betaG1,
//      betaG2 = last.betaG2.  Only when power = ceremonyPower: nextChallenge' = last.nextChallenge (step 17).
//   verifyContribution(record i, record i - 1 or initial) for i = n - 2 down to 0.
//   18 a prepared file (sections 12-15 all present; otherwise the caller warns): the Lagrange sections below.
// sameRatio(a, b, c, d) claims e(a, d) = e(b, c); the pairings stay with the caller, as for `zkey verify` (verify.cu).
//
// Lagrange check.  snarkjs checks, per level p of each section (2 -> 12 G1, 3 -> 13 G2, 4 -> 14, 5 -> 15; levels 0 ..
// power, and power + 1 for tauG1), G.eq(sum_j r_j tau_j, sum_i Fr.fft(r)_i L^(p)_i).  That identity holds for any r when
// L^(p) = ifft(tau_0 .. tau_(2^p - 1)): sum_i (sum_j r_j w^(ij)) (1/N) sum_k w^(-ik) tau_k = sum_j r_j tau_j.  On the top
// tauG1 level the last tau slot is the point at infinity and r_last = 0, so the same holds for what prepare wrote there.
// Here one check covers all levels of a section: r^(p) is drawn independently for every level, and MSM(tau section,
// sum_p r^(p)_j) is compared with MSM(the whole Lagrange section, the transforms back to back).  If any level is wrong the
// two sums differ except with probability 1/r: Fr.fft is a bijection, so each level's transformed scalars are uniform and
// independent, and the error of a wrong level is a nonzero vector of the order-r group (G1 has cofactor 1).  A section-13
// point off the G2 subgroup can escape with a higher probability, as in snarkjs, which checks no such point either.  The
// transforms are radix-2 DIF stages over every level of a section in one launch per stage (as ptau.cu stages its group
// FFT), then a bit-reversal; ntt.cu is not used: it stops at 2^27, and the top tauG1 level of a power-27 file has 2^28.
// Scalars are full-width F.fromRng draws of one ChaCha seeded with 32 OS-random bytes (or the test seed), in the order:
// the N - 1 of sections 2, 3, 4, 5, then the levels 0, 1, ... of 12, 13, 14, 15 (the top tauG1 level's last scalar is 0,
// not drawn).  snarkjs draws 32-bit scalars (deviation, as in `zkey verify`).
// Errors, all before any device work: read_ptau's and the section-size rejections of `contribute`, sections 12-15 of a
// size other than `zkey new` requires, ceremonyPower outside [power, 28], section 7 rejections, a partialHash with c >
// 128, t >= 2^64 or outlen != 64 (NZCP_E_FORMAT), a beacon record without its parameters, and a prepared file of power 28
// (NZCP_E_ARG).  A file that parses but fails a check is a false verdict, never an error.
//
// B200 design.  One section resides in HBM at a time (tauG1 at power 28: 34 GB), with its Lagrange section when the file
// is prepared.  The resident section is encoded for the nextChallenge' hash (mpc.cuh Hasher), is the base array of both
// R1 and R2 (one bucket sort of the N - 1 scalars, two table-free runs over the views at x and x + 1), and the tau side
// of the Lagrange check.  The first challenge hash, a host BLAKE2b pass as long as the nextChallenge' pass, runs on its own
// host thread from entry until record 0 is checked, so with two or more records it overlaps the section work; a check
// that fails before record 0 is reached cancels it.
#include <future>

#include "mpc.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ shared host/device code
struct PtauVerifyTwiddle {   // Exec op: tw[k] = w^k, Montgomery
  Fr* tw;
  Fr w;
  HD void operator()(uint64_t k) const {
    Fr r = Fr::one(), b = w;
    for (uint64_t e = k; e; e >>= 1) {
      if (e & 1) r = fp_mul(r, b);
      b = fp_sqr(b);
    }
    tw[k] = r;
  }
};

// Exec op: acc[j] = sum of scalar j of every level p <= top with 2^p > j; levels back to back (level p at 2^p - 1), plain.
struct LevelSum {
  const Fr* t;
  Fr* acc;
  int top;
  HD void operator()(uint64_t j) const {
    Fr s = Fr::zero();
    for (int p = j ? ilog2_u64(j) + 1 : 0; p <= top; p++) s = fp_add(s, t[((uint64_t)1 << p) - 1 + j]);
    acc[j] = s;
  }
};

// Exec op: butterfly u (< 2^top - 2^s) of radix-2 DIF stage s over the levels p = s+1 .. top (the index map of ptau.cu
// prep_butterfly): (a, b) -> (a + b, (a - b) w^k), w of order 2^(s+1) = tw[k << (t_log - 1 - s)], tw[k] = Fr.w[t_log]^k.
// Plain scalars, Montgomery twiddles.
struct LevelStage {
  Fr* x;
  const Fr* tw;
  int t_log, s;
  HD void operator()(uint64_t u) const {
    const uint64_t half = (uint64_t)1 << s, v = u + half;
    const int p = ilog2_u64(v) + 1;
    const uint64_t b = v - ((uint64_t)1 << (p - 1)), k = b & (half - 1);
    const uint64_t i0 = ((uint64_t)1 << p) - 1 + ((b >> s) << (s + 1)) + k, i1 = i0 + half;
    const Fr a = x[i0], c = x[i1];
    x[i0] = fp_add(a, c);
    x[i1] = fp_mul(fp_sub(a, c), tw[k << (t_log - 1 - s)]);
  }
};

// Exec op: slot i of the levels back to back swaps with its bit-reversed partner within its level (the DIF output order
// becomes natural order).
struct LevelBitrev {
  Fr* x;
  HD void operator()(uint64_t i) const {
    const int p = ilog2_u64(i + 1);
    const uint64_t base = ((uint64_t)1 << p) - 1, j = i - base, r = bitrev_bits(j, p);
    if (r > j) {
      const Fr t = x[base + j];
      x[base + j] = x[base + r];
      x[base + r] = t;
    }
  }
};

namespace {

constexpr uint32_t kHostMaxPower = 4;
constexpr size_t kPartialOff = 1216, kNextOff = 1432;

uint64_t level_points(uint32_t top) { return ((uint64_t)2 << top) - 1; }   // levels 0 .. top back to back

// Lagrange section id (12..15): its source section and top level.
int lag_src(int id) { return id - 10; }
uint32_t lag_top(uint32_t power, int id) { return id == 12 ? power + 1 : power; }

struct VerifyIn : Ptau {
  std::vector<Rec> recs;
  bool prepared = false;
};

// Everything `powersoftau verify` needs from its input, validated before any device work.
VerifyIn parse_verify_in(const uint8_t* b, size_t len) {
  VerifyIn v{read_ptau(b, len)};
  need_sections(v.s, 2, 7);
  v.prepared = v.s[12].p && v.s[13].p && v.s[14].p && v.s[15].p;
  if (v.prepared && v.power == kPtauMaxPower) throw ApiError(NZCP_E_ARG, kPtauPower28Phase2);
  for (int id = 2; id <= 6; id++)
    if (v.s[id].len != sect_bytes(v.power, id))
      throw ApiError(NZCP_E_FORMAT, "ptau: section " + std::to_string(id) + " size does not match the header power");
  if (v.ceremony_power < v.power || v.ceremony_power > kPtauMaxPower)
    throw ApiError(NZCP_E_FORMAT, "ptau: ceremonyPower out of range [power, 28]");
  for (int id = 12; id <= 15; id++)
    if (v.s[id].p && v.s[id].len != level_points(lag_top(v.power, id)) * (id == 13 ? 128 : 64))
      throw ApiError(NZCP_E_FORMAT, "ptau: section size does not match the header power");
  std::vector<const uint8_t*> recs;
  std::vector<size_t> rec_len;
  parse_records(v.s[7].p, v.s[7].len, 0, kPtauRecFixed, "ptau: section 7", recs, rec_len);
  for (size_t i = 0; i < recs.size(); i++) {
    const uint8_t* ph = recs[i] + kPartialOff;
    if (rd32u(ph + 208) > 128 || rd64u(ph + 200) != 0 || rd32u(ph + 212) != 64)
      throw ApiError(NZCP_E_FORMAT, "ptau: section 7 record " + std::to_string(i) + " has a malformed partialHash");
    v.recs.push_back(read_record(recs[i], kPtauRecFixed, "ptau"));
  }
  return v;
}

// The public key of a record (Montgomery affine, toPtauPubKeyRpr order); prv and g2_sp are not stored.
void record_key(const uint8_t* r, KeyPart k[3]) {
  for (int j = 0; j < 3; j++) {
    k[j].g1_s = load_pt<Fq>(r + 128 * j);
    k[j].g1_sx = load_pt<Fq>(r + 128 * j + 64);
    k[j].g2_spx = load_pt<Fq2>(r + 384 + 128 * j);
  }
}

void response_hash(const uint8_t* r, uint8_t out[64]) {
  KeyPart k[3];
  record_key(r, k);
  uint8_t pk[kPubKeyLen];
  pub_key(k, false, pk);
  Blake2b512 h = Blake2b512::from_partial(r + kPartialOff);
  h.update(pk, kPubKeyLen);
  h.final(out);
}

// What a contribution follows: a record's points and nextChallenge, or the initial accumulator.
struct Prev {
  G1Affine tau1, alpha1, beta1;
  G2Affine tau2, beta2;
  const uint8_t* next;
};

Prev rec_points(const uint8_t* r) {
  return {load_pt<Fq>(r + 768), load_pt<Fq>(r + 960), load_pt<Fq>(r + 1024), load_pt<Fq2>(r + 832), load_pt<Fq2>(r + 1088),
          r + kNextOff};
}

Prev initial(const uint8_t* first_challenge_hash) {
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  return {g1, g1, g1, g2, g2, first_challenge_hash};
}

// Step 1 for the points of sections 2-6, 12-15 (prepared) and of the records.
void check_verify_points(const VerifyIn& v) {
  const Fq b1 = curve_b(g1_generator());
  const Fq2 b2 = curve_b(g2_generator());
  try {
    for (int id = 2; id <= 6; id++) {
      if (sect_g2(id)) check_points<Fq2>("ptau", v.s[id].p, sect_points(v.power, id), id, b2);
      else check_points<Fq>("ptau", v.s[id].p, sect_points(v.power, id), id, b1);
    }
    for (int id = 12; v.prepared && id <= 15; id++) {
      const uint64_t n = level_points(lag_top(v.power, id));
      if (id == 13) check_points<Fq2>("ptau", v.s[id].p, n, id, b2);
      else check_points<Fq>("ptau", v.s[id].p, n, id, b1);
    }
  } catch (const ApiError& e) {
    throw Verdict{1, -1, e.what()};
  }
  static const char* kG1[9] = {"tau.g1_s", "tau.g1_sx", "alpha.g1_s", "alpha.g1_sx", "beta.g1_s", "beta.g1_sx", "tauG1",
                               "alphaG1", "betaG1"};
  static const size_t kG1Off[9] = {0, 64, 128, 192, 256, 320, 768, 960, 1024};
  static const char* kG2[5] = {"tau.g2_spx", "alpha.g2_spx", "beta.g2_spx", "tauG2", "betaG2"};
  static const size_t kG2Off[5] = {384, 512, 640, 832, 1088};
  bool inf;
  for (size_t i = 0; i < v.recs.size(); i++) {
    const std::string w = "ptau: section 7 record " + std::to_string(i) + " ";
    for (int q = 0; q < 9; q++)
      if (!point_ok(load_pt<Fq>(v.recs[i].p + kG1Off[q]), b1, &inf))
        throw Verdict{1, (int)i, w + kG1[q] + " is not a canonical point of G1"};
    for (int q = 0; q < 5; q++) {
      const G2Affine a = load_pt<Fq2>(v.recs[i].p + kG2Off[q]);
      if (!point_ok(a, b2, &inf)) throw Verdict{1, (int)i, w + kG2[q] + " is not a canonical point of the twist"};
      if (!in_g2_subgroup(a)) throw Verdict{1, (int)i, w + kG2[q] + " is not in the order-r subgroup of G2"};
    }
  }
}

// verifyContribution(cur = record i, prev): the beacon check (step 3), then claims 4-11.
void verify_contribution(const Rec& c, int i, const Prev& prev, Claims& cl) {
  const std::string id = std::to_string(i + 1);
  if (c.type == 1) {
    static const char* kParts[9] = {"tauG1_s", "tauG1_sx", "alphaG1_s", "alphaG1_sx", "betaG1_s", "betaG1_sx",
                                    "tauG2_spx", "alphaG2_spx", "betaG2_spx"};
    uint8_t s[32];
    beacon_seed(c.beacon, c.beacon_len, c.exp, s);
    ChaCha rng(s);
    KeyPart bk[3];
    create_key(rng, prev.next, bk);
    uint8_t want[kPubKeyLen];
    pub_key(bk, true, want);
    for (int q = 0; q < 9; q++) {
      const size_t off = q < 6 ? 64 * q : 384 + 128 * (q - 6), len = q < 6 ? 64 : 128;
      if (memcmp(want + off, c.p + off, len) != 0)
        throw Verdict{3, i, std::string("BEACON key (") + kParts[q] + ") is not generated correctly in challenge #" + id + "  " +
                                (c.name ? std::string(reinterpret_cast<const char*>(c.name), c.name_len) : std::string())};
    }
  }
  KeyPart k[3];
  record_key(c.p, k);
  for (int j = 0; j < 3; j++) {
    Blake2b512 h;
    const uint8_t pers = (uint8_t)j;
    h.update(&pers, 1);
    h.update(prev.next, 64);
    hash_g1(h, c.p + 128 * j);
    hash_g1(h, c.p + 128 * j + 64);
    uint8_t d[64];
    h.final(d);
    k[j].g2_sp = hash_to_g2(d);
  }
  const Prev cur = rec_points(c.p);
  for (int j = 0; j < 3; j++) cl.add(4 + j, i, k[j].g1_s, k[j].g1_sx, k[j].g2_sp, k[j].g2_spx);
  cl.add(7, i, prev.tau1, cur.tau1, k[0].g2_sp, k[0].g2_spx);
  cl.add(8, i, k[0].g1_s, k[0].g1_sx, prev.tau2, cur.tau2);
  cl.add(9, i, prev.alpha1, cur.alpha1, k[1].g2_sp, k[1].g2_spx);
  cl.add(10, i, prev.beta1, cur.beta1, k[2].g2_sp, k[2].g2_spx);
  cl.add(11, i, k[2].g1_s, k[2].g1_sx, prev.beta2, cur.beta2);
}

// The Lagrange check of one section (see the header): x = the resident source section (n_tau points), lx <- Lagrange
// section `lid`, d_t / d_acc scalar buffers of level_points(top) / n_tau entries.  Draws the levels' scalars from rng.
template <class F>
bool lagrange_check(const Exec& ex, ChaCha& rng, const VerifyIn& v, int lid, const Affine<F>* x, Affine<F>* lx, Fr* d_t,
                    Fr* d_acc, const Fr* tw, float* ms) {
  const uint32_t top = lag_top(v.power, lid);
  const uint64_t n_tau = sect_points(v.power, lag_src(lid)), nl = level_points(top);
  std::vector<Fr> r(nl);
  for (uint32_t p = 0; p <= top; p++)
    for (uint64_t j = 0; j < ((uint64_t)1 << p); j++) r[((uint64_t)1 << p) - 1 + j] = j < n_tau ? fp_from_rng<FrParams>(rng) : Fr::zero();
  ex.upload(lx, v.s[lid].p, nl * sizeof(Affine<F>));
  ex.upload(d_t, r.data(), nl * sizeof(Fr));
  Timer t = ex.timer();
  ex.run<256>(n_tau, LevelSum{d_t, d_acc, (int)top});
  for (int s = (int)top - 1; s >= 0; s--)
    ex.run<256>(((uint64_t)1 << top) - ((uint64_t)1 << s), LevelStage{d_t, tw, (int)v.power + 1, s});
  ex.run<256>(nl, LevelBitrev{d_t});
  const Affine<F> lhs = msm_sum(ex, x, d_acc, n_tau), rhs = msm_sum(ex, lx, d_t, nl);
  *ms += t.stop();
  return memcmp(&lhs, &rhs, sizeof lhs) == 0;
}

// Everything after parsing; throws Verdict at the first failed check.  ms: see nzcp_ptau_verify.
void verify_checks(const VerifyIn& v, const uint8_t* seed, bool host, Claims& cl, uint8_t next_out[64], float ms[5]) {
  // calculateFirstChallengeHash(ceremonyPower), on its own thread.  A verdict or error before record 0 is checked cancels
  // it (the guard runs before the future's destructor, which joins the thread), so a failing file does not wait for it.
  std::atomic<bool> cancel{false};
  std::future<std::vector<uint8_t>> first;
  struct CancelOnExit {
    std::atomic<bool>& c;
    ~CancelOnExit() { c = true; }
  } guard{cancel};
  if (!v.recs.empty())
    first = std::async(std::launch::async, [p = v.ceremony_power, &cancel] {
      std::vector<uint8_t> h(64);
      first_challenge(p, h.data(), nullptr, &cancel);
      return h;
    });
  std::vector<uint8_t> first_hash;
  auto prev_of = [&](size_t i) {   // what record i follows
    if (i > 0) return rec_points(v.recs[i - 1].p);
    if (first_hash.empty()) first_hash = first.get();
    return initial(first_hash.data());
  };

  const auto t0 = std::chrono::steady_clock::now();
  check_verify_points(v);
  ms[0] = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();

  // 2. the last contribution
  if (v.recs.empty()) throw Verdict{2, -1, "This file has no contribution! It cannot be used in production"};
  const size_t n = v.recs.size();
  const Rec& last = v.recs.back();
  verify_contribution(last, (int)n - 1, prev_of(n - 1), cl);
  const Prev cur = rec_points(last.p);

  // 3. sections 2-6: the R1 / R2 scalars of sections 2-5 first, then (prepared) the Lagrange levels as each comes
  uint8_t sd[32];
  verify_seed("ptau verify", seed, sd);
  ChaCha rng(sd);
  const uint32_t P = v.power;
  std::vector<Fr> rs[6];
  for (int id = 2; id <= 5; id++) {
    rs[id].resize(sect_points(P, id) - 1);
    for (Fr& s : rs[id]) s = fp_from_rng<FrParams>(rng);
  }
  Exec ex(host);
  void* buf = ex.alloc<unsigned char>(std::max(sect_bytes(P, 2), sect_bytes(P, 3)));
  Fr* d_sc = ex.alloc<Fr>(sect_points(P, 2));
  void* lbuf = nullptr;
  Fr *d_t = nullptr, *tw = nullptr;
  if (v.prepared) {
    lbuf = ex.alloc<unsigned char>(level_points(P + 1) * 64);   // section 12, the largest
    d_t = ex.alloc<Fr>(level_points(P + 1));
    tw = ex.alloc<Fr>((uint64_t)1 << P);
    ex.run<256>((uint64_t)1 << P, PtauVerifyTwiddle{tw, host_fr_root((int)P + 1)});
  }
  Hasher nx(ex, Enc::U);
  uint8_t resp[64];
  response_hash(last.p, resp);
  nx.update(resp, 64);
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  bool lag_ok = true;
  auto need_eq = [](const uint8_t* got, const void* want, size_t len, const char* msg) {
    if (memcmp(got, want, len) != 0) throw Verdict{16, -1, msg};
  };
  for (int id = 2; id <= 6; id++) {
    const uint64_t np = sect_points(P, id);
    const uint8_t* s = v.s[id].p;
    ex.upload(buf, s, v.s[id].len);
    if (sect_g2(id)) nx.points(static_cast<const G2Affine*>(buf), np);
    else nx.points(static_cast<const G1Affine*>(buf), np);
    if (id == 6) {
      need_eq(s, &cur.beta2, 128, "betaG2 element in betaG2 section does not match the one in the contribution section");
      break;
    }
    ex.upload(d_sc, rs[id].data(), (np - 1) * sizeof(Fr));
    Timer t = ex.timer();
    if (id == 3) {
      const G2Affine* x = static_cast<const G2Affine*>(buf);
      const G2Affine* b[2] = {x, x + 1};
      G2Affine r[2];
      msm_sums(ex, b, 2, d_sc, np - 1, r);
      ms[3] += t.stop();
      if (!in_g2_subgroup(r[0]) || !in_g2_subgroup(r[1]))
        throw Verdict{1, -1, "ptau: a random combination of the tauG2 section is not in the order-r subgroup of G2"};
      cl.add(13, -1, g1, cur.tau1, r[0], r[1]);
      need_eq(s, &g2, 128, "First element of tau*G2 section must be the generator");
      need_eq(s + 128, &cur.tau2, 128, "Second element of tau*G2 section does not match the one in the contribution section");
      if (v.prepared) lag_ok &= lagrange_check(ex, rng, v, 13, x, static_cast<G2Affine*>(lbuf), d_t, d_sc, tw, &ms[4]);
      continue;
    }
    const G1Affine* x = static_cast<const G1Affine*>(buf);
    const G1Affine* b[2] = {x, x + 1};
    G1Affine r[2];
    msm_sums(ex, b, 2, d_sc, np - 1, r);
    ms[3] += t.stop();
    cl.add(10 + id, -1, r[0], r[1], g2, cur.tau2);
    if (id == 2) {
      need_eq(s, &g1, 64, "First element of tau*G1 section must be the generator");
      need_eq(s + 64, &cur.tau1, 64, "Second element of tau*G1 section does not match the one in the contribution section");
    } else if (id == 4) {
      need_eq(s, &cur.alpha1, 64,
              "First element of alpha*tau*G1 section (alpha*G1) does not match the one in the contribution section");
    } else {
      need_eq(s, &cur.beta1, 64,
              "First element of beta*tau*G1 section (beta*G1) does not match the one in the contribution section");
    }
    if (v.prepared) lag_ok &= lagrange_check(ex, rng, v, id + 10, x, static_cast<G1Affine*>(lbuf), d_t, d_sc, tw, &ms[4]);
  }
  nx.h.final(next_out);
  ms[1] = nx.kernel_ms;
  ms[2] = nx.blake_ms;
  if (P == v.ceremony_power && memcmp(next_out, last.p + kNextOff, 64) != 0)
    throw Verdict{17, -1, "Hash of the values does not match the next challenge of the last contributor in the contributions section"};

  // 4. the earlier contributions, 5. the Lagrange sections
  for (size_t i = n - 1; i-- > 0;) verify_contribution(v.recs[i], (int)i, prev_of(i), cl);
  if (!lag_ok) throw Verdict{18, -1, "Phase2 caclutation does not match with powers of tau"};   // snarkjs's spelling
}

struct Out {
  const uint8_t* seed;
  nzcp_zkey_verify_claim* claims;
  size_t claims_cap;
  nzcp_ptau_contribution* records;
  size_t records_cap;
  nzcp_ptau_verify_report* report;
  float* ms;
};

void check_out(const Out& o, size_t n_recs) {
  if (!o.report || (n_recs && !o.records) || !o.claims) throw ApiError(NZCP_E_ARG, "null argument");
  if (o.claims_cap < 8 * n_recs + 4 || o.records_cap < n_recs)
    throw ApiError(NZCP_E_ARG, "claims or records buffer too small (see nzcp_ptau_verify_size)");
}

void fill_records(const VerifyIn& v, nzcp_ptau_contribution* out) {
  for (size_t i = 0; i < v.recs.size(); i++) {
    const Rec& c = v.recs[i];
    nzcp_ptau_contribution& o = out[i];
    memset(&o, 0, sizeof o);
    response_hash(c.p, o.response_hash);
    memcpy(o.next_challenge, c.p + kNextOff, 64);
    o.type = c.type;
    o.num_iterations_exp = c.exp;
    o.name_len = (uint32_t)c.name_len;
    if (c.name) memcpy(o.name, c.name, c.name_len);
    o.beacon_hash_len = (uint32_t)c.beacon_len;
    if (c.beacon) memcpy(o.beacon_hash, c.beacon, c.beacon_len);
  }
}

// device < 0: the host hook.
void verify_impl(const uint8_t* b, size_t len, int device, const Out& o) {
  const VerifyIn v = parse_verify_in(b, len);
  check_out(o, v.recs.size());
  const bool host = device < 0;
  if (host && v.power > kHostMaxPower) throw ApiError(NZCP_E_ARG, "ptau: the host run is limited to power 4");
  if (!host) use_device(device);
  nzcp_ptau_verify_report& rep = *o.report;
  memset(&rep, 0, sizeof rep);
  rep.failed_record = -1;
  rep.n_contributions = (uint32_t)v.recs.size();
  rep.prepared = v.prepared;
  fill_records(v, o.records);
  float ms[5] = {0, 0, 0, 0, 0};
  Claims cl{o.claims};
  try {
    verify_checks(v, o.seed, host, cl, rep.next_challenge, ms);
  } catch (const Verdict& e) {
    rep.failed_step = e.step;
    rep.failed_record = e.record;
    snprintf(rep.message, sizeof rep.message, "%s", e.msg.c_str());
  }
  rep.n_claims = (uint32_t)cl.n;
  if (o.ms) memcpy(o.ms, ms, sizeof ms);
}

}  // namespace
}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_ptau_verify_size(const uint8_t* ptau, size_t len, size_t* n_claims, size_t* n_records) {
  return api_guard([&] {
    if (!ptau || !n_claims || !n_records) throw ApiError(NZCP_E_ARG, "null argument");
    const VerifyIn v = parse_verify_in(ptau, len);
    *n_records = v.recs.size();
    *n_claims = 8 * v.recs.size() + 4;
  });
}

int nzcp_ptau_verify(const uint8_t* ptau, size_t len, const uint8_t* seed, int device, nzcp_zkey_verify_claim* claims,
                     size_t claims_cap, nzcp_ptau_contribution* records, size_t records_cap, nzcp_ptau_verify_report* report,
                     float ms[5]) {
  return api_guard([&] {
    if (!ptau) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    verify_impl(ptau, len, device, Out{seed, claims, claims_cap, records, records_cap, report, ms});
  });
}

int nzcp_host_ptau_verify(const uint8_t* ptau, size_t len, const uint8_t* seed, nzcp_zkey_verify_claim* claims,
                          size_t claims_cap, nzcp_ptau_contribution* records, size_t records_cap,
                          nzcp_ptau_verify_report* report) {
  return api_guard([&] {
    if (!ptau) throw ApiError(NZCP_E_ARG, "null argument");
    verify_impl(ptau, len, -1, Out{seed, claims, claims_cap, records, records_cap, report, nullptr});
  });
}

}  // extern "C"
