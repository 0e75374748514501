// `powersoftau new`, `powersoftau contribute` and `powersoftau beacon` on the GPU: phase-1 contributions to tau, alpha and
// beta of a powers-of-tau file.
//
// Replaces snarkjs 0.4.12 src/powersoftau_new.js newAccumulator(curve, power, fileName), src/powersoftau_contribute.js
// contribute(oldPtauFilename, newPTauFilename, name, entropy) and src/powersoftau_beacon.js beacon(oldPtauFilename,
// newPTauFilename, name, beaconHashStr, numIterationsExp), with the parts of src/keypair.js and src/powersoftau_utils.js
// they use (upstream, not vendored: package.json:12, yarn.lock:987-999).  Restated:
//   new        section 1 writePTauHeader: n8 = 32, q, power, ceremonyPower = power; sections 2-6 the G1 / G2 generator
//              repeated 2^(p+1) - 1, 2^p, 2^p, 2^p, 1 times (Montgomery affine); section 7 a u32 count of 0.  Powers 1..28.
//   first challenge (calculateFirstChallengeHash)  BLAKE2b-512(BLAKE2b-512("") || U(G1) x (2^(p+1) - 1) || U(G2) x 2^p ||
//              U(G1) x 2^p || U(G1) x 2^p || U(G2)); snarkjs `new` logs it as "First Contribution Hash".
//   challenge  the last record's nextChallenge; with no records the first challenge hash
//   rng        as `zkey contribute` / `zkey beacon` (contribute.cu): ChaCha seeded by BLAKE2b(64 OS bytes || entropy), or
//              by SHA-256 applied 2^numIterationsExp times to the beacon hash (keyFromBeacon)
//   key        createPTauKey: tau, alpha, beta = Fr.fromRng in that order (Montgomery buffers); then for each, with
//              personalization 0, 1, 2: g1_s = G1.fromRng, g1_sx = k g1_s, g2_sp = hashToG2(BLAKE2b-512([pers] ||
//              challenge || U(g1_s) || U(g1_sx))) (cofactor included), g2_spx = k g2_sp
//   sections   processSection: point i of 2 tauG1 (2^(p+1) - 1 points), 3 tauG2, 4 alphaTauG1, 5 betaTauG1 (2^p each),
//              6 betaG2 (1 point) becomes (first * tau^i) P_i with first = 1, 1, alpha, beta, beta; infinity stays (0,0)
//   response   BLAKE2b-512(challenge || C(every new point of sections 2, 3, 4, 5, 6) || U(pubkey)), pubkey =
//              toPtauPubKeyRpr(montgomery = false): tau.g1_s tau.g1_sx alpha.g1_s alpha.g1_sx beta.g1_s beta.g1_sx
//              tau.g2_spx alpha.g2_spx beta.g2_spx (768 bytes).  partialHash = the hasher's state before U(pubkey).
//   next       nextChallenge = BLAKE2b-512(response || U(every new point of sections 2, 3, 4, 5, 6))
//   record     writeContribution: the pubkey (Montgomery affine, same order), tauG1 = new tauG1[1], tauG2 = new tauG2[1],
//              alphaG1 = new alphaTauG1[0], betaG1 = new betaTauG1[0], betaG2 = new betaG2[0], partialHash (216 bytes),
//              nextChallenge, u32 type (0 contribute, 1 beacon), u32 paramLength, parameters (tag 1 name, tag 2
//              numIterationsExp, tag 3 beaconHash, as in phase 2).  Section 7 = u32 count + 1, the earlier records, this one.
//   output     sections 1-7 in id order, section 1 rewritten by writePTauHeader; sections 12-15 of a prepared input are
//              dropped.  Returns the response hash.
// U = the uncompressed encoding of mpc.cuh (big-endian plain x, y; G2 as c1 c0; infinity 0x40 then zeros).  C =
// wasmcurves LEMtoC: big-endian plain x (G2 x.c1 || x.c0), 0x80 ORed into byte 0 when y is negative (wasmcurves sign:
// plain value > (q-1)/2; for Fq2 c1 decides, c0 when c1 = 0), infinity 0x40 then zeros.  partialHash is blake2b-wasm's
// context, RFC 7693's blake2b_ctx: b[128] (stale bytes kept), h[8], t[2] as u64 LE, c, outlen as u32 LE (Blake2b512::partial).
// Earlier records are copied byte for byte (snarkjs re-serializes them from their parsed form: the same bytes for every
// record snarkjs writes).  Deviations: a name longer than 64 bytes is rejected (snarkjs cuts it at 64 characters), and
// input points must be canonical and on their curve (snarkjs does not check).  A G2 point outside the order-r subgroup,
// which no ceremony file holds, is scaled by the folded window of scalar_mul_accumulate and then differs from snarkjs's.
//
// B200 design.  One section at a time resides in HBM (tauG1 at power 28: 2^29 - 1 points, 34 GB).  ptau_key_kernel runs
// one thread per point: s = first * tau^i by square-and-multiply over the <= 29 bits of i (~45 Fr products against ~3 300
// Fq products for the G1 multiplication, so no power table), then the signed 4-bit window of ec.cuh scalar_mul_accumulate
// and to_affine_fast.  Unlike zkey_scale_kernel every lane has its own scalar.  The response pass encodes the points still
// resident after the key kernel (c_encode_kernel); the nextChallenge pass re-uploads each finished section from the output
// (u_encode_kernel); both run through mpc.cuh's chunked Hasher, whose host BLAKE2b of chunk j overlaps the encoding and
// copy of chunk j + 1.  The host BLAKE2b is a single sequential stream and likely takes longer than the kernels.
#include "mpc.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ shared host/device code
// (first * inc^i) * P; first, inc Montgomery.
template <class F>
HD Affine<F> ptau_key_point(const Affine<F>& p, const Fr& first, const Fr& inc, uint64_t i) {
  Fr s = first, b = inc;
  for (uint64_t e = i; e; e >>= 1) {
    if (e & 1) s = fp_mul(s, b);
    b = fp_sqr(b);
  }
  XYZZ<F> acc = XYZZ<F>::inf();
  scalar_mul_accumulate(acc, p, fp_from_mont(s));
  return to_affine_fast(acc);
}

template <class F>
__global__ void __launch_bounds__(128) ptau_key_kernel(Affine<F>* __restrict__ x, Fr first, Fr inc, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = ptau_key_point(x[i], first, inc, i);
}

namespace {

constexpr uint32_t kHostMaxPower = 4;
constexpr size_t kPubKeyLen = 6 * 64 + 3 * 128;                               // 768
constexpr size_t kPartialLen = 216;
// pubkey tauG1 tauG2 alphaG1 betaG1 betaG2 partialHash nextChallenge type paramLength
constexpr size_t kPtauRecFixed = kPubKeyLen + 3 * 64 + 2 * 128 + kPartialLen + 64 + 4 + 4;   // 1504

size_t new_size(uint32_t power) {
  size_t total = 12 + 7 * 12 + kPtauHeaderLen + 4;
  for (int id = 2; id <= 6; id++) total += sect_bytes(power, id);
  return total;
}

void check_power(uint32_t power) {
  if (power < 1 || power > kPtauMaxPower) throw ApiError(NZCP_E_ARG, "ptau: power out of range [1, 28]");
}

struct ContribIn : Ptau {
  std::vector<const uint8_t*> recs;   // section-7 records
  std::vector<size_t> rec_len;
};

// Everything contribute / beacon need from their input, validated before any device work.
ContribIn parse_contrib_in(const uint8_t* b, size_t len) {
  ContribIn p{read_ptau(b, len)};
  check_ptau_sections(p);
  if (p.ceremony_power != p.power)
    throw ApiError(NZCP_E_ARG, "This file has been reduced. You cannot contribute into a reduced file.");
  parse_records(p.s[7].p, p.s[7].len, 0, kPtauRecFixed, "ptau: section 7", p.recs, p.rec_len);
  return p;
}

size_t contribute_size(const ContribIn& p, size_t name_len, size_t beacon_len) {
  size_t total = 12 + 7 * 12 + kPtauHeaderLen;
  for (int id = 2; id <= 7; id++) total += p.s[id].len;
  return total + kPtauRecFixed + params_len(name_len, beacon_len);
}

// calculateFirstChallengeHash; blake_ms += the host time.
void first_challenge(uint32_t power, uint8_t out[64], float* blake_ms) {
  const auto t0 = std::chrono::steady_clock::now();
  Blake2b512 h;
  uint8_t empty[64];
  Blake2b512().final(empty);
  h.update(empty, 64);
  const G1Affine g1 = g1_generator();
  const G2Affine g2 = g2_generator();
  constexpr int kRep = 1024;
  std::vector<uint32_t> r1(kRep * 16), r2(kRep * 32);
  for (int i = 0; i < kRep; i++) {
    u_encode(g1, r1.data() + 16 * i);
    u_encode(g2, r2.data() + 32 * i);
  }
  auto block = [&](const std::vector<uint32_t>& r, size_t psz, uint64_t count) {
    for (uint64_t i = 0; i < count; i += kRep) h.update(r.data(), std::min<uint64_t>(kRep, count - i) * psz);
  };
  const uint64_t n = (uint64_t)1 << power;
  block(r1, 64, 2 * n - 1);
  block(r2, 128, n);
  block(r1, 64, n);
  block(r1, 64, n);
  block(r2, 128, 1);
  h.final(out);
  if (blake_ms) *blake_ms += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// One of tau, alpha, beta (keypair.js calculatePubKey).
struct KeyPart {
  Fr prv;   // Montgomery
  G1Affine g1_s, g1_sx;
  G2Affine g2_sp, g2_spx;
};

void create_key(ChaCha& rng, const uint8_t challenge[64], KeyPart k[3]) {
  for (int j = 0; j < 3; j++) {
    k[j].prv = fp_from_rng<FrParams>(rng);
    if (k[j].prv.is_zero()) throw ApiError(NZCP_E_INTERNAL, "ptau contribute: the rng drew a zero key");
  }
  const Fq b1 = curve_b(g1_generator());
  for (int j = 0; j < 3; j++) {
    const Fr kp = fp_from_mont(k[j].prv);
    k[j].g1_s = point_from_rng(rng, b1, nullptr);
    k[j].g1_sx = mul_plain(k[j].g1_s, kp.v);
    Blake2b512 h;
    const uint8_t pers = (uint8_t)j;
    h.update(&pers, 1);
    h.update(challenge, 64);
    hash_g1(h, reinterpret_cast<const uint8_t*>(&k[j].g1_s));
    hash_g1(h, reinterpret_cast<const uint8_t*>(&k[j].g1_sx));
    uint8_t d[64];
    h.final(d);
    k[j].g2_sp = hash_to_g2(d);
    k[j].g2_spx = mul_plain(k[j].g2_sp, kp.v);
  }
}

// toPtauPubKeyRpr order, Montgomery affine (montgomery = true) or uncompressed (false).
void pub_key(const KeyPart k[3], bool montgomery, uint8_t out[kPubKeyLen]) {
  for (int j = 0; j < 3; j++) {
    if (montgomery) {
      memcpy(out + 128 * j, &k[j].g1_s, 64);
      memcpy(out + 128 * j + 64, &k[j].g1_sx, 64);
      memcpy(out + 384 + 128 * j, &k[j].g2_spx, 128);
    } else {
      u_encode(k[j].g1_s, reinterpret_cast<uint32_t*>(out + 128 * j));
      u_encode(k[j].g1_sx, reinterpret_cast<uint32_t*>(out + 128 * j + 64));
      u_encode(k[j].g2_spx, reinterpret_cast<uint32_t*>(out + 384 + 128 * j));
    }
  }
}

template <class F>
void key_section_host(uint8_t* x, uint64_t n, const Fr& first, const Fr& inc) {
  for (uint64_t i = 0; i < n; i++) {
    Affine<F> a;
    memcpy(&a, x + i * sizeof a, sizeof a);
    a = ptau_key_point(a, first, inc, i);
    memcpy(x + i * sizeof a, &a, sizeof a);
  }
}

// Upload, key kernel in place, response-hash the resident points, download; returns the key kernel's device ms.
template <class F>
float key_section_device(const uint8_t* src, uint64_t n, const Fr& first, const Fr& inc, Affine<F>* d_x, Hasher& resp,
                         uint8_t* dst) {
  Events ev;
  NZCP_CUDA(cudaMemcpy(d_x, src, n * sizeof(Affine<F>), cudaMemcpyHostToDevice));
  NZCP_CUDA(cudaEventRecord(ev.a, 0));
  ptau_key_kernel<F><<<div_up(n, 128), 128>>>(d_x, first, inc, n);
  NZCP_LAUNCH_CHECK();
  NZCP_CUDA(cudaEventRecord(ev.b, 0));
  resp.points_device(d_x, n);
  NZCP_CUDA(cudaMemcpy(dst, d_x, n * sizeof(Affine<F>), cudaMemcpyDeviceToHost));
  float ms = 0;
  NZCP_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
  return ms;
}

// device < 0: the host hook.  ms: [0..4] key kernels of sections 2..6, [5] encode kernels, [6] host BLAKE2b.
void contribute_impl(const uint8_t* b, size_t len, ContribArgs a, int device, uint8_t* out, size_t cap, size_t* written,
                     uint8_t* hash_out, float* ms_out) {
  check_contrib_args("ptau", a);
  const bool beacon = a.beacon != nullptr;
  const ContribIn p = parse_contrib_in(b, len);
  const size_t total = contribute_size(p, a.name_len, beacon ? a.beacon_len : 0);
  if (cap < total) throw ApiError(NZCP_E_ARG, "output buffer too small");
  const bool host = device < 0;
  if (host && p.power > kHostMaxPower) throw ApiError(NZCP_E_ARG, "ptau: the host run is limited to power 4");
  if (!host) use_device(device);
  float ms[7] = {0, 0, 0, 0, 0, 0, 0};

  // ---- the challenge, the rng and the key (host: O(1) work)
  uint8_t challenge[64];
  if (p.recs.empty()) first_challenge(p.power, challenge, &ms[6]);
  else memcpy(challenge, p.recs.back() + kPtauRecFixed - 8 - 64, 64);
  uint8_t seed[64];
  contrib_seed(a, seed);
  ChaCha rng(seed);
  KeyPart key[3];
  create_key(rng, challenge, key);
  const Fr one = Fr::one(), &tau = key[0].prv, &alpha = key[1].prv, &beta = key[2].prv;
  const Fr* first[7] = {nullptr, nullptr, &one, &one, &alpha, &beta, &beta};

  // ---- sections 2-6 and the response hash
  Writer w(out, cap);
  write_ptau_header(w, p.power, 7);
  Hasher resp(host, Enc::C);
  resp.update(challenge, 64);
  std::unique_ptr<DevMem> d_buf;
  if (!host) d_buf.reset(new DevMem(sect_bytes(p.power, 3)));   // the largest section: 2^p G2 points
  uint8_t* sect[7] = {};
  for (int id = 2; id <= 6; id++) {
    const uint64_t n = sect_points(p.power, id);
    w.section(id, p.s[id].len);
    sect[id] = w.reserve(p.s[id].len);
    if (host) {
      memcpy(sect[id], p.s[id].p, p.s[id].len);
      if (sect_g2(id)) {
        key_section_host<Fq2>(sect[id], n, *first[id], tau);
        resp.points_host(reinterpret_cast<const G2Affine*>(sect[id]), n);
      } else {
        key_section_host<Fq>(sect[id], n, *first[id], tau);
        resp.points_host(reinterpret_cast<const G1Affine*>(sect[id]), n);
      }
    } else if (sect_g2(id)) {
      ms[id - 2] = key_section_device(p.s[id].p, n, *first[id], tau, static_cast<G2Affine*>(d_buf->p), resp, sect[id]);
    } else {
      ms[id - 2] = key_section_device(p.s[id].p, n, *first[id], tau, static_cast<G1Affine*>(d_buf->p), resp, sect[id]);
    }
  }
  uint8_t partial[kPartialLen], pk[kPubKeyLen], response[64];
  resp.h.partial(partial);
  pub_key(key, false, pk);
  resp.update(pk, kPubKeyLen);
  resp.h.final(response);

  // ---- nextChallenge: the new sections again, uncompressed
  Hasher nx(host, Enc::U);
  nx.update(response, 64);
  for (int id = 2; id <= 6; id++) {
    const uint64_t n = sect_points(p.power, id);
    if (host) {
      if (sect_g2(id)) nx.points_host(reinterpret_cast<const G2Affine*>(sect[id]), n);
      else nx.points_host(reinterpret_cast<const G1Affine*>(sect[id]), n);
    } else {
      NZCP_CUDA(cudaMemcpy(d_buf->p, sect[id], p.s[id].len, cudaMemcpyHostToDevice));
      if (sect_g2(id)) nx.points_device(static_cast<const G2Affine*>(d_buf->p), n);
      else nx.points_device(static_cast<const G1Affine*>(d_buf->p), n);
    }
  }
  uint8_t next[64];
  nx.h.final(next);
  ms[5] = resp.kernel_ms + nx.kernel_ms;
  ms[6] += resp.blake_ms + nx.blake_ms;

  // ---- section 7: the earlier records, then the new one
  const uint32_t type = beacon ? 1 : 0, plen = (uint32_t)params_len(a.name_len, beacon ? a.beacon_len : 0);
  std::vector<uint8_t> rec(kPtauRecFixed);
  uint8_t* r = rec.data();
  pub_key(key, true, r);
  memcpy(r + 768, sect[2] + 64, 64);     // tauG1[1]
  memcpy(r + 832, sect[3] + 128, 128);   // tauG2[1]
  memcpy(r + 960, sect[4], 64);          // alphaTauG1[0]
  memcpy(r + 1024, sect[5], 64);         // betaTauG1[0]
  memcpy(r + 1088, sect[6], 128);        // betaG2
  memcpy(r + 1216, partial, kPartialLen);
  memcpy(r + 1432, next, 64);
  memcpy(r + 1496, &type, 4);
  memcpy(r + 1500, &plen, 4);
  append_params(rec, a);
  w.section(7, p.s[7].len + rec.size());
  w.u32((uint32_t)p.recs.size() + 1);
  w.raw(p.s[7].p + 4, p.s[7].len - 4);
  w.raw(rec.data(), rec.size());
  if (w.pos != total) throw ApiError(NZCP_E_INTERNAL, "ptau contribute: size accounting error");
  if (written) *written = w.pos;
  if (hash_out) memcpy(hash_out, response, 64);
  if (ms_out) memcpy(ms_out, ms, sizeof ms);
}

}  // namespace
}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_ptau_new_size(uint32_t power, size_t* out_size) {
  return api_guard([&] {
    if (!out_size) throw ApiError(NZCP_E_ARG, "null argument");
    check_power(power);
    *out_size = new_size(power);
  });
}

int nzcp_ptau_new(uint32_t power, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]) {
  return api_guard([&] {
    if (!out) throw ApiError(NZCP_E_ARG, "null argument");
    check_power(power);
    const size_t total = new_size(power);
    if (cap < total) throw ApiError(NZCP_E_ARG, "output buffer too small");
    Writer w(out, cap);
    write_ptau_header(w, power, 7);
    const G1Affine g1 = g1_generator();
    const G2Affine g2 = g2_generator();
    for (int id = 2; id <= 6; id++) {
      const uint64_t n = sect_points(power, id);
      const size_t psz = sect_g2(id) ? 128 : 64;
      w.section(id, n * psz);
      uint8_t* dst = w.reserve(n * psz);
      for (uint64_t i = 0; i < n; i++) memcpy(dst + i * psz, sect_g2(id) ? (const void*)&g2 : (const void*)&g1, psz);
    }
    w.section(7, 4);
    w.u32(0);
    if (w.pos != total) throw ApiError(NZCP_E_INTERNAL, "ptau new: size accounting error");
    if (written) *written = w.pos;
    if (hash) first_challenge(power, hash, nullptr);
  });
}

int nzcp_ptau_contribute_size(const uint8_t* ptau, size_t len, const char* name, size_t beacon_hash_len, size_t* out_size) {
  return api_guard([&] {
    if (!ptau || !out_size) throw ApiError(NZCP_E_ARG, "null argument");
    size_t name_len;
    check_name("ptau", name, &name_len);
    check_beacon_len(beacon_hash_len);
    *out_size = contribute_size(parse_contrib_in(ptau, len), name_len, beacon_hash_len);
  });
}

int nzcp_ptau_contribute(const uint8_t* ptau, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                         const uint8_t* seed, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                         float ms[7]) {
  return api_guard([&] {
    if (!ptau || !out || (entropy_len && !entropy)) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    ContribArgs a;
    a.name = name;
    a.entropy = entropy;
    a.entropy_len = entropy_len;
    a.seed = seed;
    contribute_impl(ptau, len, a, device, out, cap, written, hash, ms);
  });
}

int nzcp_ptau_beacon(const uint8_t* ptau, size_t len, const char* name, const uint8_t* beacon_hash, size_t beacon_hash_len,
                     uint32_t num_iterations_exp, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                     float ms[7]) {
  return api_guard([&] {
    if (!ptau || !out || !beacon_hash) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    ContribArgs a;
    a.name = name;
    a.beacon = beacon_hash;
    a.beacon_len = beacon_hash_len;
    a.exp = num_iterations_exp;
    contribute_impl(ptau, len, a, device, out, cap, written, hash, ms);
  });
}

int nzcp_host_ptau_contribute(const uint8_t* ptau, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                              const uint8_t* seed, const uint8_t* beacon_hash, size_t beacon_hash_len,
                              uint32_t num_iterations_exp, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]) {
  return api_guard([&] {
    if (!ptau || !out || (entropy_len && !entropy)) throw ApiError(NZCP_E_ARG, "null argument");
    ContribArgs a;
    a.name = name;
    a.entropy = entropy;
    a.entropy_len = entropy_len;
    a.seed = seed;
    a.beacon = beacon_hash;
    a.beacon_len = beacon_hash_len;
    a.exp = num_iterations_exp;
    contribute_impl(ptau, len, a, -1, out, cap, written, hash, nullptr);
  });
}

}  // extern "C"
