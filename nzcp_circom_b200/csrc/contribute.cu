// `zkey contribute` and `zkey beacon` on the GPU: one phase-2 contribution to the delta of a Groth16 key.
//
// Replaces snarkjs 0.4.12 src/zkey_contribute.js phase2contribute(zkeyNameOld, zkeyNameNew, name, entropy) and
// src/zkey_beacon.js beacon(zkeyNameOld, zkeyNameNew, name, beaconHashStr, numIterationsExp) (upstream, not vendored:
// package.json:12, yarn.lock:987-999).  The two differ only in where the random generator comes from.  Restated:
//   rng        ffjavascript ChaCha(seed), seed = 8 u32 read BIG-endian from the first 32 bytes of
//                contribute: BLAKE2b-512(64 OS-random bytes || UTF-8 entropy)       (snarkjs misc.js getRandomRng)
//                beacon:     SHA-256 applied 2^numIterationsExp times to beaconHash  (misc.js rngFromBeaconParams)
//   k          Fr.fromRng(rng): the drawn buffer is taken as the MONTGOMERY form, k = v * 2^-256 mod r
//   g1_s       G1.fromRng(rng) (cofactor 1), g1_sx = k * g1_s
//   transcript BLAKE2b-512(csHash || hashPubKey(c) for every earlier contribution || U(g1_s) || U(g1_sx))
//   g2_sp      hashToG2(transcript) = G2.fromRng(ChaCha(transcript[0..32) as 8 BE words)) incl. the cofactor 2q - r,
//              g2_spx = k * g2_sp
//   header     delta1 <- k * delta1, delta2 <- k * delta2, nothing else; deltaAfter = the new delta1
//   sections   1-7 copied (2 with the new delta), 8 (L) and 9 (H): every point * k^-1 (applyKeyToSection(invDelta, 1)),
//              infinity stays (0,0); 10 = the earlier records + the new one (type 0 contribute / 1 beacon; parameters
//              tag 1 name, tag 2 numIterationsExp, tag 3 beaconHash).  Output: 10 sections in the order 1, 2, ..., 10.
//   returns    BLAKE2b-512(hashPubKey(new contribution))
// hashPubKey(c) = U(deltaAfter) || U(g1_s) || U(g1_sx) || U(g2_spx) || c.transcript, U = uncompressed encoding: big-endian
// plain coordinates, G2 as x.c1 x.c0 y.c1 y.c0, infinity = all zero but the first byte 0x40.
// Earlier records are copied byte for byte; snarkjs re-serializes them from their parsed form, which gives the same bytes
// for every record snarkjs writes.  Deviation: a name longer than 64 bytes is rejected (snarkjs cuts it at 64 characters,
// and a cut in bytes could split a UTF-8 sequence).
//
// B200 design.  The O(1) part (rng, hashes, the few header / record multiplications) runs on the host.  The bulk is
// sections 8 and 9, 2 x 2^27 points at most (8.6 GB each, resident in HBM one at a time): one thread per point,
// x[i] = to_affine_fast(k^-1 * x[i]) with the signed 4-bit window of ec.cuh scalar_mul_accumulate.  The scalar is the
// same for the whole launch, so every lane takes the same additions at the same digits.
#include "mpc.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ shared host/device code
HD G1Affine scale_point(const G1Affine& p, const Fr& k) {   // k plain, < r
  G1XYZZ acc = G1XYZZ::inf();
  scalar_mul_accumulate(acc, p, k);
  return to_affine_fast(acc);
}

struct ZkeyScale {   // Exec op
  G1Affine* x;
  Fr k;
  HD void operator()(uint64_t i) const { x[i] = scale_point(x[i], k); }
};

namespace {

size_t contribute_size(const ZkeyIn& z, size_t name_len, size_t beacon_len) {
  size_t total = 12 + 10 * 12 + 4 + kZkeyHeaderLen;
  for (int id = 3; id <= 10; id++) total += z.s[id].len;
  return total + kRecFixed + params_len(name_len, beacon_len);
}

// device < 0: the host hook.
void contribute_impl(const uint8_t* b, size_t len, ContribArgs a, int device, uint8_t* out, size_t cap, size_t* written,
                     uint8_t* hash_out, float* section_ms) {
  check_contrib_args("zkey", a);
  const bool beacon = a.beacon != nullptr;
  const ZkeyIn z = parse_zkey_in(b, len);
  const size_t total = contribute_size(z, a.name_len, beacon ? a.beacon_len : 0);
  if (cap < total) throw ApiError(NZCP_E_ARG, "output buffer too small");
  const bool host = device < 0;
  if (host && z.n_l() + z.domain_size > kHostMaxPoints)
    throw ApiError(NZCP_E_ARG, "zkey: the host run is limited to 4096 points in sections 8 and 9");
  if (!host) use_device(device);

  // ---- the rng
  uint8_t seed[64];
  contrib_seed(a, seed);
  ChaCha rng(seed);

  // ---- the contribution (host: O(1) multiplications)
  const Fr k_mont = fp_from_rng<FrParams>(rng);
  if (k_mont.is_zero()) throw ApiError(NZCP_E_INTERNAL, "zkey contribute: the rng drew the zero key");
  const Fr k = fp_from_mont(k_mont), k_inv = fp_from_mont(fp_inv(k_mont));
  const Fq b1 = curve_b(g1_generator());
  const G1Affine g1_s = point_from_rng(rng, b1, nullptr);
  const G1Affine g1_sx = mul_plain(g1_s, k.v);

  Blake2b512 th;
  th.update(z.s[10].p, 64);                                   // csHash
  for (const uint8_t* r : z.recs) hash_pub_key(th, r);
  uint8_t tmp[64];
  memcpy(tmp, &g1_s, 64);
  hash_g1(th, tmp);
  memcpy(tmp, &g1_sx, 64);
  hash_g1(th, tmp);
  uint8_t transcript[64];
  th.final(transcript);

  const G2Affine g2_sp = hash_to_g2(transcript);
  const G2Affine g2_spx = mul_plain(g2_sp, k.v);

  G1Affine d1;
  G2Affine d2;
  memcpy(&d1, z.s[2].p + kZkeyDelta1Off, 64);
  memcpy(&d2, z.s[2].p + kZkeyDelta2Off, 128);
  d1 = mul_plain(d1, k.v);
  d2 = mul_plain(d2, k.v);

  // ---- the new record
  uint8_t fixed[kRecFixed];
  memcpy(fixed, &d1, 64);                                      // deltaAfter
  memcpy(fixed + 64, &g1_s, 64);
  memcpy(fixed + 128, &g1_sx, 64);
  memcpy(fixed + 192, &g2_spx, 128);
  memcpy(fixed + 320, transcript, 64);
  const uint32_t type = beacon ? 1 : 0, plen = (uint32_t)params_len(a.name_len, beacon ? a.beacon_len : 0);
  memcpy(fixed + 384, &type, 4);
  memcpy(fixed + 388, &plen, 4);
  std::vector<uint8_t> rec(fixed, fixed + kRecFixed);
  append_params(rec, a);
  if (hash_out) {
    Blake2b512 ch;
    hash_pub_key(ch, rec.data());
    ch.final(hash_out);
  }

  // ---- the file, sections 1 .. 10 in id order
  Writer w(out, cap);
  w.raw("zkey", 4);
  w.u32(1);
  w.u32(10);
  w.section(1, 4);
  w.u32(1);
  w.section(2, kZkeyHeaderLen);
  uint8_t* hdr = w.reserve(kZkeyHeaderLen);
  memcpy(hdr, z.s[2].p, kZkeyHeaderLen);
  memcpy(hdr + kZkeyDelta1Off, &d1, 64);
  memcpy(hdr + kZkeyDelta2Off, &d2, 128);
  for (int id = 3; id <= 7; id++) {
    w.section(id, z.s[id].len);
    w.raw(z.s[id].p, z.s[id].len);
  }
  Exec ex(host);
  const size_t buf_bytes = std::max<uint64_t>(z.n_l(), z.domain_size) * 64;
  G1Affine* buf = reinterpret_cast<G1Affine*>(ex.alloc<unsigned char>(buf_bytes ? buf_bytes : 16));
  for (int id = 8; id <= 9; id++) {
    const uint64_t n = id == 8 ? z.n_l() : z.domain_size;
    w.section(id, n * 64);
    uint8_t* dst = w.reserve(n * 64);
    float ms = 0;
    if (n) {   // the scale alone is timed
      ex.upload(buf, z.s[id].p, n * 64);
      Timer t = ex.timer();
      ex.run<128>(n, ZkeyScale{buf, k_inv});
      t.end();
      ex.download(dst, buf, n * 64);
      ms = t.ms();
    }
    if (section_ms) section_ms[id - 8] = ms;
  }
  w.section(10, z.s[10].len + rec.size());
  w.raw(z.s[10].p, 64);
  w.u32((uint32_t)z.recs.size() + 1);
  w.raw(z.s[10].p + 68, z.s[10].len - 68);
  w.raw(rec.data(), rec.size());
  if (w.pos != total) throw ApiError(NZCP_E_INTERNAL, "zkey contribute: size accounting error");
  if (written) *written = w.pos;
}

}  // namespace
}  // namespace nzcp

using namespace nzcp;

extern "C" {

int nzcp_zkey_contribute_size(const uint8_t* zkey, size_t len, const char* name, size_t beacon_hash_len, size_t* out_size) {
  return api_guard([&] {
    if (!zkey || !out_size) throw ApiError(NZCP_E_ARG, "null argument");
    size_t name_len;
    check_name("zkey", name, &name_len);
    check_beacon_len(beacon_hash_len);
    *out_size = contribute_size(parse_zkey_in(zkey, len), name_len, beacon_hash_len);
  });
}

int nzcp_zkey_contribute(const uint8_t* zkey, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                         const uint8_t* seed, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                         float section_ms[2]) {
  return api_guard([&] {
    if (!zkey || !out || (entropy_len && !entropy)) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    ContribArgs a;
    a.name = name;
    a.entropy = entropy;
    a.entropy_len = entropy_len;
    a.seed = seed;
    contribute_impl(zkey, len, a, device, out, cap, written, hash, section_ms);
  });
}

int nzcp_zkey_beacon(const uint8_t* zkey, size_t len, const char* name, const uint8_t* beacon_hash, size_t beacon_hash_len,
                     uint32_t num_iterations_exp, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                     float section_ms[2]) {
  return api_guard([&] {
    if (!zkey || !out || !beacon_hash) throw ApiError(NZCP_E_ARG, "null argument");
    if (device < 0) throw ApiError(NZCP_E_ARG, "device index out of range");
    ContribArgs a;
    a.name = name;
    a.beacon = beacon_hash;
    a.beacon_len = beacon_hash_len;
    a.exp = num_iterations_exp;
    contribute_impl(zkey, len, a, device, out, cap, written, hash, section_ms);
  });
}

int nzcp_host_zkey_contribute(const uint8_t* zkey, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                              const uint8_t* seed, const uint8_t* beacon_hash, size_t beacon_hash_len,
                              uint32_t num_iterations_exp, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]) {
  return api_guard([&] {
    if (!zkey || !out || (entropy_len && !entropy)) throw ApiError(NZCP_E_ARG, "null argument");
    ContribArgs a;
    a.name = name;
    a.entropy = entropy;
    a.entropy_len = entropy_len;
    a.seed = seed;
    a.beacon = beacon_hash;
    a.beacon_len = beacon_hash_len;
    a.exp = num_iterations_exp;
    contribute_impl(zkey, len, a, -1, out, cap, written, hash, nullptr);
  });
}

}  // extern "C"
