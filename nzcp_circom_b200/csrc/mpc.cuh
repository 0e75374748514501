// Code shared by the ceremony entry points (contribute.cu `zkey contribute` / `zkey beacon`, verify.cu `zkey verify`,
// setup.cu `zkey new`, ptau_contribute.cu `powersoftau new` / `contribute` / `beacon`, ptau_verify.cu `powersoftau verify`):
// BLAKE2b-512 and SHA-256, ffjavascript's ChaCha, F/G.fromRng, the uncompressed and compressed point encodings (host and
// device) with the chunked point hasher, the contribution records with the .zkey input of `zkey contribute` / `zkey
// verify`, the phase-1 key, and the claims and chunked MSM sums of the two verify steps.
#pragma once
#include <sys/random.h>

#include <chrono>

#include "binfile.cuh"

namespace nzcp {
namespace {

// ------------------------------------------------------------------------------------------------ hashes (host)
struct Blake2b512 {   // RFC 7693, unkeyed, 64-byte digest
  uint64_t h[8], t = 0;
  uint8_t buf[128] = {};   // zero at init, as the RFC's blake2b_ctx: partial() serializes stale bytes too
  size_t n = 0;
  static constexpr uint64_t kIv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull,
                                      0xa54ff53a5f1d36f1ull, 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full,
                                      0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
  Blake2b512() {
    for (int i = 0; i < 8; i++) h[i] = kIv[i];
    h[0] ^= 0x01010000ull ^ 64;
  }
  static uint64_t rotr(uint64_t x, int c) { return (x >> c) | (x << (64 - c)); }
  void compress(bool last) {
    static const uint8_t kSigma[10][16] = {
        {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
        {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
        {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
        {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
        {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0}};
    uint64_t m[16], v[16];
    memcpy(m, buf, 128);   // little-endian host
    for (int i = 0; i < 8; i++) { v[i] = h[i]; v[i + 8] = kIv[i]; }
    v[12] ^= t;
    if (last) v[14] = ~v[14];
    auto g = [&](int a, int b, int c, int d, uint64_t x, uint64_t y) {
      v[a] += v[b] + x; v[d] = rotr(v[d] ^ v[a], 32); v[c] += v[d]; v[b] = rotr(v[b] ^ v[c], 24);
      v[a] += v[b] + y; v[d] = rotr(v[d] ^ v[a], 16); v[c] += v[d]; v[b] = rotr(v[b] ^ v[c], 63);
    };
    for (int r = 0; r < 12; r++) {
      const uint8_t* s = kSigma[r % 10];
      g(0, 4, 8, 12, m[s[0]], m[s[1]]); g(1, 5, 9, 13, m[s[2]], m[s[3]]);
      g(2, 6, 10, 14, m[s[4]], m[s[5]]); g(3, 7, 11, 15, m[s[6]], m[s[7]]);
      g(0, 5, 10, 15, m[s[8]], m[s[9]]); g(1, 6, 11, 12, m[s[10]], m[s[11]]);
      g(2, 7, 8, 13, m[s[12]], m[s[13]]); g(3, 4, 9, 14, m[s[14]], m[s[15]]);
    }
    for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
  }
  void update(const void* p, size_t len) {
    const uint8_t* s = static_cast<const uint8_t*>(p);
    while (len) {
      if (n == 128) {   // a full block is compressed only once more input follows: the last block takes the final flag
        t += 128;
        compress(false);
        n = 0;
      }
      const size_t c = std::min(128 - n, len);
      memcpy(buf + n, s, c);
      n += c; s += c; len -= c;
    }
  }
  void final(uint8_t out[64]) {
    t += n;
    memset(buf + n, 0, 128 - n);
    compress(true);
    memcpy(out, h, 64);
  }
  // The state as blake2b-wasm's getPartialHash returns it: RFC 7693's blake2b_ctx, 216 bytes: b[128] (stale bytes past c
  // kept), h[8] and t[2] as u64 LE, c and outlen (64) as u32 LE.  c = 128 when a full block waits (lazy compression).
  void partial(uint8_t out[216]) const {
    const uint64_t tt[2] = {t, 0};
    const uint32_t c = (uint32_t)n, outlen = 64;
    memcpy(out, buf, 128);
    memcpy(out + 128, h, 64);
    memcpy(out + 192, tt, 16);
    memcpy(out + 208, &c, 4);
    memcpy(out + 212, &outlen, 4);
  }
  // The inverse of partial(): the hasher a partialHash describes, to be resumed with update().  The caller has checked
  // c <= 128, t[1] = 0 and outlen = 64.
  static Blake2b512 from_partial(const uint8_t in[216]) {
    Blake2b512 s;
    memcpy(s.buf, in, 128);
    memcpy(s.h, in + 128, 64);
    memcpy(&s.t, in + 192, 8);
    s.n = rd32u(in + 208);
    return s;
  }
};

void sha256(const uint8_t* msg, size_t len, uint8_t out[32]) {   // FIPS 180-4
  static const uint32_t kK[64] = {
      0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01,
      0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc,
      0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147,
      0x06ca6351, 0x14292967, 0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85,
      0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08,
      0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208,
      0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
  uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
  auto rotr = [](uint32_t x, int c) { return (x >> c) | (x << (32 - c)); };
  std::vector<uint8_t> m(msg, msg + len);
  m.push_back(0x80);
  while (m.size() % 64 != 56) m.push_back(0);
  for (int i = 7; i >= 0; i--) m.push_back((uint8_t)(((uint64_t)len * 8) >> (8 * i)));
  for (size_t off = 0; off < m.size(); off += 64) {
    uint32_t w[64];
    for (int i = 0; i < 16; i++)
      w[i] = (uint32_t)m[off + 4 * i] << 24 | (uint32_t)m[off + 4 * i + 1] << 16 | (uint32_t)m[off + 4 * i + 2] << 8 | m[off + 4 * i + 3];
    for (int i = 16; i < 64; i++) {
      const uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
      const uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
      w[i] = w[i - 16] + s0 + w[i - 7] + s1;
    }
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
    for (int i = 0; i < 64; i++) {
      const uint32_t t1 = hh + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + kK[i] + w[i];
      const uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
      hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
  }
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(h[i] >> (24 - 8 * j));
}

// ------------------------------------------------------------------------------------------------ ffjavascript ChaCha
// RFC 8439 ChaCha20 with key = the little-endian bytes of the 8 seed words, counter and nonce 0; word 12 is the block
// counter and carries into words 13-15.  nextU32 walks the 16 output words of each block.
struct ChaCha {
  uint32_t state[16], out[16];
  int idx = 16;
  explicit ChaCha(const uint8_t seed_be[32]) {
    const uint32_t c[4] = {0x61707865, 0x3320646E, 0x79622D32, 0x6B206574};
    for (int i = 0; i < 4; i++) state[i] = c[i];
    for (int i = 0; i < 8; i++)
      state[4 + i] = (uint32_t)seed_be[4 * i] << 24 | (uint32_t)seed_be[4 * i + 1] << 16 | (uint32_t)seed_be[4 * i + 2] << 8 |
                     seed_be[4 * i + 3];
    for (int i = 12; i < 16; i++) state[i] = 0;
  }
  static uint32_t rotl(uint32_t x, int c) { return (x << c) | (x >> (32 - c)); }
  void update() {
    uint32_t x[16];
    memcpy(x, state, sizeof x);
    auto qr = [&](int a, int b, int c, int d) {
      x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16); x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12);
      x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8); x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7);
    };
    for (int i = 0; i < 10; i++) {
      qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15);
      qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14);
    }
    for (int i = 0; i < 16; i++) out[i] = x[i] + state[i];
    idx = 0;
    for (int i = 12; i < 16 && ++state[i] == 0; i++) {}
  }
  uint32_t next_u32() {
    if (idx == 16) update();
    return out[idx++];
  }
  uint64_t next_u64() {   // the first draw is the high half
    const uint64_t hi = next_u32();
    return hi << 32 | next_u32();
  }
  bool next_bool() { return next_u32() & 1; }
};

// ------------------------------------------------------------------------------------------------ fields and points (host)
// F.fromRng of wasmcurves: v = sum_i nextU64 * 2^(64 i), masked to 254 bits, redrawn while v >= p; the buffer v is the
// Montgomery form of the element.
template <class P>
Fp<P> fp_from_rng(ChaCha& rng) {
  Fp<P> v;
  do {
    for (int i = 0; i < 4; i++) {
      const uint64_t w = rng.next_u64();
      v.v[2 * i] = (uint32_t)w;
      v.v[2 * i + 1] = (uint32_t)(w >> 32);
    }
    v.v[7] &= 0x3FFFFFFFu;
  } while (fp_geq_mod<P>(v.v));
  return v;
}

// (q + add) >> shift as 8 limbs; add = +-1 changes limb 0 alone (q's low limb is 0xd87cfd47)
void q_exp(int add, int shift, uint32_t e[8]) {
  for (int i = 0; i < 8; i++) e[i] = FqParams::mod(i);
  e[0] += add;
  for (int i = 0; i < 8; i++) e[i] = (e[i] >> shift) | (i < 7 ? e[i + 1] << (32 - shift) : 0);
}

bool fq_is_square(const Fq& a) {   // Euler: a^((q-1)/2) in {0, 1}
  uint32_t e[8];
  q_exp(-1, 1, e);
  const Fq t = fp_pow(a, e);
  return a.is_zero() || t == Fq::one();
}

Fq fq_sqrt(const Fq& a) {   // q = 3 mod 4: a^((q+1)/4), valid for a square a
  uint32_t e[8];
  q_exp(1, 2, e);
  return fp_pow(a, e);
}

// isNegative as wasmcurves defines it: the plain value is > (q-1)/2.  For Fq2: c1 decides, c0 when c1 = 0.
bool fq_is_negative(const Fq& a) {
  uint32_t h[8];
  q_exp(-1, 1, h);
  const Fq p = fp_from_mont(a);
  for (int i = 7; i >= 0; i--)
    if (p.v[i] != h[i]) return p.v[i] > h[i];
  return false;
}
bool fq2_is_negative(const Fq2& a) { return a.c1.is_zero() ? fq_is_negative(a.c0) : fq_is_negative(a.c1); }

// Fq2 = Fq[u]/(u^2 + 1), q = 3 mod 4 (-1 is not a square in Fq): a is a square iff its norm c0^2 + c1^2 is a square in Fq.
bool fq2_is_square(const Fq2& a) { return fq_is_square(fp_add(fp_sqr(a.c0), fp_sqr(a.c1))); }

Fq2 fq2_sqrt(const Fq2& a) {   // a square; x0^2 = (c0 +- sqrt(norm)) / 2, x1 = c1 / (2 x0)
  Fq2 r;
  if (a.c1.is_zero()) {
    if (fq_is_square(a.c0)) r = Fq2{fq_sqrt(a.c0), Fq::zero()};
    else r = Fq2{Fq::zero(), fq_sqrt(fp_neg(a.c0))};
  } else {
    const Fq n = fq_sqrt(fp_add(fp_sqr(a.c0), fp_sqr(a.c1)));
    const Fq half = fp_inv(fp_add(Fq::one(), Fq::one()));
    Fq t = fp_mul(fp_add(a.c0, n), half);
    if (!fq_is_square(t)) t = fp_mul(fp_sub(a.c0, n), half);
    const Fq x0 = fq_sqrt(t);
    r = Fq2{x0, fp_mul(a.c1, fp_inv(fp_add(x0, x0)))};
  }
  if (f_sqr(r) != a) throw ApiError(NZCP_E_INTERNAL, "zkey contribute: Fq2 square root failed");
  return r;
}

bool is_square(const Fq& a) { return fq_is_square(a); }
bool is_square(const Fq2& a) { return fq2_is_square(a); }
Fq sqrt_of(const Fq& a) { return fq_sqrt(a); }
Fq2 sqrt_of(const Fq2& a) { return fq2_sqrt(a); }
bool is_negative(const Fq& a) { return fq_is_negative(a); }
bool is_negative(const Fq2& a) { return fq2_is_negative(a); }
Fq f_from_rng(ChaCha& rng, Fq*) { return fp_from_rng<FqParams>(rng); }
Fq2 f_from_rng(ChaCha& rng, Fq2*) {
  const Fq c0 = fp_from_rng<FqParams>(rng);
  return Fq2{c0, fp_from_rng<FqParams>(rng)};
}

// k * P for a plain 256-bit k (xyzz_mul: no reduction of k, valid for any point of the curve).
template <class F>
Affine<F> mul_plain(const Affine<F>& p, const uint32_t k[8]) { return xyzz_to_affine(xyzz_mul(XYZZ<F>::from_affine(p), k)); }

// G.fromRng: x = F.fromRng, greatest = nextBool, until x^3 + b is a square; y = sqrt, negated when greatest differs from
// isNegative(y); then times the cofactor (a plain integer: the point is not in the order-r subgroup yet).
template <class F>
Affine<F> point_from_rng(ChaCha& rng, const F& b, const uint32_t* cofactor) {
  F x, rhs;
  bool greatest;
  do {
    x = f_from_rng(rng, (F*)nullptr);
    greatest = rng.next_bool();
    rhs = f_add(f_mul(f_sqr(x), x), b);
  } while (!is_square(rhs));
  F y = sqrt_of(rhs);
  if (greatest != is_negative(y)) y = f_neg(y);
  const Affine<F> p{x, y};
  return cofactor ? mul_plain(p, cofactor) : p;
}

// rngFromBeaconParams (misc.js): SHA-256 applied 2^exp times to the beacon hash; the first 32 bytes seed the ChaCha.
void beacon_seed(const uint8_t* beacon, size_t len, uint32_t exp, uint8_t seed[32]) {
  std::vector<uint8_t> cur(beacon, beacon + len);
  const uint64_t inner = exp < 32 ? (uint64_t)1 << exp : (uint64_t)1 << 32;
  const uint64_t outer = exp < 32 ? 1 : (uint64_t)1 << (exp - 32);
  for (uint64_t o = 0; o < outer; o++)
    for (uint64_t i = 0; i < inner; i++) {
      uint8_t d[32];
      sha256(cur.data(), cur.size(), d);
      cur.assign(d, d + 32);
    }
  memcpy(seed, cur.data(), 32);
}

// ------------------------------------------------------------------------------------------------ contribute / beacon
// What a caller of `contribute` (beacon == nullptr) or `beacon` asks for.
struct ContribArgs {
  const char* name = nullptr;
  size_t name_len = 0;
  const uint8_t* entropy = nullptr;
  size_t entropy_len = 0;
  const uint8_t* seed = nullptr;
  const uint8_t* beacon = nullptr;
  size_t beacon_len = 0;
  uint32_t exp = 0;
};

// kind: "zkey" or "ptau", for the message.  A name longer than 64 bytes is rejected (snarkjs cuts it at 64 characters,
// and a cut in bytes could split a UTF-8 sequence).
void check_name(const char* kind, const char* name, size_t* len) {
  *len = name ? strlen(name) : 0;
  if (*len > 64) throw ApiError(NZCP_E_ARG, std::string(kind) + ": contribution name longer than 64 bytes");
}

void check_beacon_len(size_t len) {
  if (len >= 256) throw ApiError(NZCP_E_ARG, "Maximum lenght of beacon hash is 255 bytes");
}

void check_contrib_args(const char* kind, ContribArgs& a) {
  check_name(kind, a.name, &a.name_len);
  check_beacon_len(a.beacon_len);
  if (a.beacon) {
    if (a.beacon_len == 0) throw ApiError(NZCP_E_ARG, "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)");
    if (a.exp < 10 || a.exp > 63) throw ApiError(NZCP_E_ARG, "Invalid numIterationsExp. (Must be between 10 and 63)");
  }
}

size_t params_len(size_t name_len, size_t beacon_len) {
  return (name_len ? 2 + name_len : 0) + (beacon_len ? 2 + 2 + beacon_len : 0);
}

// The record's parameters: tag 1 name (if any), tag 2 numIterationsExp and tag 3 beaconHash (beacon only).
void append_params(std::vector<uint8_t>& rec, const ContribArgs& a) {
  if (a.name_len) {
    rec.insert(rec.end(), {1, (uint8_t)a.name_len});
    rec.insert(rec.end(), a.name, a.name + a.name_len);
  }
  if (a.beacon) {
    rec.insert(rec.end(), {2, (uint8_t)a.exp, 3, (uint8_t)a.beacon_len});
    rec.insert(rec.end(), a.beacon, a.beacon + a.beacon_len);
  }
}

// The ChaCha seed: beacon_seed for a beacon; else BLAKE2b-512(64 OS-random bytes || entropy) (misc.js getRandomRng), or the
// 32-byte test seed.
void contrib_seed(const ContribArgs& a, uint8_t seed[64]) {
  if (a.beacon) {
    beacon_seed(a.beacon, a.beacon_len, a.exp, seed);
  } else if (a.seed) {
    memcpy(seed, a.seed, 32);
  } else {
    uint8_t os[64];
    for (size_t got = 0; got < sizeof os;) {
      const ssize_t r = getrandom(os + got, sizeof os - got, 0);
      if (r <= 0) throw ApiError(NZCP_E_INTERNAL, "contribute: no OS randomness");
      got += (size_t)r;
    }
    Blake2b512 h;
    h.update(os, sizeof os);
    if (a.entropy_len) h.update(a.entropy, a.entropy_len);
    h.final(seed);
  }
}

// hashToG2 (zkey_utils.js): G2.fromRng(ChaCha(transcript[0..32) as 8 BE words)), times the G2 cofactor 2q - r.
G2Affine hash_to_g2(const uint8_t transcript[64]) {
  uint32_t h2[8];
  int64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += 2 * (int64_t)FqParams::mod(i) - (int64_t)FrParams::mod(i);
    h2[i] = (uint32_t)c;
    c >>= 32;                                                // arithmetic: a borrow is -1
  }
  ChaCha rng(transcript);
  return point_from_rng(rng, curve_b(g2_generator()), h2);
}

// ------------------------------------------------------------------------------------------------ hashPubKey encodings
void be32(const Fq& a, uint8_t* out) {   // plain value, big-endian
  const Fq p = fp_from_mont(a);
  for (int i = 0; i < 32; i++) out[i] = (uint8_t)(p.v[7 - i / 4] >> (8 * (3 - i % 4)));
}
void hash_g1(Blake2b512& h, const uint8_t* mont64) {
  G1Affine a;
  memcpy(&a, mont64, 64);
  uint8_t u[64] = {0};
  if (a.is_inf()) {
    u[0] = 0x40;
  } else {
    be32(a.x, u);
    be32(a.y, u + 32);
  }
  h.update(u, 64);
}
void hash_g2(Blake2b512& h, const uint8_t* mont128) {
  G2Affine a;
  memcpy(&a, mont128, 128);
  uint8_t u[128] = {0};
  if (a.is_inf()) {
    u[0] = 0x40;
  } else {
    be32(a.x.c1, u);
    be32(a.x.c0, u + 32);
    be32(a.y.c1, u + 64);
    be32(a.y.c0, u + 96);
  }
  h.update(u, 128);
}

constexpr size_t kRecFixed = 3 * 64 + 128 + 64 + 4 + 4;   // deltaAfter g1_s g1_sx g2_spx transcript type paramLength

void hash_pub_key(Blake2b512& h, const uint8_t* rec) {
  hash_g1(h, rec);
  hash_g1(h, rec + 64);
  hash_g1(h, rec + 128);
  hash_g2(h, rec + 192);
  h.update(rec + 320, 64);
}

// ------------------------------------------------------------------------------------------------ input
constexpr uint64_t kHostMaxPoints = 1u << 12;

struct ZkeyIn : Zkey {
  std::vector<const uint8_t*> recs;   // section-10 records
  std::vector<size_t> rec_len;
};

// readMPCParams (zkey_utils.js) / readContributions (powersoftau_utils.js): `head` bytes (the zkey's csHash), u32
// nContributions, then the records: rec_fixed bytes whose last u32 is paramLength, then the parameters, tag-prefixed and
// strictly increasing.  `what` names the section in the messages.
void parse_records(const uint8_t* p, uint64_t len, uint64_t head, size_t rec_fixed, const std::string& what,
                   std::vector<const uint8_t*>& recs, std::vector<size_t>& rec_len) {
  if (len < head + 4) throw ApiError(NZCP_E_FORMAT, what + " is truncated");
  const uint32_t n = rd32u(p + head);
  uint64_t pos = head + 4;
  for (uint32_t c = 0; c < n; c++) {
    if (len - pos < rec_fixed) throw ApiError(NZCP_E_FORMAT, what + " is truncated");
    const uint64_t start = pos;
    const uint32_t plen = rd32u(p + pos + rec_fixed - 4);
    pos += rec_fixed;
    const uint64_t end = pos + plen;
    int last = 0;
    while (pos < end) {
      auto need = [&](uint64_t k) {
        if (pos + k > len) throw ApiError(NZCP_E_FORMAT, what + " is truncated");
      };
      need(1);
      const int tag = p[pos++];
      if (tag <= last) throw ApiError(NZCP_E_FORMAT, "Parameters in the contribution must be sorted");
      last = tag;
      if (tag == 1 || tag == 3) {
        need(1);
        const uint64_t l = p[pos++];
        need(l);
        pos += l;
      } else if (tag == 2) {
        need(1);
        pos += 1;
      } else {
        throw ApiError(NZCP_E_FORMAT, "Parameter not recognized");
      }
    }
    if (pos != end) throw ApiError(NZCP_E_FORMAT, "Parametes do not match");   // snarkjs's spelling
    recs.push_back(p + start);
    rec_len.push_back(end - start);
  }
  if (pos != len) throw ApiError(NZCP_E_FORMAT, what + " has trailing bytes");
}

void parse_mpc(ZkeyIn& z) { parse_records(z.s[10].p, z.s[10].len, 64, kRecFixed, "zkey: section 10", z.recs, z.rec_len); }

// The input of `zkey contribute` / `zkey verify`: read_zkey, then a header of exactly 660 bytes, sections 3-10, the sizes
// of 8 and 9 and the records.  check_pts = false: the caller checks the points of sections 2, 8 and 9 itself.
ZkeyIn parse_zkey_in(const uint8_t* b, size_t len, bool check_pts = true) {
  ZkeyIn z{read_zkey(b, len)};
  if (z.s[2].len != kZkeyHeaderLen) throw ApiError(NZCP_E_FORMAT, "zkey: header section 2 is not 660 bytes");
  need_sections(z.s, 3, 10);
  if (z.s[8].len != z.n_l() * 64) throw ApiError(NZCP_E_FORMAT, "zkey: section 8 size does not match nVars - nPublic - 1");
  if (z.s[9].len != (uint64_t)z.domain_size * 64)
    throw ApiError(NZCP_E_FORMAT, "zkey: section 9 size does not match domainSize");
  parse_mpc(z);
  if (!check_pts) return z;
  const Fq b1 = curve_b(g1_generator());
  const Fq2 b2 = curve_b(g2_generator());
  check_points<Fq>("zkey", z.s[2].p + kZkeyDelta1Off, 1, 2, b1);
  check_points<Fq2>("zkey", z.s[2].p + kZkeyDelta2Off, 1, 2, b2);
  check_points<Fq>("zkey", z.s[8].p, z.n_l(), 8, b1);
  check_points<Fq>("zkey", z.s[9].p, z.domain_size, 9, b1);
  return z;
}

// ------------------------------------------------------------------------------------------------ point encodings (device)
HD uint32_t bswap32(uint32_t v) { return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24); }
HD void put_be(const Fq& a, uint32_t* w) {
  const Fq p = fp_from_mont(a);
  for (int j = 0; j < 8; j++) w[j] = bswap32(p.v[7 - j]);
}
HD void put_be(const Fq2& a, uint32_t* w) {   // c1 first
  put_be(a.c1, w);
  put_be(a.c0, w + 8);
}

// wasmcurves isNegative / F2 sign: the plain value is > (q-1)/2 = q >> 1; for Fq2 c1 decides, c0 when c1 = 0.
HD bool y_negative(const Fq& a) {
  const Fq p = fp_from_mont(a);
  for (int i = 7; i >= 0; i--) {
    const uint32_t h = (FqParams::mod(i) >> 1) | (i < 7 ? FqParams::mod(i + 1) << 31 : 0);
    if (p.v[i] != h) return p.v[i] > h;
  }
  return false;
}
HD bool y_negative(const Fq2& a) { return a.c1.is_zero() ? y_negative(a.c0) : y_negative(a.c1); }

// U(P) as little-endian words: big-endian plain coordinates; infinity = 0x40 then zeros.
template <class F>
HD void u_encode(const Affine<F>& a, uint32_t* w) {
  constexpr int n = sizeof(Affine<F>) / 4;
  if (a.is_inf()) {
    for (int i = 0; i < n; i++) w[i] = 0;
    w[0] = 0x40;
    return;
  }
  put_be(a.x, w);
  put_be(a.y, w + n / 2);
}

// C(P), wasmcurves LEMtoC: big-endian plain x, 0x80 ORed into byte 0 when y is negative; infinity = 0x40 then zeros.
template <class F>
HD void c_encode(const Affine<F>& a, uint32_t* w) {
  constexpr int n = sizeof(Affine<F>) / 8;
  if (a.is_inf()) {
    for (int i = 0; i < n; i++) w[i] = 0;
    w[0] = 0x40;
    return;
  }
  put_be(a.x, w);
  if (y_negative(a.y)) w[0] |= 0x80;   // byte 0 is the low byte of the first little-endian word
}

template <class F>
struct UEncode {   // Exec op: point i of in -> words [i w, (i + 1) w) of out, w = sizeof(Affine<F>) / 4
  const Affine<F>* in;
  uint32_t* out;
  HD void operator()(uint64_t i) const {
    const Affine<F> a = in[i];   // a copy: the stores to out cannot alias it
    u_encode(a, out + i * (sizeof(Affine<F>) / 4));
  }
};

template <class F>
struct CEncode {   // Exec op: w = sizeof(Affine<F>) / 8
  const Affine<F>* in;
  uint32_t* out;
  HD void operator()(uint64_t i) const {
    const Affine<F> a = in[i];
    c_encode(a, out + i * (sizeof(Affine<F>) / 8));
  }
};

// ------------------------------------------------------------------------------------------------ chunked point hashing
enum class Enc { U, C };   // uncompressed (hashPubKey, the circuit hash, nextChallenge) or compressed (the response hash)

constexpr uint64_t kHashChunk = 1u << 16;     // points per conversion chunk

// BLAKE2b-512 over a stream of bytes and encoded points.  Points in the executor's memory are encoded by its ops; on the
// device in chunks, so the host BLAKE2b of chunk j (one sequential stream) overlaps the conversion and copy of chunk j + 1.
struct Hasher {
  Blake2b512 h;
  const Exec& ex;
  Enc enc;
  float kernel_ms = 0, blake_ms = 0;
  uint32_t* d_enc[2] = {nullptr, nullptr};
  uint8_t* h_enc[2] = {nullptr, nullptr};
  cudaEvent_t ev[6] = {};   // per buffer: kernel start, kernel end, copy done
  CudaResources res;

  explicit Hasher(const Exec& x, Enc e = Enc::U) : ex(x), enc(e) {
    if (ex.host()) return;
    for (int b = 0; b < 2; b++) {
      d_enc[b] = res.device<uint32_t>(kHashChunk * 32);
      h_enc[b] = res.pinned<uint8_t>(kHashChunk * 128);
    }
    for (auto& e : ev) e = res.event();
  }
  template <class F>
  static constexpr size_t enc_bytes(Enc e) { return e == Enc::U ? sizeof(Affine<F>) : sizeof(Affine<F>) / 2; }
  void update(const void* p, size_t n) {
    const auto t0 = std::chrono::steady_clock::now();
    h.update(p, n);
    blake_ms += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  void u32be(uint32_t v) {
    const uint8_t b[4] = {(uint8_t)(v >> 24), (uint8_t)(v >> 16), (uint8_t)(v >> 8), (uint8_t)v};
    update(b, 4);
  }
  // n points in host memory (the header points and other small arrays)
  template <class F>
  void points_host(const Affine<F>* p, uint64_t n) {
    const size_t w = enc_bytes<F>(enc) / 4;
    std::vector<uint32_t> buf(std::min<uint64_t>(n, 4096) * w);
    for (uint64_t i = 0; i < n; i += 4096) {
      const uint64_t m = std::min<uint64_t>(4096, n - i);
      for (uint64_t j = 0; j < m; j++) {
        Affine<F> a;
        memcpy(&a, p + i + j, sizeof a);
        if (enc == Enc::U) u_encode(a, buf.data() + j * w);
        else c_encode(a, buf.data() + j * w);
      }
      update(buf.data(), m * w * 4);
    }
  }
  template <class F>
  void encode(const Affine<F>* x, uint32_t* out, uint64_t n) {
    if (enc == Enc::U) ex.run<128>(n, UEncode<F>{x, out});
    else ex.run<128>(n, CEncode<F>{x, out});
  }
  // n points in the executor's memory.  On the device chunk j's host hash overlaps the conversion and copy of chunk j + 1.
  template <class F>
  void points(const Affine<F>* x, uint64_t n) {
    const size_t esz = enc_bytes<F>(enc);
    if (ex.host()) {
      std::vector<uint32_t> buf(n * esz / 4);
      encode(x, buf.data(), n);
      return update(buf.data(), n * esz);
    }
    const uint64_t nch = (n + kHashChunk - 1) / kHashChunk;
    for (uint64_t j = 0; j <= nch; j++) {
      if (j < nch) {
        const int b = j & 1;
        const uint64_t off = j * kHashChunk, m = std::min(kHashChunk, n - off);
        NZCP_CUDA(cudaEventRecord(ev[3 * b], 0));
        encode(x + off, d_enc[b], m);
        NZCP_CUDA(cudaEventRecord(ev[3 * b + 1], 0));
        NZCP_CUDA(cudaMemcpyAsync(h_enc[b], d_enc[b], m * esz, cudaMemcpyDeviceToHost, 0));
        NZCP_CUDA(cudaEventRecord(ev[3 * b + 2], 0));
      }
      if (j > 0) {
        const int b = (j - 1) & 1;
        const uint64_t m = std::min(kHashChunk, n - (j - 1) * kHashChunk);
        NZCP_CUDA(cudaEventSynchronize(ev[3 * b + 2]));
        float ms = 0;
        NZCP_CUDA(cudaEventElapsedTime(&ms, ev[3 * b], ev[3 * b + 1]));
        kernel_ms += ms;
        update(h_enc[b], m * esz);
      }
    }
  }
  // n points in host memory
  template <class F>
  void section(const uint8_t* p, uint64_t n) {
    if (n == 0) return;
    Exec staged(ex.host());   // freed when the section is hashed
    Affine<F>* x = staged.alloc<Affine<F>>(n);
    staged.upload(x, p, n * sizeof(Affine<F>));
    points(x, n);
  }
};

// ------------------------------------------------------------------------------------------------ phase-1 keys and records
constexpr size_t kPubKeyLen = 6 * 64 + 3 * 128;                               // 768
constexpr size_t kPartialLen = 216;
// pubkey tauG1 tauG2 alphaG1 betaG1 betaG2 partialHash nextChallenge type paramLength
constexpr size_t kPtauRecFixed = kPubKeyLen + 3 * 64 + 2 * 128 + kPartialLen + 64 + 4 + 4;   // 1504

// calculateFirstChallengeHash; blake_ms += the host time.  A caller that no longer needs the hash may set *cancel: the
// pass then stops within 1024 points and `out` is meaningless.
void first_challenge(uint32_t power, uint8_t out[64], float* blake_ms, const std::atomic<bool>* cancel = nullptr) {
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
    for (uint64_t i = 0; i < count && !(cancel && cancel->load(std::memory_order_relaxed)); i += kRep)
      h.update(r.data(), std::min<uint64_t>(kRep, count - i) * psz);
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

// ------------------------------------------------------------------------------------------------ verification
// `zkey verify` (verify.cu) and `powersoftau verify` (ptau_verify.cu): the library decides every check but the pairings and
// returns each pairing check before its first failure as a claim e(a, d) = e(b, c), for the caller to check in order.
struct Verdict {   // the first failed check the library decides
  int step, record;
  std::string msg;
};

// A record parse_records accepted: rec_fixed bytes ending in u32 type, u32 paramLength, then the parameters.
struct Rec {
  const uint8_t* p;
  uint32_t type, exp = 0;
  const uint8_t *name = nullptr, *beacon = nullptr;
  size_t name_len = 0, beacon_len = 0;
};

// kind: "zkey" or "ptau", for the message.
Rec read_record(const uint8_t* r, size_t rec_fixed, const char* kind) {
  Rec c{r, rd32u(r + rec_fixed - 8)};
  const uint8_t* q = r + rec_fixed;
  const uint8_t* end = q + rd32u(r + rec_fixed - 4);
  while (q < end) {   // parse_records has checked the layout
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
    throw ApiError(NZCP_E_FORMAT, std::string(kind) + ": beacon record without a beacon hash or with numIterationsExp > 63");
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

// The 32 bytes that seed the ChaCha of the random checks: the test seed, or OS randomness.  what: "zkey verify" / "ptau
// verify", for the message.
void verify_seed(const char* what, const uint8_t* seed, uint8_t out[32]) {
  if (seed) {
    memcpy(out, seed, 32);
    return;
  }
  for (size_t got = 0; got < 32;) {
    const ssize_t r = getrandom(out + got, 32 - got, 0);
    if (r <= 0) throw ApiError(NZCP_E_INTERNAL, std::string(what) + ": no OS randomness");
    got += (size_t)r;
  }
}

// ------------------------------------------------------------------------------------------------ MSM
constexpr uint64_t kMsmChunk = 1u << 22;   // bases per table-free MSM: the plan rejects windows x points >= 2^31

template <class F>
XYZZ<F> msm_finish(const MsmRun* r) {
  if constexpr (sizeof(F) == sizeof(Fq)) return msm_run_finish_g1(r);
  else return msm_run_finish_g2(r);
}

// out[b] = sum_i s_i P_b,i for k base arrays P_b (b < k) of n points against one vector of n plain scalars, all in the
// executor's memory.  On the device: the table-free MSM of msm_plan.cu in chunks of at most kMsmChunk bases, one bucket
// sort per chunk for all k runs, the chunk sums added.  On the host: host_msm_sim, the MSM kernels' code on the CPU.
template <class F>
void msm_sums(const Exec& ex, const Affine<F>* const* bases, int k, const Fr* scalars, uint64_t n, Affine<F>* out) {
  std::vector<XYZZ<F>> acc(k, XYZZ<F>::inf());
  for (uint64_t off = 0; off < n; off += kMsmChunk) {
    const uint64_t m = std::min(kMsmChunk, n - off);
    const int c = msm_pick_window_free(m);
    if (ex.host()) {
      for (int b = 0; b < k; b++)
        xyzz_add(acc[b], host_msm_sim<F>(reinterpret_cast<const uint8_t*>(bases[b] + off),
                                         reinterpret_cast<const uint8_t*>(scalars + off), m, c, msm_pick_rounds(m, c), 4));
      continue;
    }
    MsmSort sort;
    MsmRun run;
    msm_sort_create(&sort, m, c, -1, true);
    msm_run_create(&run, &sort, sizeof(F) != sizeof(Fq));
    msm_sort_launch(&sort, scalars + off, m, 0);
    for (int b = 0; b < k; b++) {
      MsmTable tab;
      msm_table_view(&tab, const_cast<Affine<F>*>(bases[b] + off), m, sizeof(F) != sizeof(Fq), c);
      msm_run_launch(&run, &sort, &tab, 0);
      NZCP_CUDA(cudaStreamSynchronize(0));
      if (b == 0) msm_sort_check(&sort);
      xyzz_add(acc[b], msm_finish<F>(&run));
    }
  }
  for (int b = 0; b < k; b++) out[b] = xyzz_to_affine(acc[b]);
}

template <class F>
Affine<F> msm_sum(const Exec& ex, const Affine<F>* bases, const Fr* scalars, uint64_t n) {
  Affine<F> r;
  msm_sums(ex, &bases, 1, scalars, n, &r);
  return r;
}

}  // namespace
}  // namespace nzcp
