/* libnzcp_prover.so -- C ABI of the B200-native Groth16 (BN254) prover for the NZCP circuit.
 *
 * This is the drop-in boundary for the one hot path of noway/nzcp-circom: snarkjs `groth16.prove(zkey, wtns)`
 * (and the `groth16.fullProve` wrapper around it).  The reference tree pins snarkjs ^0.4.12 in
 * /root/reference/package.json:12 (resolved 0.4.12 at yarn.lock:987-999; arithmetic in ffjavascript 0.2.48,
 * yarn.lock:408-416; WASM kernels in wasmcurves 0.1.0, yarn.lock:1132-1135); the artefacts these calls exchange are
 * the `.zkey` / `.wtns` files ignored at /root/reference/.gitignore:2-4.  A Node N-API addon (or Python ctypes,
 * see INTEGRATION.md) binds these entry points 1:1.
 *
 * What each entry point replaces.  The reference has NO call site for the prover (its tests stop at
 * `cir.calculateWitness(input, true)`, /root/reference/test/nzcp.js:39, and read the public signals as witness[1..513],
 * test/nzcp.js:41-48); the interface replaced is that of the pinned, un-vendored packages, cited here by the lock-file
 * line that pins each one:
 *   nzcp_zkey_load      binfileutils readBinFile + snarkjs zkey_utils.js readHeader + the readSection(4..9) calls of
 *                       groth16_prove.js (yarn.lock:385-388 @iden3/binfileutils 0.0.10; yarn.lock:987-999 snarkjs 0.4.12)
 *   nzcp_prove*         snarkjs groth16_prove.js groth16Prove(zkeyFileName, witnessFileName) incl. wtns_utils.js
 *                       readHeader and the three error checks (yarn.lock:987-999)
 *   nzcp_prove_batch    no snarkjs equivalent (one proof per call there); BASELINE.json configs[2] batch mode
 *   nzcp_ntt[_coset]    ffjavascript engine_fft.js Fr.fft / Fr.ifft, engine_applykey.js batchApplyKey (yarn.lock:408-416)
 *   nzcp_msm, nzcp_msm_var, nzcp_msm_plan_*
 *                       ffjavascript engine_multiexp.js G1/G2.multiExpAffine (yarn.lock:408-416) over wasmcurves
 *                       build_multiexp.js (yarn.lock:1132-1135); the *_partial / sum_partials pair is the per-rank half of
 *                       the split MSM of BASELINE.json configs[4]
 *   nzcp_zkey_selfcheck no snarkjs equivalent: the format facts of SURVEY.md 8c-3, for the first real key
 *   nzcp_ptau_prepare*  snarkjs powersoftau_preparephase2.js preparePhase2(oldPtauFilename, newPTauFilename) and the group
 *                       ifft of ffjavascript engine_fft.js it runs per level (yarn.lock:987-999, 408-416)
 *   nzcp_ptau_new*, nzcp_ptau_contribute*, nzcp_ptau_beacon
 *                       snarkjs powersoftau_new.js newAccumulator, powersoftau_contribute.js contribute and
 *                       powersoftau_beacon.js beacon, with keypair.js createPTauKey (yarn.lock:987-999)
 *   nzcp_zkey_contribute*, nzcp_zkey_beacon
 *                       snarkjs zkey_contribute.js phase2contribute and zkey_beacon.js beacon, with the ChaCha of
 *                       ffjavascript random.js (yarn.lock:987-999, 408-416)
 *   nzcp_zkey_circuit_hash, nzcp_zkey_verify*
 *                       snarkjs zkey_new.js's circuit hash, zkey_verify_fromr1cs.js verifyFromR1cs and
 *                       zkey_verify_frominit.js verifyFromInit (yarn.lock:987-999); the pairings stay with the caller
 *   nzcp_field_op       wasmcurves build_f1m.js f1m_mul / f1m_add / f1m_sub (yarn.lock:1132-1135)
 *   nzcp_synth_*        snarkjs zkey_new.js with a known tau in place of the ptau file /root/reference/Makefile:31 names;
 *                       shapes from circuits/nzcp_exampleTest.circom:4 and circuits/nzcp_liveTest.circom:4
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative NZCP_E_* code and
 * never throws across the boundary; `nzcp_last_error()` returns a thread-local message for the last failure.
 * All field elements crossing the ABI are 32-byte little-endian integers.  A handle may be used by one thread at a
 * time; the library owns all device memory.  There is NO CPU fallback: without a CUDA device every compute entry
 * point fails with NZCP_E_CUDA.
 */
#ifndef NZCP_PROVER_H
#define NZCP_PROVER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NZCP_OK 0
#define NZCP_E_ARG (-1)        /* null pointer / bad size / bad option */
#define NZCP_E_FORMAT (-2)     /* malformed .zkey / .wtns container */
#define NZCP_E_NOT_GROTH16 (-3)/* snarkjs: "zkey file is not groth16" */
#define NZCP_E_CURVE (-4)      /* snarkjs: "Curve of the witness does not match the curve of the proving key" */
#define NZCP_E_WITNESS_LEN (-5)/* snarkjs: "Invalid witness length. Circuit: X, witness: Y" */
#define NZCP_E_CUDA (-6)       /* CUDA runtime failure (incl. no device) */
#define NZCP_E_RANGE (-7)      /* a witness value is not a canonical field element */
#define NZCP_E_INTERNAL (-8)

typedef struct nzcp_zkey nzcp_zkey;     /* proving key resident on one GPU (replaces the per-call readSection()s of */
                                        /* snarkjs groth16_prove.js: sections 4-9 are parsed and uploaded once)     */
typedef struct nzcp_prover nzcp_prover; /* per-stream work buffers for one in-flight proof                          */

/* zkey section 2 header as snarkjs zkey_utils.js readHeader() returns it (coordinates plain, not Montgomery). */
typedef struct nzcp_zkey_info {
  uint32_t n_vars;
  uint32_t n_public;
  uint32_t domain_size;
  uint32_t power;
  uint64_t n_coefs;
  uint8_t alpha1[64], beta1[64], delta1[64];     /* G1: x, y                      */
  uint8_t beta2[128], gamma2[128], delta2[128];  /* G2: x.c0, x.c1, y.c0, y.c1    */
  uint64_t device_bytes;
} nzcp_zkey_info;

/* The proof: 8 plain 32-byte LE values  A.x A.y | B.x.c0 B.x.c1 B.y.c0 B.y.c1 | C.x C.y
 * (snarkjs proof.pi_a / pi_b / pi_c before stringification; a point at infinity is all zero). */
typedef struct nzcp_proof {
  uint8_t pi_a[64];
  uint8_t pi_b[128];
  uint8_t pi_c[64];
} nzcp_proof;

/* Intermediate results the parity tests compare bit-for-bit against the oracle (north_star: "H coefficients, each
 * MSM result and the final proof").  Affine, plain, same coordinate order as nzcp_proof. */
typedef struct nzcp_prove_debug {
  uint8_t msm_a[64];
  uint8_t msm_b1[64];
  uint8_t msm_b2[128];
  uint8_t msm_c[64];
  uint8_t msm_h[64];
  uint8_t* h_scalars;      /* optional: caller buffer of domain_size*32 bytes receiving the joinABC output, or NULL */
  float stage_ms[8];       /* device time: 0 upload, 1 r1cs eval, 2 ntt pipeline+join, 3 msm A, 4 msm B1, 5 msm B2, */
                           /*              6 msm C, 7 msm H (bucket sort of h included)                             */
  float sort_ms[2];        /* bucket sort of the witness (shared by A, B1, B2, C) / of the h scalars                */
  float accumulate_ms[5];  /* the bucket-accumulate kernel alone (CUDA events on its stream): A, B1, B2, C, H       */
  uint32_t n_entries[2];   /* non-zero signed digits (= mixed additions per MSM): witness, h                        */
  float total_ms;          /* first event to end of the H MSM on the main stream                                    */
} nzcp_prove_debug;

const char* nzcp_last_error(void);
int nzcp_device_count(void);

/* Parse a snarkjs .zkey held in host memory and upload it to `device`.  Caller keeps ownership of `bytes`. */
int nzcp_zkey_load(const uint8_t* bytes, size_t len, int device, nzcp_zkey** out);
int nzcp_zkey_info_get(const nzcp_zkey* zk, nzcp_zkey_info* info);
void nzcp_zkey_free(nzcp_zkey* zk);

/* Format self-checks on a .zkey image (SURVEY.md 8c-3) -- what a snarkjs-made Groth16 key must satisfy, checked without a
 * reference implementation: moduli, section sizes, canonical coefficient values, the nPublic+1 appended public-input rows
 * (value R^2 mod r: pins the "coef * R^2" convention of section 4), and every base point of sections 3, 5-9 and of the header
 * on its curve.  The point checks run on `device`.  Returns NZCP_OK when the file could be examined; the verdict is
 * report->ok. */
typedef struct nzcp_zkey_check {
  uint32_t n_vars, n_public, domain_size;
  uint32_t n_constraints;      /* constraint index of the first appended public-input row */
  uint64_t n_coefs;
  uint64_t bad_coef_values;    /* section 4 values >= r */
  uint64_t bad_coef_indices;   /* records with matrix > 1, constraint >= domainSize or signal >= nVars */
  uint64_t off_curve[6];       /* per section A(5), B1(6), B2(7), C(8), H(9), IC(3): points off the curve / non-canonical */
  uint64_t infinity[6];        /* per section: (0,0) infinity markers (informational) */
  uint32_t header_moduli_ok;   /* q, r are the BN254 moduli */
  uint32_t header_points_ok;   /* alpha1, beta1, delta1 on G1, beta2, gamma2, delta2 on the twist, none at infinity */
  uint32_t public_rows_ok;     /* last nPublic+1 coefficient records = (A, nConstraints+i, i, R^2 mod r) */
  uint32_t ok;                 /* every check passed */
} nzcp_zkey_check;
int nzcp_zkey_selfcheck(const uint8_t* bytes, size_t len, int device, nzcp_zkey_check* report);

/* snarkjs `zkey new` (zkey_new.js newZKey(r1csName, ptauName, zkeyName)): the circuit-specific Groth16 key from an .r1cs
 * (circom --r1cs, /root/reference/Makefile:5-9) and a PREPARED powers-of-tau file (sections 12-15 present;
 * /root/reference/Makefile:31 names powersOfTau28_hez_final_22.ptau).  gamma = delta = 1 as after `zkey new`; section 10
 * (circuit hash) is written zero-filled -- see csrc/setup.cu.  Errors carry snarkjs's messages ("Powers of tau is not
 * prepared.", "circuit too big for this power of tau ceremony. ...", "r1cs curve does not match powers of tau ceremony
 * curve").  The sparse point combinations run on `device`. */
int nzcp_zkey_new_size(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, size_t* out_size);
int nzcp_zkey_new(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, int device, uint8_t* out,
                  size_t cap, size_t* written);

/* snarkjs `powersoftau prepare phase2` (powersoftau_preparephase2.js preparePhase2(oldPtau, newPtau)): the file `zkey new`
 * needs from the output of a phase-1 ceremony.  Sections 2-7 are copied, the header gets ceremonyPower = power, and the
 * Lagrange-basis sections 12 (from tauG1, levels 0 .. power+1), 13 (tauG2), 14 (alphaTauG1) and 15 (betaTauG1) (levels
 * 0 .. power) are computed by an inverse FFT over curve points on `device`; sections 12-15 already in the input are
 * ignored.  As in snarkjs, the top tauG1 level takes the point at infinity for the tauG1 power the file lacks (see
 * csrc/ptau.cu).  Output: 11 sections in the order 1-7, 12-15.
 * Both functions reject before any device work: a file that is not a ptau (NZCP_E_FORMAT) or not over bn128
 * (NZCP_E_CURVE); power outside 1..27 (NZCP_E_FORMAT; power 28 needs snarkjs's coset branch and is NZCP_E_ARG); a missing
 * section 2-7 ("Missing section N") or a section 2-6 whose size does not match the power (NZCP_E_FORMAT); an input point
 * with a coordinate >= q or off its curve (NZCP_E_RANGE).  nzcp_ptau_prepare_size is host-only.
 * section_ms (optional): device time of output sections 12, 13, 14, 15. */
int nzcp_ptau_prepare_size(const uint8_t* ptau, size_t len, size_t* out_size);
int nzcp_ptau_prepare(const uint8_t* ptau, size_t len, int device, uint8_t* out, size_t cap, size_t* written,
                      float section_ms[4]);

/* snarkjs `powersoftau new` (powersoftau_new.js newAccumulator): a fresh phase-1 file of 2^power, power 1..28 (else
 * NZCP_E_ARG): header (n8, q, power, ceremonyPower = power), sections 2-6 the G1 / G2 generators (tau = alpha = beta = 1),
 * section 7 no contributions.  Host only.  `hash` (optional, NULL: skipped; it costs a BLAKE2b pass over ~384 * 2^power
 * bytes) receives the first challenge hash, snarkjs's "First Contribution Hash".  nzcp_ptau_new_size gives the file size. */
int nzcp_ptau_new_size(uint32_t power, size_t* out_size);
int nzcp_ptau_new(uint32_t power, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]);

/* snarkjs `powersoftau contribute` / `powersoftau beacon` (powersoftau_contribute.js contribute, powersoftau_beacon.js
 * beacon): one phase-1 contribution (tau, alpha, beta) drawn by keypair.js createPTauKey from the rng and the challenge
 * (the last record's nextChallenge, or the first challenge hash).  Point i of sections 2 (tauG1), 3 (tauG2), 4 (alphaTauG1),
 * 5 (betaTauG1) and 6 (betaG2) becomes (first * tau^i) * P_i with first = 1, 1, alpha, beta, beta, on `device`; section 7
 * gets a new record after the earlier ones (type 0 contribute, 1 beacon; parameters as nzcp_zkey_contribute).  Output:
 * sections 1-7 in id order, header rewritten with ceremonyPower = power; sections 12-15 of a prepared input are dropped.
 * `hash` receives the 64-byte response hash snarkjs returns.  The rng is that of nzcp_zkey_contribute / nzcp_zkey_beacon
 * (`seed`: 32 bytes, test hook, NULL in use).  See csrc/ptau_contribute.cu for the restated algorithm.
 * All functions reject before any device work: a file that is not a ptau or has no header (NZCP_E_FORMAT); not over bn128
 * (NZCP_E_CURVE); power outside 1..28, a missing section 2-7 ("Missing section N"), a section 2-6 whose size does not match
 * the power, a section 7 that is truncated, has trailing bytes, unsorted or unknown parameters (NZCP_E_FORMAT); power !=
 * ceremonyPower (NZCP_E_ARG, "This file has been reduced. You cannot contribute into a reduced file."); an input point with
 * a coordinate >= q or off its curve (NZCP_E_RANGE); a name longer than 64 bytes, a beacon hash of 0 or >= 256 bytes or
 * num_iterations_exp outside 10..63 (NZCP_E_ARG, as nzcp_zkey_contribute).  nzcp_ptau_contribute_size is host-only.
 * ms (optional): [0]-[4] key-kernel device time of sections 2-6, [5] encode-kernel device time, [6] host BLAKE2b time. */
int nzcp_ptau_contribute_size(const uint8_t* ptau, size_t len, const char* name, size_t beacon_hash_len, size_t* out_size);
int nzcp_ptau_contribute(const uint8_t* ptau, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                         const uint8_t* seed, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                         float ms[7]);
int nzcp_ptau_beacon(const uint8_t* ptau, size_t len, const char* name, const uint8_t* beacon_hash, size_t beacon_hash_len,
                     uint32_t num_iterations_exp, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                     float ms[7]);

/* snarkjs `zkey contribute` / `zkey beacon` (zkey_contribute.js phase2contribute, zkey_beacon.js beacon): one phase-2
 * contribution k to a Groth16 key.  delta1 and delta2 of the header become k * delta, every point of sections 8 (L) and 9
 * (H) becomes k^-1 * P on `device`, sections 1 and 3-7 are copied, and section 10 gets a new record after the earlier
 * ones (type 0 contribute, 1 beacon; parameter tag 1 = name if name is non-empty, tags 2 / 3 = num_iterations_exp /
 * beacon hash).  Output: 10 sections in the order 1..10.  `hash` receives the 64-byte contribution hash snarkjs prints.
 * contribute: k comes from ffjavascript's ChaCha seeded by BLAKE2b-512(64 OS-random bytes || entropy); `seed` (32 bytes,
 * test hook; NULL in use) seeds the ChaCha directly instead.  beacon: from SHA-256 iterated 2^num_iterations_exp times
 * over beacon_hash.  See csrc/contribute.cu for the restated algorithm.
 * All functions reject before any device work: a file that is not a zkey or has no header (NZCP_E_FORMAT); protocol != 1
 * (NZCP_E_NOT_GROTH16); moduli other than bn128's (NZCP_E_CURVE); section 2 not 660 bytes, a missing section 2-10
 * ("Missing section N"), a section 8 / 9 size that does not match nVars - nPublic - 1 / domainSize, a section 10 that is
 * truncated, has trailing bytes, unsorted ("Parameters in the contribution must be sorted") or unknown ("Parameter not
 * recognized") parameters (NZCP_E_FORMAT); a point of sections 8 / 9 or the header delta1 / delta2 with a coordinate >= q
 * or off its curve (NZCP_E_RANGE); a name longer than 64 bytes (NZCP_E_ARG; snarkjs would cut it at 64 characters); a
 * beacon hash of 0 or >= 256 bytes or num_iterations_exp outside 10..63 (NZCP_E_ARG, snarkjs's messages).
 * nzcp_zkey_contribute_size is host-only; beacon_hash_len = 0 sizes a contribute record.
 * section_ms (optional): device time of sections 8 and 9. */
int nzcp_zkey_contribute_size(const uint8_t* zkey, size_t len, const char* name, size_t beacon_hash_len, size_t* out_size);
int nzcp_zkey_contribute(const uint8_t* zkey, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                         const uint8_t* seed, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                         float section_ms[2]);
int nzcp_zkey_beacon(const uint8_t* zkey, size_t len, const char* name, const uint8_t* beacon_hash, size_t beacon_hash_len,
                     uint32_t num_iterations_exp, int device, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64],
                     float section_ms[2]);

/* snarkjs `zkey verify` (zkey_verify_fromr1cs.js verifyFromR1cs, zkey_verify_frominit.js verifyFromInit) and the circuit
 * hash of zkey_new.js (csrc/verify.cu restates both).
 * nzcp_zkey_circuit_hash: the csHash snarkjs's newZKey writes into section 10, from an initial key (`zkey new` output) and
 * the prepared ptau it was made from; ms (optional): [0] device time of the hash kernels, [1] host BLAKE2b time.
 * nzcp_zkey_verify_from_init checks `zkey` against the initial key `init`; nzcp_zkey_verify_from_r1cs first builds the
 * initial key from the .r1cs and the ptau (nzcp_zkey_new in host memory, with its circuit hash).
 * The verdict is split: the pairings are left to the caller.  The library decides every other check in snarkjs's order and
 * stops at the first that fails (report->failed_step != 0, report->message).  Each pairing check before that point is
 * returned as a claim e(a, d) = e(b, c), in order.  The verdict is the first false claim, else the library's failure, else
 * true (nzcp_circom_b200/verifier.py checks the claims, as groth16.verify does).  The C ABI alone does not give it.
 * Steps (failed_step and claim.step): 1 a point of the key's header, section 10 records or sections 8 / 9 that is not
 * canonical and on its curve, or delta2 / a g2_spx outside the order-r subgroup (snarkjs checks none of this); 2 "INVALID(i):
 * Inconsistent transcript"; 3 claim "INVALID(i): public key G1 and G2 do not have the same ration"; 4 claim "INVALID(i):
 * deltaAfter does not fillow the public key"; 5 "INVALID(i): Key of the beacon does not match. g1_s" / "... g1_sx"; 6
 * "Different circuit parameters"; 7 "Invalid alpha1" / beta1 / beta2 / gamma2 / delta1; 8 claim "Invalid delta2"; 9
 * "Circuit does not match"; 10 "IC" / "Coeffs" / "A" / "B1" / "B2" " section is not identical"; 11 claim "L section does not
 * match"; 12 claim "H section does not match".  (snarkjs's spellings.)
 * Deviation: the L check draws full-width scalars (snarkjs: 32-bit).  seed (32 bytes, test hook; NULL in use) replaces the
 * OS randomness that seeds the L and H scalars.
 * Errors (before any device work): the zkey / ptau / r1cs rejections of nzcp_zkey_contribute and nzcp_zkey_new, a beacon
 * record without its parameters, an initial key whose sections 3 / 5-7 do not match its header or whose domainSize is not
 * a power of two, and cirPower = power with N > 2^14, where snarkjs's hashHPoints reads past ptau section 2 (NZCP_E_ARG).
 * nzcp_zkey_verify_size (host-only) gives the claim and record counts the buffers must hold (2 n + 3 and n).
 * section_ms (optional): [0] device time of the hash kernels, [1] host BLAKE2b of the circuit hash, [2] the L MSMs,
 * [3] the H scalar transform, NTT and MSMs. */
typedef struct nzcp_zkey_verify_claim {
  int32_t step, record;      /* record: section-10 index for steps 3 and 4, else -1 */
  uint8_t a[64], b[64];      /* G1, plain x, y (all zero = infinity) */
  uint8_t c[128], d[128];    /* G2, plain x.c0 x.c1 y.c0 y.c1 */
} nzcp_zkey_verify_claim;
typedef struct nzcp_zkey_contribution {
  uint8_t hash[64];          /* BLAKE2b-512(hashPubKey(record)): the contribution hash snarkjs prints */
  uint32_t type;             /* 0 contribute, 1 beacon */
  uint32_t num_iterations_exp, name_len, beacon_hash_len;
  char name[256];            /* parameter tag 1, not NUL-terminated */
  uint8_t beacon_hash[256];  /* parameter tag 3 */
} nzcp_zkey_contribution;
typedef struct nzcp_zkey_verify_report {
  int32_t failed_step;       /* 0: every check the library decides passed */
  int32_t failed_record;     /* section-10 index for steps 2 and 5, else -1 */
  char message[256];
  uint32_t n_contributions, n_claims;
  uint8_t cs_hash[64];       /* the circuit hash computed from the initial key and the ptau */
} nzcp_zkey_verify_report;
int nzcp_zkey_circuit_hash(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, int device,
                           uint8_t hash[64], float ms[2]);
int nzcp_zkey_verify_size(const uint8_t* zkey, size_t len, size_t* n_claims, size_t* n_records);
int nzcp_zkey_verify_from_init(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, const uint8_t* zkey,
                               size_t zkey_len, const uint8_t* seed, int device, nzcp_zkey_verify_claim* claims,
                               size_t claims_cap, nzcp_zkey_contribution* records, size_t records_cap,
                               nzcp_zkey_verify_report* report, float section_ms[4]);
int nzcp_zkey_verify_from_r1cs(const uint8_t* r1cs, size_t r1cs_len, const uint8_t* ptau, size_t ptau_len, const uint8_t* zkey,
                               size_t zkey_len, const uint8_t* seed, int device, nzcp_zkey_verify_claim* claims,
                               size_t claims_cap, nzcp_zkey_contribution* records, size_t records_cap,
                               nzcp_zkey_verify_report* report, float section_ms[4]);

/* Work buffers + streams for proofs against `zk`.  Several provers may share one zkey (one per host thread). */
int nzcp_prover_create(nzcp_zkey* zk, nzcp_prover** out);   /* = mode 0 */
/* mode 0 = latency (one proof at a time), mode 1 = throughput (meant to run beside other provers on the same GPU;
 * nzcp_prove_batch uses these).  Same proofs, bit for bit, in both modes; today both run the same kernels (batched-affine
 * pair rounds on every large MSM, ~6 GB of scratch per prover at the NZCP size) -- the distinction is kept in the ABI so
 * that a caller states its use. */
int nzcp_prover_create_mode(nzcp_zkey* zk, int mode, nzcp_prover** out);
void nzcp_prover_free(nzcp_prover* p);

/* groth16.prove: `wtns` is a complete .wtns file image.  r, s: 32-byte LE blinding scalars (< r); NULL draws them
 * from the OS CSPRNG as snarkjs's Fr.random() does.  `dbg` may be NULL. */
int nzcp_prove(nzcp_prover* p, const uint8_t* wtns, size_t wtns_len, const uint8_t* r, const uint8_t* s,
               nzcp_proof* proof, nzcp_prove_debug* dbg);
/* Throughput mode (SURVEY.md 8e batch mode on one GPU): n_proofs independent .wtns images against one resident key, proved by
 * `n_provers` host threads (0 = 3), each with its own prover (stream set + work buffers, kept in the key between calls), so
 * that the latency-bound tail of one proof overlaps the multiplier-bound kernels of the next.  r, s: n_proofs x 32 bytes or
 * NULL (random).  status (optional): per-proof return code.  Returns the first failure's code, or NZCP_OK. */
int nzcp_prove_batch(nzcp_zkey* zk, const uint8_t* const* wtns, const size_t* wtns_len, size_t n_proofs, const uint8_t* r,
                     const uint8_t* s, nzcp_proof* proofs, int n_provers, int* status);
/* Same, but the witness is a bare array of n_vars 32-byte LE values (section 2 of a .wtns). */
int nzcp_prove_witness(nzcp_prover* p, const uint8_t* witness, uint32_t n_witness, const uint8_t* r, const uint8_t* s,
                       nzcp_proof* proof, nzcp_prove_debug* dbg);
/* Device-resident variant used for kernel-only timing: witness already in HBM (device pointer, n_vars * 32 B). */
int nzcp_prove_device(nzcp_prover* p, const void* d_witness, const uint8_t* r, const uint8_t* s, nzcp_proof* proof,
                      nzcp_prove_debug* dbg);
/* Device pointer of the prover's own witness buffer (n_vars * 32 B), for callers that fill it themselves. */
void* nzcp_prover_witness_buffer(nzcp_prover* p);
/* Number of kernel launches issued for this prover so far (NULL: by the whole process). */
uint64_t nzcp_prover_launch_count(const nzcp_prover* p);

/* ---- standalone kernels (BASELINE config 4: NTT + MSM sweeps; also the fine-grained parity tests) ---- */
/* Natural-order NTT / iNTT over Fr of 2^log_n Montgomery-form elements in host memory (snarkjs Fr.fft / Fr.ifft). */
int nzcp_ntt(uint8_t* data, int log_n, int inverse, int device, float* kernel_ms);
/* The prover's H pipeline on `batch` polynomials: evaluations on the subgroup -> evaluations on the odd coset. */
int nzcp_ntt_coset(uint8_t* data, int log_n, int batch, int device, float* kernel_ms);
/* MSM over G1 (g2 = 0, 64-byte bases) or G2 (g2 = 1, 128-byte bases): Montgomery affine bases as in the zkey, plain
 * scalars.  window_bits = 0 picks the default.  out = plain affine point (64 / 128 bytes). */
int nzcp_msm(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int device,
             uint8_t* out, float* kernel_ms);
/* MSM plans: a base set made resident once, any number of scalar vectors against it (csrc/msm_plan.cu).
 *   mode 0  fixed-base: the bases are expanded into the 2^(c w) window table once (what nzcp_zkey_load does per section)
 *   mode 1  variable-base: no table -- ffjavascript multiExpAffine's contract (arbitrary bases per call) at one pass over them
 * build_ms (optional) = host wall time of the upload + table build.  Scalars are host buffers of n_scalars <= n_points
 * plain 32-byte values. */
typedef struct nzcp_msm_plan nzcp_msm_plan;
int nzcp_msm_plan_create(const uint8_t* bases, size_t n_points, int g2, int window_bits, int mode, int device,
                         nzcp_msm_plan** out, float* build_ms);
void nzcp_msm_plan_free(nzcp_msm_plan* p);
int nzcp_msm_plan_run(nzcp_msm_plan* p, const uint8_t* scalars, size_t n_scalars, uint8_t* out, float* kernel_ms);
/* Device time of the bucket accumulation alone (pair rounds + XYZZ kernel) in the plan's last run. */
int nzcp_msm_plan_accumulate_ms(const nzcp_msm_plan* p, float* ms);
/* Split MSM (BASELINE.json configs[4]; SURVEY.md 8e-2): the result stays in HBM as ONE extended-Jacobian point (x, y, zz,
 * zzz Montgomery: 128 B for G1, 256 B for G2) written to the device pointer d_out, e.g. this rank's slot of an NCCL
 * all-gather buffer.  nzcp_msm_sum_partials then adds `count` such points on the GPU and returns the plain affine sum. */
int nzcp_msm_plan_run_partial(nzcp_msm_plan* p, const uint8_t* scalars, size_t n_scalars, void* d_out, float* kernel_ms);
int nzcp_msm_sum_partials(const void* d_partials, size_t count, int g2, int device, uint8_t* out);
/* One-shot variable-base MSM.  ms (optional): [0] host wall time of the whole call incl. uploads, [1] kernel time. */
int nzcp_msm_var(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int device,
                 uint8_t* out, float ms[2]);
/* Device self-test of the field / curve arithmetic against the host build of the same code; returns the number of
 * mismatches in *n_bad (0 = pass). */
int nzcp_selftest(int device, uint64_t seed, uint32_t n_cases, uint32_t* n_bad);
/* Element-wise Fr/Fq ops on the device, for limb-exact parity tests: op 0 mul, 1 add, 2 sub (3..5: the portable code paths), 6 inverse by division steps, 7 Fermat inverse (Montgomery-form in/out),
 * field 0 = Fr, 1 = Fq. */
int nzcp_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int device);
/* Device Fq / Fq2 arithmetic on n little-endian records, one thread per record, through the functions the kernels call.
 * Fq2 = c0 | c1.  op (input / output bytes per record):
 *   0 fp_mul_wide: a | b -> 512-bit a * b (64 / 64); a, b < 2^255
 *   1 fp_redc_wide<Fq>: T -> T / 2^256 mod q (64 / 32); T < q * 2^256
 *   2 f_mulsub(Fq), the lazy-reduction body, and 3 its eager form fp_sub(fp_mul, fp_mul): a | b | c | d -> a b - c d (128 / 32)
 *   4 f_mul(Fq2) as the kernels call it, 5 f2_mul_inline: a | b -> a b (128 / 64)
 *   6 f_sqr(Fq2) (64 / 64), 7 f_inv(Fq2) Fermat (64 / 64), 8 f_inv_fast(Fq2) division steps (64 / 64)
 *   9 f_mulsub(Fq2): a | b | c | d -> a b - c d (256 / 64)
 * Ops 2-9 take and return Montgomery form.  Ops 0 and 1 reject inputs outside their domain with NZCP_E_ARG. */
int nzcp_arith_op(int op, const uint8_t* in, uint8_t* out, size_t n, int device);
/* Device XYZZ group law on n records (x, y, zz, zzz Montgomery, as nzcp_msm_plan_run_partial writes them: 128 B for G1,
 * 256 B for G2; zz == 0 is infinity).  op: 0 xyzz_add(a, b), b XYZZ; 1 xyzz_madd(a, b), b affine in the zkey layout;
 * 2 xyzz_madd(a, -b); 3 xyzz_dbl(a), b unused; 4 xyzz_to_affine(a) -> affine records.  Ops 0-3 write XYZZ records.
 * A madd operand equal to (0, 0) is rejected with NZCP_E_ARG. */
int nzcp_curve_op(int g2, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int device);

/* Tuning knobs for experiments and tests (process-wide, read when a plan is created / a run is launched):
 *   "msm_rounds"  batched-affine pair rounds per MSM: -1 = automatic (by size), 0..3 forced
 *   "prover_rounds_w" / "prover_rounds_h"  the same for a prover's witness MSMs / H MSM (read by nzcp_prover_create)
 *   "pair_k1" / "pair_k2" / "pair_k3"  additions per thread in round 1 / 2 / 3: 4, 8, 16 or 32
 *   "pair_prefetch_fwd" / "pair_prefetch_bwd"  operand prefetch in the pair-round kernels: 0 = none (default), 1 = L1, 2 = L2
 *   "pair_stage"  1 = round 1's forward pass stages the operands it gathered and the backward pass streams them (set it before
 *                 the prover / plan is created); 0 (default) = the backward pass gathers them from the window table again
 *   "sort_threads"  threads per block of the bucket sort's shared-memory histogram passes: 1024 (default), 512, 256, 128
 *   "gather_hint"  experiment: 1 = the round-1 table gathers carry the PTX .L2::64B fetch-size qualifier (default 0)
 *   "acc_prefetch"  1 (default) = the XYZZ accumulate kernel prefetches its next table point to L1, 0 = no prefetch
 *   "stage_mode"  host witness upload in nzcp_prove*: -1 = automatic (pageable memory through the prover's pinned staging
 *                 buffer in chunks, caller-pinned memory directly), 0 = always direct, 1 = always staged
 *   "stage_chunk_kb"  staging chunk size in KiB (default 1024)
 *   "prover_rounds_b2"  pair rounds of the G2 MSM alone (-1 = as the other witness MSMs; another value gives it its own sort)
 *   "prover_c_h" / "prover_c_w"  window bits of the H / witness MSM tables, read by nzcp_zkey_load (0 = default: 16 at 2^20)
 *   "ntt_tma"     1 (default) = TMA-staged low NTT pass (bulk copies + mbarrier, twiddles in shared memory), 0 = thread-loaded
 *   "stage_threads"   host threads sharing the copy into the staging buffer (default 4; 1 = the calling thread alone) */
int nzcp_tuning_set(const char* name, int value);

/* Integer-pipe microbenchmark (the MSM / NTT roofline denominator): out[0] = IMAD.WIDE.U32 (32x32->64 multiply-add) per
 * second, out[1] = 32-bit IMAD per second, out[2] = dependent-chain Fq Montgomery products per second, out[3] = SM count. */
int nzcp_intpipe_bench(int device, int iters, double out[4]);
/* Diagnostic: rates of the carry-chain variants (modes 0..8 of csrc/standalone.cu intpipe_kernel), out[9] = SM count. */
int nzcp_intpipe_modes(int device, int iters, double out[10]);
/* Diagnostic: which instructions issue beside IMAD.WIDE (csrc/standalone.cu pipeprobe_kernel).  out[0] = DFMA/s alone;
 * out[1..3] = IMAD.WIDE/s with DFMA (1:1), xor (1:2), carry-free add (1:2) issued beside it; out[4] = DFMA/s in probe 1. */
int nzcp_pipe_probe(int device, int iters, double out[5]);

/* ---- host hooks: the library's __host__ __device__ arithmetic compiled for the CPU (what the O(1) host glue runs).
 * Test-only; they let the no-GPU suite pin that code against the oracle.  op: 0 mul, 1 add, 2 sub, 3 inverse by
 * division steps (fp_inv_fast; b ignored), 4 inverse by the Fermat ladder. */
int nzcp_host_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
/* k * base (Montgomery affine base as in the zkey, NULL = the group generator); out = plain affine. */
int nzcp_host_scalar_mul(int g2, const uint8_t* base_mont, const uint8_t* scalar, uint8_t* out_plain);
/* The MSM data path INCLUDING the batched-affine pair rounds of csrc/msm_pair.cuh, executed on the CPU with the same
 * __host__ __device__ code the kernels run (rounds = 0..3 pair rounds, adds_per_thread = 4, 8, 16 or 32).  Lets the
 * no-GPU suite check the rounds' index arithmetic and special-pair handling against the oracle.  out = plain affine. */
int nzcp_host_msm_sim(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int rounds,
                      int adds_per_thread, uint8_t* out);
/* Fr.w[k] of ffjavascript (plain form). */
int nzcp_host_root_of_unity(int k, uint8_t* out_plain);
/* nzcp_ptau_prepare with the kernels' load, stage indexing and butterflies run one thread after the other on the CPU,
 * for power <= 4 (larger powers: NZCP_E_ARG).  Same validation, same output bytes. */
int nzcp_host_ptau_prepare(const uint8_t* ptau, size_t len, uint8_t* out, size_t cap, size_t* written);

/* nzcp_zkey_contribute (beacon_hash == NULL) or nzcp_zkey_beacon with the kernel's per-point code run on the CPU, for
 * sections 8 + 9 of at most 4096 points (more: NZCP_E_ARG).  Same validation, same output bytes and hash. */
int nzcp_host_zkey_contribute(const uint8_t* zkey, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                              const uint8_t* seed, const uint8_t* beacon_hash, size_t beacon_hash_len,
                              uint32_t num_iterations_exp, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]);

/* nzcp_ptau_contribute (beacon_hash == NULL) or nzcp_ptau_beacon with the kernels' per-point code (key, encodings) run
 * on the CPU, for power <= 4 (more: NZCP_E_ARG).  Same validation, same output bytes and hash. */
int nzcp_host_ptau_contribute(const uint8_t* ptau, size_t len, const char* name, const uint8_t* entropy, size_t entropy_len,
                              const uint8_t* seed, const uint8_t* beacon_hash, size_t beacon_hash_len,
                              uint32_t num_iterations_exp, uint8_t* out, size_t cap, size_t* written, uint8_t hash[64]);

/* nzcp_zkey_circuit_hash with the kernels' per-point code (H differences, point encoding) run on the CPU, for a domain of
 * at most 4096 (more: NZCP_E_ARG).  Same validation, same hash. */
int nzcp_host_zkey_circuit_hash(const uint8_t* init, size_t init_len, const uint8_t* ptau, size_t ptau_len, uint8_t hash[64]);

/* ---- synthetic circuits of the NZCP shape (no circom / snarkjs in this environment; SURVEY.md 8d) ---- */
typedef struct nzcp_synth nzcp_synth;
/* n_points pseudo-random group elements k_i * G (Montgomery affine, 64 / 128 B each) into a host buffer -- bases for the
 * standalone MSM sweeps.  Computed on `device` by the fixed-base kernel. */
int nzcp_synth_points(uint64_t seed, size_t n_points, int g2, int device, uint8_t* out);
/* Random forward-solvable R1CS: n_constraints constraints, n_public public outputs, n_free free inputs, each
 * constraint defines one fresh wire.  Wire value classes (bits / bytes / full-width) follow SURVEY.md 8d. */
int nzcp_synth_create(uint64_t seed, uint32_t n_constraints, uint32_t n_public, uint32_t n_free, nzcp_synth** out);
void nzcp_synth_free(nzcp_synth* c);
int nzcp_synth_dims(const nzcp_synth* c, uint32_t* n_vars, uint32_t* n_constraints, uint32_t* n_public,
                    uint32_t* domain_size, uint64_t* n_coefs);
/* Size in bytes of the .zkey / .r1cs / .wtns images the writers below produce. */
size_t nzcp_synth_zkey_size(const nzcp_synth* c);
size_t nzcp_synth_r1cs_size(const nzcp_synth* c);
size_t nzcp_synth_wtns_size(const nzcp_synth* c);
/* Groth16 setup from explicit toxic waste (5 x 32-byte LE: tau, alpha, beta, gamma, delta) -> snarkjs-format .zkey.
 * The fixed-base scalar multiplications run on `device`. */
int nzcp_synth_write_zkey(const nzcp_synth* c, const uint8_t toxic[160], int device, uint8_t* out, size_t cap);
int nzcp_synth_write_r1cs(const nzcp_synth* c, uint8_t* out, size_t cap);
/* Satisfying witness for the given seed -> .wtns image. */
int nzcp_synth_write_wtns(const nzcp_synth* c, uint64_t witness_seed, uint8_t* out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* NZCP_PROVER_H */
