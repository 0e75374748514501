// Shared host-side declarations for libnzcp_prover.so (internal; the public C ABI is include/nzcp_prover.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <stdexcept>
#include <string>
#include <vector>

#include "ec.cuh"

namespace nzcp {

struct CudaError : std::runtime_error {
  explicit CudaError(const std::string& s) : std::runtime_error(s) {}
};

#define NZCP_CUDA(expr)                                                                              \
  do {                                                                                               \
    cudaError_t e__ = (expr);                                                                        \
    if (e__ != cudaSuccess) {                                                                        \
      char b__[512];                                                                                 \
      snprintf(b__, sizeof b__, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e__), __FILE__,    \
               __LINE__, #expr);                                                                     \
      throw nzcp::CudaError(b__);                                                                    \
    }                                                                                                \
  } while (0)

extern std::atomic<uint64_t> g_launch_count;  // every kernel launch of this library, process-wide
// Launches are also charged to the prover the calling thread is working for (prove_impl points this at the prover's own
// counter for the duration of the call): nzcp_prover_launch_count / bench.py "gpu_launches" are per prover.
extern thread_local std::atomic<uint64_t>* t_launch_sink;
#define NZCP_LAUNCH_CHECK()                                        \
  do {                                                             \
    nzcp::g_launch_count.fetch_add(1);                             \
    if (nzcp::t_launch_sink) nzcp::t_launch_sink->fetch_add(1);    \
    NZCP_CUDA(cudaGetLastError());                                 \
  } while (0)

static inline unsigned div_up(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

G1Affine g1_generator();   // synth.cu: the BN254 generators, Montgomery affine
G2Affine g2_generator();
Fr host_fr_root(int k);    // ntt.cu: ffjavascript's Fr.w[k], Montgomery

// ---------------------------------------------------------------------------------------------- NTT (ntt.cu)
// Tables for one domain size n = 2^log_n (Montgomery-form Fr, device memory).
struct NttDomain {
  int log_n = 0;
  Fr* tw_fwd = nullptr;   // w^j, j < n/2, w = Fr.w[log_n]
  Fr* tw_inv = nullptr;   // w^-j
  Fr* coset_scale = nullptr;  // n^-1 * inc^bitrev(p), p < n   (iNTT scale fused with batchApplyKey)
  Fr* ninv_scale = nullptr;   // unused slot kept for standalone iNTT: single element n^-1 (device)
  unsigned char* tw_lo_fwd = nullptr;   // log_n >= 10: w^(j n/1024), j < 512, padded layout (ntt.cu tw_pad_off): the twiddles
  unsigned char* tw_lo_inv = nullptr;   // of every stage of a 2^10 tile, bulk-copied into shared memory by the low pass
};
void ntt_domain_create(NttDomain* d, int log_n, cudaStream_t st);
void ntt_domain_destroy(NttDomain* d);
// H pipeline on `batch` polynomials laid out back to back (batch * n elements), in place:
//   evaluations on the 2^log_n subgroup (natural order)  ->  evaluations on the coset inc*subgroup (natural order)
void ntt_coset_pipeline(const NttDomain& d, Fr* data, int batch, cudaStream_t st);
// Standalone natural-order transforms (snarkjs Fr.fft / Fr.ifft semantics); `tmp` is an n-element scratch.
void ntt_forward(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st);
void ntt_inverse(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st);
// h[i] = fromMontgomery(a[i]*b[i] - c[i])
void ntt_join_abc(const Fr* a, const Fr* b, const Fr* c, Fr* h, size_t n, cudaStream_t st);

// ---------------------------------------------------------------------------------------------- R1CS (r1cs.cu)
struct R1csDevice {
  uint32_t n = 0;            // domain size (rows per matrix)
  uint64_t nnz = 0;
  uint32_t* row_ptr = nullptr;  // 2n+1 entries: rows 0..n-1 = A, n..2n-1 = B
  uint32_t* col = nullptr;      // signal index per coefficient
  Fr* val = nullptr;            // coef * R^2 mod r exactly as stored in zkey section 4
  uint32_t* order = nullptr;    // thread t evaluates constraint order[t]: each 128-row block sorted by row length
};
// abc = [A_T | B_T | C_T], each n Montgomery-form Fr.  witness: plain Fr, n_vars entries.
void r1cs_eval(const R1csDevice& m, const Fr* witness, Fr* abc, cudaStream_t st);

// ---------------------------------------------------------------------------------------------- MSM (msm.cu)
// Precomputed window table of one base section (built once per proving key; the bases never change between proofs):
//   pts[w * n_points + i] = 2^(c*w) * P_i   affine Montgomery, (0,0) = infinity
// so that all windows of a scalar feed ONE bucket set and the Horner pass over windows disappears.
struct MsmTable {
  void* pts = nullptr;
  size_t n_points = 0;   // including pad_front leading infinity points
  int c = 0, n_windows = 0;
  bool g2 = false;
  bool owned = true;     // false: a view over the caller's bases (msm_table_view)
  size_t bytes = 0;
};
int msm_pick_window(size_t n_points);
int msm_num_windows(int c);
int msm_pick_window_free(size_t n_points);
// d_bases: device array of n_src affine points; the table gets pad_front infinity points in front of them.
void msm_table_create(MsmTable* t, const void* d_bases, size_t n_src, size_t pad_front, bool g2, int c, cudaStream_t st);
// "Table" view of raw bases for the table-free path (one window, memory owned by the caller).
void msm_table_view(MsmTable* t, void* d_bases, size_t n_points, bool g2, int c);
void msm_table_destroy(MsmTable* t);

static constexpr int kMsmMaxRounds = 3;

// Bucket sort of one scalar vector: signed c-bit digits -> (table index | sign) entries grouped by bucket, cut into
// tasks of <= kTaskLen entries.  Shared by every MSM that uses the same scalars (A, B1, B2, C all use the witness).
struct MsmSort {
  size_t n_points = 0;
  int c = 0, n_windows = 0;
  size_t n_buckets = 0;     // all buckets: group_buckets * n_groups
  size_t group_buckets = 0; // 2^(c-1)
  int n_groups = 1;         // 1: window-table mode (all windows share the buckets); n_windows: table-free mode
  bool table_free = false;  // entries index the raw bases (no window table); window w accumulates into bucket group w
  bool smem_hist = false;   // histogram in shared memory (<= 2^15 buckets) or with global atomics
  uint32_t n_copies = 0;    // private copies of each bucket counter (smem path: one per block)
  uint32_t* counts = nullptr;
  uint32_t* offsets = nullptr;
  uint32_t* cursors = nullptr;
  uint32_t* block_sums = nullptr;  // scratch of the multi-block scan
  uint32_t* entries = nullptr;
  uint32_t* task_off = nullptr;
  uint2* tasks = nullptr;
  uint32_t* flags = nullptr;      // [1] error flags, [2] total tasks, [3] total entries, [4] task length,
                                  // [5] points left after the affine pair rounds (= [3] when rounds == 0)
  uint32_t* flags_host = nullptr; // pinned mirror
  size_t max_tasks = 0;
  size_t scratch_bytes = 0;
  // Batched-affine pair rounds (msm.cu "pair rounds"): round r halves every bucket's point list (ceil(len / 2)) with
  // affine additions that share one field inversion per thread.  round_off[r * (n_buckets + 1) + b] = first slot of
  // bucket b in the round-r point array (r = 0: the entry list itself, compact copy of `offsets`); red_count[b] =
  // points of bucket b after the last round -- what the task list and the XYZZ accumulation then work on.
  int rounds = 0;
  uint32_t* round_off = nullptr;
  uint32_t* red_count = nullptr;
  size_t round_max[kMsmMaxRounds + 1] = {0, 0, 0, 0};   // upper bound of the point count after round r
};
int msm_pick_rounds(size_t n_points, int c);
int msm_pick_rounds_prover(size_t n_points, int c);
void msm_sort_create(MsmSort* s, size_t n_points, int c, int rounds = -1, bool table_free = false);   // rounds < 0: msm_pick_rounds
void msm_sort_destroy(MsmSort* s);
void msm_sort_launch(MsmSort* s, const Fr* scalars, size_t n_points, cudaStream_t st);
// After the stream drained: throws if the device flagged a scalar >= r.  Returns the number of non-zero digits.
uint32_t msm_sort_check(const MsmSort* s);

// One MSM against a sorted scalar vector: accumulate -> combine -> bucket reduction.
struct MsmRun {
  bool g2 = false;
  void* partial = nullptr;
  void* buckets = nullptr;
  void* marg = nullptr;       // marginal bucket sums M_k[j], k < n_digits, j < 32
  int n_digits = 0;           // base-32 digits of a bucket id
  int n_groups = 1, c = 0;    // bucket groups (table-free: one per window) and window bits, copied from the sort plan
  uint32_t* marg_done = nullptr;   // per (group, digit): marginal blocks finished (self-resetting)
  void* result = nullptr;     // device: the finished sum as one XYZZ point (msm_run_finish_device)
  uint32_t* heavy_list = nullptr;
  uint32_t* heavy_count = nullptr;   // [0] heavy buckets, [1] heavy chunks
  uint32_t* chunk_off = nullptr;
  void* chunk_partial = nullptr;
  void* out = nullptr;        // device: S_0 .. S_{n_digits-1}, T
  void* out_host = nullptr;   // pinned
  cudaEvent_t ev_acc0 = nullptr, ev_acc1 = nullptr;  // around the bucket accumulation (pair rounds + XYZZ kernel)
  void* round_pts[2] = {nullptr, nullptr};   // affine point arrays of the pair rounds (ping-pong)
  void* round_prefix = nullptr;              // prefix products of the shared inversion, [step][thread]
  void* round_ops = nullptr;                 // round 1: the two operands of every addition, staged by the forward pass
  void* round_prod = nullptr;                // per-thread denominator products, inverted in place between the passes
  size_t scratch_bytes = 0;
};
void msm_run_create(MsmRun* r, const MsmSort* sort, bool g2);
void msm_run_destroy(MsmRun* r);
void msm_run_launch(MsmRun* r, const MsmSort* sort, const MsmTable* table, cudaStream_t st);
void msm_run_finish_device(MsmRun* r, cudaStream_t st);
void msm_sum_points(const void* d_pts, uint32_t count, bool g2, void* d_result, cudaStream_t st);
G1XYZZ msm_run_finish_g1(const MsmRun* r);
G2XYZZ msm_run_finish_g2(const MsmRun* r);
float msm_run_accumulate_ms(const MsmRun* r);

}  // namespace nzcp
