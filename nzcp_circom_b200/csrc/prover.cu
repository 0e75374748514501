// groth16.prove on one B200: zkey resident in HBM, one call per proof.
//
// Replaces snarkjs 0.4.12 src/groth16_prove.js groth16Prove() (upstream, not vendored: package.json:12,
// yarn.lock:987-999) together with the container readers it uses (@iden3/binfileutils readBinFile/readSection,
// snarkjs src/zkey_utils.js readHeader, src/wtns_utils.js readHeader).  Order of work and every formula follow
// that function: buildABC1 -> (ifft, batchApplyKey, fft) x3 -> joinABC -> 5 multiexps -> r/s blinding -> affine.
// Differences that do not change any output bit: sections 4-9 are parsed and uploaded once per zkey instead of
// re-read per proof; the COO coefficient list is regrouped to CSR; the four witness MSMs run on their own streams
// concurrently with the H pipeline.
#include <stdlib.h>
#include <memory>
#include <mutex>
#include <thread>

#include "binfile.cuh"

namespace nzcp {

extern std::atomic<int> g_tune_rounds_w, g_tune_rounds_h;   // msm.cu
std::atomic<uint64_t> g_launch_count{0};
thread_local std::atomic<uint64_t>* t_launch_sink = nullptr;
// "stage_mode" knob: how nzcp_prove moves a HOST witness to the GPU.  -1 = automatic: pageable memory (a Node Buffer, a
// Python bytes object) goes through the prover's pinned staging buffer in chunks, so the CPU copy of chunk k+1 overlaps
// the DMA of chunk k; memory the caller pinned (cudaHostAlloc / cudaHostRegister) is handed to the copy engine directly.
// 0 = always direct (the driver stages pageable memory itself), 1 = always through the staging buffer.
std::atomic<int> g_tune_rounds_b2{-1};   // "prover_rounds_b2": pair rounds of the G2 MSM (-1 = as the other witness MSMs)
std::atomic<int> g_tune_c_h{0}, g_tune_c_w{0};   // "prover_c_h" / "prover_c_w": window bits of the H / witness MSM tables (0 = default)
std::atomic<int> g_tune_stage_mode{-1};
std::atomic<int> g_tune_stage_chunk_kb{1024};
std::atomic<int> g_tune_stage_threads{4};      // host threads sharing the copy into the staging buffer (1 = the caller alone)

static thread_local std::string t_last_error;
void set_last_error(const std::string& s) { t_last_error = s; }

}  // namespace nzcp

using namespace nzcp;

struct nzcp_zkey {
  int device = 0;
  std::mutex pool_mu;                    // guards `pool` (provers owned by the key, used by nzcp_prove_batch)
  std::vector<nzcp_prover*> pool;
  uint32_t n_vars = 0, n_public = 0, domain_size = 0, power = 0;
  uint64_t n_coefs = 0;
  G1Affine alpha1, beta1, delta1;  // Montgomery affine, as stored
  G2Affine beta2, gamma2, delta2;
  R1csDevice r1cs;
  int c_w = 0, c_h = 0;                          // MSM window bits for the witness MSMs / the H MSM
  MsmTable tab_a, tab_b1, tab_b2, tab_c, tab_h;  // window tables of sections 5-9 (tab_c front-padded to n_vars)
  NttDomain dom;
  size_t device_bytes = 0;
};

struct nzcp_prover {
  nzcp_zkey* zk = nullptr;
  int device = 0;                               // copy of zk->device: release must not touch a key freed before it
  std::atomic<uint64_t> launches{0};            // kernel launches issued for this prover (nzcp_prover_launch_count)
  uint8_t* h_stage = nullptr;                   // pinned staging buffer for pageable host witnesses (n_vars * 32 B, lazy)
  cudaStream_t st_main = nullptr;
  cudaStream_t st_msm[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev[20];
  int n_ev = 0;
  Fr* d_wtns = nullptr;
  Fr* d_abc = nullptr;
  Fr* d_h = nullptr;
  MsmSort sort_w, sort_h;                       // bucket sorts of the witness and of the h scalars
  MsmSort sort_b2;                              // the G2 MSM's own witness sort when its round count differs ("prover_rounds_b2")
  bool own_b2_sort = false;
  MsmRun run_a, run_b1, run_b2, run_c, run_h;
};

namespace nzcp {

static void prover_release(nzcp_prover* p);

static void zkey_release(nzcp_zkey* zk) {
  if (!zk) return;
  cudaSetDevice(zk->device);
  for (nzcp_prover* p : zk->pool) prover_release(p);
  zk->pool.clear();
  cudaFree(zk->r1cs.row_ptr);
  cudaFree(zk->r1cs.col);
  cudaFree(zk->r1cs.val);
  cudaFree(zk->r1cs.order);
  msm_table_destroy(&zk->tab_a);
  msm_table_destroy(&zk->tab_b1);
  msm_table_destroy(&zk->tab_b2);
  msm_table_destroy(&zk->tab_c);
  msm_table_destroy(&zk->tab_h);
  ntt_domain_destroy(&zk->dom);
  delete zk;
}

template <class T>
static T* upload(const void* src, size_t bytes, size_t* total) {
  T* d = nullptr;
  NZCP_CUDA(cudaMalloc(&d, bytes ? bytes : 16));
  if (bytes) NZCP_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
  *total += bytes;
  return d;
}

static nzcp_zkey* zkey_load_impl(const uint8_t* b, size_t len, int device) {
  const Zkey z = read_zkey(b, len);
  const Sect* s = z.s;
  need_sections(s, 3, 9);
  std::unique_ptr<nzcp_zkey, void (*)(nzcp_zkey*)> zk(new nzcp_zkey(), zkey_release);
  zk->device = device;
  zk->n_vars = z.n_vars;
  zk->n_public = z.n_public;
  zk->domain_size = z.domain_size;
  zk->power = zkey_domain_power(z);
  const uint32_t n = zk->domain_size;
  const uint8_t* h = s[2].p;
  memcpy(&zk->alpha1, h + kZkeyAlpha1Off, 64);
  memcpy(&zk->beta1, h + kZkeyBeta1Off, 64);
  memcpy(&zk->beta2, h + kZkeyBeta2Off, 128);
  memcpy(&zk->gamma2, h + kZkeyGamma2Off, 128);
  memcpy(&zk->delta1, h + kZkeyDelta1Off, 64);
  memcpy(&zk->delta2, h + kZkeyDelta2Off, 128);
  // section sizes
  const uint64_t m = zk->n_vars;
  if (s[5].len != m * 64 || s[6].len != m * 64 || s[7].len != m * 128 || s[8].len != z.n_l() * 64 ||
      s[9].len != (uint64_t)n * 64)
    throw ApiError(NZCP_E_FORMAT, "zkey: point section size does not match header");
  // section 4: COO coefficients -> CSR (rows 0..n-1 = A, n..2n-1 = B)
  if (s[4].len < 4) throw ApiError(NZCP_E_FORMAT, "zkey: short coefficient section");
  uint64_t nc = rd32u(s[4].p);
  if (s[4].len != 4 + nc * 44) throw ApiError(NZCP_E_FORMAT, "zkey: coefficient section size mismatch");
  zk->n_coefs = nc;
  std::vector<uint32_t> row_ptr(2 * (size_t)n + 1, 0);
  const uint8_t* cp = s[4].p + 4;
  for (uint64_t i = 0; i < nc; i++) {
    const uint8_t* rec = cp + i * 44;
    uint32_t mtx = rd32u(rec), c = rd32u(rec + 4), sg = rd32u(rec + 8);
    if (mtx > 1 || c >= n || sg >= zk->n_vars) throw ApiError(NZCP_E_FORMAT, "zkey: coefficient record out of range");
    row_ptr[(size_t)mtx * n + c + 1]++;
  }
  for (size_t i = 0; i < 2 * (size_t)n; i++) row_ptr[i + 1] += row_ptr[i];
  std::vector<uint32_t> fill(row_ptr.begin(), row_ptr.end() - 1);
  std::vector<uint32_t> col(nc ? nc : 1);
  std::vector<Fr> val(nc ? nc : 1);
  for (uint64_t i = 0; i < nc; i++) {
    const uint8_t* rec = cp + i * 44;
    uint32_t mtx = rd32u(rec), c = rd32u(rec + 4), sg = rd32u(rec + 8);
    uint32_t pos = fill[(size_t)mtx * n + c]++;
    col[pos] = sg;
    memcpy(val[pos].v, rec + 12, 32);
  }
  use_device(device);
  size_t tot = 0;
  zk->r1cs.n = n;
  zk->r1cs.nnz = nc;
  zk->r1cs.row_ptr = upload<uint32_t>(row_ptr.data(), row_ptr.size() * 4, &tot);
  zk->r1cs.col = upload<uint32_t>(col.data(), nc * 4, &tot);
  zk->r1cs.val = upload<Fr>(val.data(), nc * 32, &tot);
  // Constraint order for the evaluation kernel (one thread per constraint): inside every block of 128 consecutive
  // constraints the rows are handed to threads longest first, so the 32 lanes of a warp walk rows of similar length
  // (NZCP rows have 1..8 terms; unsorted, a warp runs as long as its longest row while the average is under 3).
  {
    std::vector<uint32_t> order(n);
    uint32_t key[128];
    for (size_t b0 = 0; b0 < n; b0 += 128) {
      const size_t cnt = n - b0 < 128 ? n - b0 : 128;
      uint32_t hist[64] = {0};
      for (size_t j = 0; j < cnt; j++) {
        const size_t i = b0 + j;
        uint32_t len = (row_ptr[i + 1] - row_ptr[i]) + (row_ptr[n + i + 1] - row_ptr[n + i]);
        key[j] = len > 63 ? 63 : len;
        hist[key[j]]++;
      }
      uint32_t start[64], run = 0;
      for (int l = 63; l >= 0; l--) { start[l] = run; run += hist[l]; }   // counting sort, longest first, stable
      for (size_t j = 0; j < cnt; j++) order[b0 + start[key[j]]++] = (uint32_t)(b0 + j);
    }
    zk->r1cs.order = upload<uint32_t>(order.data(), (size_t)n * 4, &tot);
  }
  // sections 5-9 -> window tables (one-time expansion; the raw section is only staged)
  zk->c_w = g_tune_c_w.load() > 0 ? g_tune_c_w.load() : msm_pick_window(m);
  zk->c_h = g_tune_c_h.load() > 0 ? g_tune_c_h.load() : msm_pick_window(n);
  auto make_table = [&](MsmTable* t, const Sect& sec, size_t count, size_t pad, bool g2, int c) {
    size_t dummy = 0;
    void* raw = upload<unsigned char>(sec.p, sec.len, &dummy);
    try {
      msm_table_create(t, raw, count, pad, g2, c, 0);
      NZCP_CUDA(cudaDeviceSynchronize());
    } catch (...) {
      cudaFree(raw);
      throw;
    }
    cudaFree(raw);
    tot += t->bytes;
  };
  make_table(&zk->tab_a, s[5], m, 0, false, zk->c_w);
  make_table(&zk->tab_b1, s[6], m, 0, false, zk->c_w);
  make_table(&zk->tab_b2, s[7], m, 0, true, zk->c_w);
  make_table(&zk->tab_c, s[8], z.n_l(), zk->n_public + 1, false, zk->c_w);
  make_table(&zk->tab_h, s[9], n, 0, false, zk->c_h);
  ntt_domain_create(&zk->dom, (int)zk->power, 0);
  tot += ((size_t)n / 2 * 2 + n) * sizeof(Fr);
  zk->device_bytes = tot;
  return zk.release();
}

static void prover_release(nzcp_prover* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->h_stage) cudaFreeHost(p->h_stage);
  if (p->st_main) cudaStreamDestroy(p->st_main);
  for (int i = 0; i < 4; i++)
    if (p->st_msm[i]) cudaStreamDestroy(p->st_msm[i]);
  for (int i = 0; i < p->n_ev; i++) cudaEventDestroy(p->ev[i]);
  cudaFree(p->d_wtns);
  cudaFree(p->d_abc);
  cudaFree(p->d_h);
  msm_run_destroy(&p->run_a);
  msm_run_destroy(&p->run_b1);
  msm_run_destroy(&p->run_b2);
  msm_run_destroy(&p->run_c);
  msm_run_destroy(&p->run_h);
  msm_sort_destroy(&p->sort_w);
  msm_sort_destroy(&p->sort_b2);
  msm_sort_destroy(&p->sort_h);
  delete p;
}

// mode 0 = latency (a lone proof at a time), mode 1 = throughput (several provers in flight on one GPU).  Both run the
// batched-affine pair rounds of msm_pair.cuh on every MSM large enough to pay for their extra launches: with the rounds'
// operand prefetch off they cut a lone proof from 9.27 to 8.78 ms and raise four-in-flight throughput from 118 to 131
// proofs/s (profiles/r02_window_rounds_sweep.md).  The mode is kept in the ABI for what differs between the two uses
// (today: nothing but the name; nzcp_prove_batch creates mode-1 provers).
static nzcp_prover* prover_create_impl(nzcp_zkey* zk, int mode = 0) {
  use_device(zk->device);
  std::unique_ptr<nzcp_prover, void (*)(nzcp_prover*)> p(new nzcp_prover(), prover_release);
  p->zk = zk;
  p->device = zk->device;
  NZCP_CUDA(cudaStreamCreateWithFlags(&p->st_main, cudaStreamNonBlocking));
  for (int i = 0; i < 4; i++) NZCP_CUDA(cudaStreamCreateWithFlags(&p->st_msm[i], cudaStreamNonBlocking));
  for (int i = 0; i < 20; i++) {
    NZCP_CUDA(cudaEventCreate(&p->ev[i]));
    p->n_ev = i + 1;
  }
  size_t n = zk->domain_size;
  NZCP_CUDA(cudaMalloc(&p->d_wtns, (size_t)zk->n_vars * sizeof(Fr)));
  NZCP_CUDA(cudaMalloc(&p->d_abc, 3 * n * sizeof(Fr)));
  NZCP_CUDA(cudaMalloc(&p->d_h, n * sizeof(Fr)));
  int rounds_h = g_tune_rounds_h.load(), rounds_w = g_tune_rounds_w.load();
  (void)mode;
  if (rounds_h < 0) rounds_h = msm_pick_rounds_prover(n, zk->c_h);
  if (rounds_w < 0) rounds_w = msm_pick_rounds_prover(zk->n_vars, zk->c_w);
  msm_sort_create(&p->sort_w, zk->n_vars, zk->c_w, rounds_w);
  msm_sort_create(&p->sort_h, n, zk->c_h, rounds_h);
  msm_run_create(&p->run_a, &p->sort_w, false);
  msm_run_create(&p->run_b1, &p->sort_w, false);
  // The round plan is part of the sort, so an MSM that wants another number of pair rounds than its siblings needs its
  // own sort of the same scalars (two more histogram passes over the witness).
  int rounds_b2 = g_tune_rounds_b2.load();
  if (rounds_b2 < 0 || rounds_b2 == rounds_w) {
    msm_run_create(&p->run_b2, &p->sort_w, true);
  } else {
    msm_sort_create(&p->sort_b2, zk->n_vars, zk->c_w, rounds_b2);
    p->own_b2_sort = true;
    msm_run_create(&p->run_b2, &p->sort_b2, true);
  }
  msm_run_create(&p->run_c, &p->sort_w, false);
  msm_run_create(&p->run_h, &p->sort_h, false);
  return p.release();
}

static void random_fr(uint8_t out[32]) {
  FILE* f = fopen("/dev/urandom", "rb");
  if (!f) throw ApiError(NZCP_E_INTERNAL, "cannot open /dev/urandom");
  for (;;) {
    if (fread(out, 1, 32, f) != 32) {
      fclose(f);
      throw ApiError(NZCP_E_INTERNAL, "short read from /dev/urandom");
    }
    out[31] &= 0x3f;  // < 2^254; rejection-sample into [0, r)
    if (fr_bytes_canonical(out)) break;
  }
  fclose(f);
}

// Host witness -> p->d_wtns on stream `st`.  Pageable source memory is copied through the prover's pinned staging buffer
// in chunks (CPU copy of chunk k+1 overlaps the DMA of chunk k, and the stream is never blocked behind the driver's own
// pageable-memory path, which serialises with every other stream of the process); pinned sources go straight to the
// copy engine.  The staging buffer is as large as the witness, so no slot is reused inside one proof, and the previous
// proof of this prover has drained its streams before the call returned.
static void upload_witness(nzcp_prover* p, const uint8_t* h_witness, size_t bytes, cudaStream_t st) {
  int mode = g_tune_stage_mode.load();
  bool stage = mode == 1;
  if (mode < 0) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, h_witness) != cudaSuccess) {
      cudaGetLastError();
      stage = true;
    } else {
      stage = attr.type == cudaMemoryTypeUnregistered;
    }
  }
  if (!stage) {
    NZCP_CUDA(cudaMemcpyAsync(p->d_wtns, h_witness, bytes, cudaMemcpyHostToDevice, st));
    return;
  }
  if (!p->h_stage) NZCP_CUDA(cudaHostAlloc((void**)&p->h_stage, (size_t)p->zk->n_vars * sizeof(Fr), cudaHostAllocDefault));
  size_t chunk = (size_t)g_tune_stage_chunk_kb.load() * 1024;
  if (chunk < 65536) chunk = 65536;
  // A single core copies ~10 GB/s: 2.8 ms for the 28 MB NZCP witness, a quarter of the whole proof.  The copy is shared by
  // a few short-lived host threads, each staging and enqueueing its own contiguous part (the H2D copies are independent,
  // their order on the stream does not matter); the caller takes the first part itself.
  int nt = g_tune_stage_threads.load();
  if (nt < 1) nt = 1;
  if (nt > 16) nt = 16;
  if (bytes < (size_t)nt * chunk) nt = (int)(bytes / chunk ? bytes / chunk : 1);
  const int device = p->device;
  uint8_t* d_dst = reinterpret_cast<uint8_t*>(p->d_wtns);
  uint8_t* stage_buf = p->h_stage;
  std::atomic<int> failed{0};
  auto part = [&](int k, bool set_device) {
    if (set_device && cudaSetDevice(device) != cudaSuccess) { failed.store(1); return; }
    const size_t per = ((bytes + nt - 1) / nt + 63) & ~(size_t)63;
    const size_t b = (size_t)k * per, e = b + per < bytes ? b + per : bytes;
    for (size_t off = b; off < e; off += chunk) {
      const size_t len = e - off < chunk ? e - off : chunk;
      memcpy(stage_buf + off, h_witness + off, len);
      if (cudaMemcpyAsync(d_dst + off, stage_buf + off, len, cudaMemcpyHostToDevice, st) != cudaSuccess) { failed.store(1); return; }
    }
  };
  std::vector<std::thread> helpers;
  for (int k = 1; k < nt; k++) helpers.emplace_back(part, k, true);
  part(0, false);
  for (auto& t : helpers) t.join();
  if (failed.load()) {
    cudaGetLastError();
    throw CudaError("staged upload of the witness failed");
  }
}

// Event slots: 0 start, 1 upload done, 2 eval done, 3 ntt+join done, 4 msm H done, 5 witness sort done,
// 6..13 msm A,B1,B2,C (begin,end), 14 h sort done
static void prove_impl(nzcp_prover* p, const uint8_t* h_witness, const Fr* d_witness_ext, const uint8_t* r_in,
                       const uint8_t* s_in, nzcp_proof* proof, nzcp_prove_debug* dbg) {
  nzcp_zkey* zk = p->zk;
  if (!proof) throw ApiError(NZCP_E_ARG, "proof pointer is null");
  uint8_t rb[32], sb[32];
  if (r_in) memcpy(rb, r_in, 32); else random_fr(rb);
  if (s_in) memcpy(sb, s_in, 32); else random_fr(sb);
  if (!fr_bytes_canonical(rb) || !fr_bytes_canonical(sb)) throw ApiError(NZCP_E_ARG, "blinding scalar r or s is not < r");
  use_device(zk->device);
  const size_t n = zk->domain_size, m = zk->n_vars;
  cudaStream_t sm = p->st_main;
  struct Sink {   // kernel launches of this call are charged to this prover
    std::atomic<uint64_t>* prev;
    explicit Sink(std::atomic<uint64_t>* c) : prev(t_launch_sink) { t_launch_sink = c; }
    ~Sink() { t_launch_sink = prev; }
  } sink(&p->launches);
  auto drain = [&] {   // leave no work in flight behind an error: the prover (and its buffers) may be reused or freed
    for (int k = 0; k < 4; k++) cudaStreamSynchronize(p->st_msm[k]);
    cudaStreamSynchronize(sm);
  };
  try {
  NZCP_CUDA(cudaEventRecord(p->ev[0], sm));
  const Fr* d_w = d_witness_ext;
  if (h_witness) {
    upload_witness(p, h_witness, m * sizeof(Fr), sm);
    d_w = p->d_wtns;
  }
  NZCP_CUDA(cudaEventRecord(p->ev[1], sm));
  // Launch order = the proof's critical path first: r1cs -> NTT -> join -> H sort go out before the ~40 launches of the
  // witness sort and MSMs, so the GPU starts on the chain that cannot be shortened while the host is still enqueueing
  // the filler (the four witness MSMs, 3 ms of full-GPU work).  Measured alternatives (lone proof, DESIGN.md section 5):
  // a high-priority stream for this chain and gating the witness accumulations behind the NTT or the H sort all lose --
  // the sort's whole-SM blocks cannot be placed while accumulate blocks keep refilling the SMs, whatever the priority.
  r1cs_eval(zk->r1cs, d_w, p->d_abc, sm);
  NZCP_CUDA(cudaEventRecord(p->ev[2], sm));
  ntt_coset_pipeline(zk->dom, p->d_abc, 3, sm);
  ntt_join_abc(p->d_abc, p->d_abc + n, p->d_abc + 2 * n, p->d_h, n, sm);
  NZCP_CUDA(cudaEventRecord(p->ev[3], sm));
  msm_sort_launch(&p->sort_h, p->d_h, n, sm);
  NZCP_CUDA(cudaEventRecord(p->ev[14], sm));
  // The four witness MSMs (snarkjs order: A, B1, B2, C) share ONE bucket sort of the witness; the C table is
  // front-padded with nPublic+1 infinity points so it is indexed by wire number like the others.
  // B2 (G2, the longest) is sorted for on its own stream and launched first.
  cudaStream_t sw = p->st_msm[2];
  NZCP_CUDA(cudaStreamWaitEvent(sw, p->ev[1], 0));
  if (p->own_b2_sort) {   // B2 sorts for itself on its stream; the shared sort moves to A's stream
    msm_sort_launch(&p->sort_b2, d_w, m, sw);
    sw = p->st_msm[0];
    NZCP_CUDA(cudaStreamWaitEvent(sw, p->ev[1], 0));
  }
  msm_sort_launch(&p->sort_w, d_w, m, sw);
  NZCP_CUDA(cudaEventRecord(p->ev[5], sw));
  struct Job { MsmRun* run; const MsmTable* tab; int stream; };
  Job jobs[4] = {{&p->run_b2, &zk->tab_b2, 2}, {&p->run_a, &zk->tab_a, 0}, {&p->run_b1, &zk->tab_b1, 1}, {&p->run_c, &zk->tab_c, 3}};
  for (int k = 0; k < 4; k++) {
    cudaStream_t st = p->st_msm[jobs[k].stream];
    const bool own = p->own_b2_sort && jobs[k].run == &p->run_b2;
    if (st != sw && !own) NZCP_CUDA(cudaStreamWaitEvent(st, p->ev[5], 0));
    NZCP_CUDA(cudaEventRecord(p->ev[6 + 2 * jobs[k].stream], st));
    msm_run_launch(jobs[k].run, own ? &p->sort_b2 : &p->sort_w, jobs[k].tab, st);
    NZCP_CUDA(cudaEventRecord(p->ev[7 + 2 * jobs[k].stream], st));
  }
  msm_run_launch(&p->run_h, &p->sort_h, &zk->tab_h, sm);
  NZCP_CUDA(cudaEventRecord(p->ev[4], sm));
  if (dbg && dbg->h_scalars) NZCP_CUDA(cudaMemcpyAsync(dbg->h_scalars, p->d_h, n * sizeof(Fr), cudaMemcpyDeviceToHost, sm));
  } catch (...) {
    drain();
    throw;
  }
  // While the GPU works: the blinding terms that depend only on r, s and the key (r*delta1, s*delta1, s*delta2,
  // -rs*delta1) -- four of the six scalar multiplications of the final combination leave the latency path.
  const Fr r = fp_from_bytes_plain<FrParams>(rb), s = fp_from_bytes_plain<FrParams>(sb);
  const Fr neg_rs = fp_neg(fp_from_mont(fp_mul(fp_to_mont(r), fp_to_mont(s))));
  const G1XYZZ d1 = G1XYZZ::from_affine(zk->delta1);
  const G1XYZZ r_d1 = xyzz_mul(d1, r.v), s_d1 = xyzz_mul(d1, s.v), nrs_d1 = xyzz_mul(d1, neg_rs.v);
  const G2XYZZ s_d2 = xyzz_mul(G2XYZZ::from_affine(zk->delta2), s.v);
  // The witness MSMs finish well before the H chain (r1cs -> NTT -> sort -> MSM): drain their streams one by one and do
  // the two result-dependent scalar multiplications (s * pi_A, r * B1') on the host while the GPU is still busy with H.
  G1XYZZ A, B1, C, H, pi_a, pib1, s_pi_a, r_pib1;
  G2XYZZ B2;
  uint32_t ent_w = 0, ent_h = 0;
  try {
    NZCP_CUDA(cudaStreamSynchronize(p->st_msm[0]));   // A (its stream waited for the witness sort and its flags)
    ent_w = msm_sort_check(&p->sort_w);
    A = msm_run_finish_g1(&p->run_a);
    pi_a = A;
    xyzz_add(pi_a, G1XYZZ::from_affine(zk->alpha1));
    xyzz_add(pi_a, r_d1);
    s_pi_a = xyzz_mul(pi_a, s.v);
    g1_to_plain_bytes(pi_a, proof->pi_a);
    NZCP_CUDA(cudaStreamSynchronize(p->st_msm[1]));   // B1
    B1 = msm_run_finish_g1(&p->run_b1);
    pib1 = B1;
    xyzz_add(pib1, G1XYZZ::from_affine(zk->beta1));
    xyzz_add(pib1, s_d1);
    r_pib1 = xyzz_mul(pib1, r.v);
    NZCP_CUDA(cudaStreamSynchronize(p->st_msm[2]));   // B2: pi_B needs nothing else
    B2 = msm_run_finish_g2(&p->run_b2);
    G2XYZZ pi_b = B2;
    xyzz_add(pi_b, G2XYZZ::from_affine(zk->beta2));
    xyzz_add(pi_b, s_d2);
    g2_to_plain_bytes(pi_b, proof->pi_b);
    NZCP_CUDA(cudaStreamSynchronize(p->st_msm[3]));   // C
    C = msm_run_finish_g1(&p->run_c);
    NZCP_CUDA(cudaStreamSynchronize(sm));             // H: only its Horner tail, four additions and one inversion remain
    ent_h = msm_sort_check(&p->sort_h);
  } catch (const std::runtime_error& e) {
    drain();
    if (dynamic_cast<const CudaError*>(&e) || dynamic_cast<const ApiError*>(&e)) throw;
    throw ApiError(NZCP_E_RANGE, e.what());
  }
  H = msm_run_finish_g1(&p->run_h);
  if (dbg) {
    g1_to_plain_bytes(A, dbg->msm_a);
    g1_to_plain_bytes(B1, dbg->msm_b1);
    g2_to_plain_bytes(B2, dbg->msm_b2);
    g1_to_plain_bytes(C, dbg->msm_c);
    g1_to_plain_bytes(H, dbg->msm_h);
    float t;
    auto el = [&](int a, int b) { cudaEventElapsedTime(&t, p->ev[a], p->ev[b]); return t; };
    dbg->stage_ms[0] = el(0, 1);
    dbg->stage_ms[1] = el(1, 2);
    dbg->stage_ms[2] = el(2, 3);
    dbg->stage_ms[3] = el(6, 7);
    dbg->stage_ms[4] = el(8, 9);
    dbg->stage_ms[5] = el(10, 11);
    dbg->stage_ms[6] = el(12, 13);
    dbg->stage_ms[7] = el(3, 4);
    dbg->sort_ms[0] = el(1, 5);
    dbg->sort_ms[1] = el(3, 14);
    dbg->accumulate_ms[0] = msm_run_accumulate_ms(&p->run_a);
    dbg->accumulate_ms[1] = msm_run_accumulate_ms(&p->run_b1);
    dbg->accumulate_ms[2] = msm_run_accumulate_ms(&p->run_b2);
    dbg->accumulate_ms[3] = msm_run_accumulate_ms(&p->run_c);
    dbg->accumulate_ms[4] = msm_run_accumulate_ms(&p->run_h);
    dbg->n_entries[0] = ent_w;
    dbg->n_entries[1] = ent_h;
    dbg->total_ms = el(0, 4);
  }
  // finalisation (tail of groth16Prove): O(1) group operations on the host, as snarkjs does on its main thread
  G1XYZZ pi_c = C;
  xyzz_add(pi_c, H);
  xyzz_add(pi_c, s_pi_a);
  xyzz_add(pi_c, r_pib1);
  xyzz_add(pi_c, nrs_d1);
  g1_to_plain_bytes(pi_c, proof->pi_c);
}

}  // namespace nzcp

// ================================================================================================ C ABI
extern "C" {

const char* nzcp_last_error(void) { return t_last_error.c_str(); }

int nzcp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int nzcp_zkey_load(const uint8_t* bytes, size_t len, int device, nzcp_zkey** out) {
  return api_guard([&] {
    if (!bytes || !out) throw ApiError(NZCP_E_ARG, "null argument");
    *out = nullptr;
    *out = zkey_load_impl(bytes, len, device);
  });
}

int nzcp_zkey_info_get(const nzcp_zkey* zk, nzcp_zkey_info* info) {
  return api_guard([&] {
    if (!zk || !info) throw ApiError(NZCP_E_ARG, "null argument");
    memset(info, 0, sizeof *info);
    info->n_vars = zk->n_vars;
    info->n_public = zk->n_public;
    info->domain_size = zk->domain_size;
    info->power = zk->power;
    info->n_coefs = zk->n_coefs;
    info->device_bytes = zk->device_bytes;
    g1_to_plain_bytes(G1XYZZ::from_affine(zk->alpha1), info->alpha1);
    g1_to_plain_bytes(G1XYZZ::from_affine(zk->beta1), info->beta1);
    g1_to_plain_bytes(G1XYZZ::from_affine(zk->delta1), info->delta1);
    g2_to_plain_bytes(G2XYZZ::from_affine(zk->beta2), info->beta2);
    g2_to_plain_bytes(G2XYZZ::from_affine(zk->gamma2), info->gamma2);
    g2_to_plain_bytes(G2XYZZ::from_affine(zk->delta2), info->delta2);
  });
}

void nzcp_zkey_free(nzcp_zkey* zk) { zkey_release(zk); }

int nzcp_prover_create(nzcp_zkey* zk, nzcp_prover** out) {
  return api_guard([&] {
    if (!zk || !out) throw ApiError(NZCP_E_ARG, "null argument");
    *out = nullptr;
    *out = prover_create_impl(zk);
  });
}

int nzcp_prover_create_mode(nzcp_zkey* zk, int mode, nzcp_prover** out) {
  return api_guard([&] {
    if (!zk || !out) throw ApiError(NZCP_E_ARG, "null argument");
    if (mode != 0 && mode != 1) throw ApiError(NZCP_E_ARG, "prover mode must be 0 (latency) or 1 (throughput)");
    *out = nullptr;
    *out = prover_create_impl(zk, mode);
  });
}

void nzcp_prover_free(nzcp_prover* p) { prover_release(p); }

int nzcp_prove(nzcp_prover* p, const uint8_t* wtns, size_t wtns_len, const uint8_t* r, const uint8_t* s,
               nzcp_proof* proof, nzcp_prove_debug* dbg) {
  return api_guard([&] {
    if (!p || !wtns) throw ApiError(NZCP_E_ARG, "null argument");
    Sect sec[3];
    parse_bin(wtns, wtns_len, "wtns", sec, 2, 2);
    if (!sec[1].p || !sec[2].p || sec[1].len < 8) throw ApiError(NZCP_E_FORMAT, "wtns: missing section");
    uint32_t n8 = rd32u(sec[1].p);
    if (n8 != 32 || sec[1].len != 4 + 32 + 4 || memcmp(sec[1].p + 4, kRBytes, 32) != 0)
      throw ApiError(NZCP_E_CURVE, "Curve of the witness does not match the curve of the proving key");
    uint32_t nw = rd32u(sec[1].p + 36);
    if (nw != p->zk->n_vars)
      throw ApiError(NZCP_E_WITNESS_LEN, "Invalid witness length. Circuit: " + std::to_string(p->zk->n_vars) +
                                             ", witness: " + std::to_string(nw));
    if (sec[2].len != (uint64_t)nw * 32) throw ApiError(NZCP_E_FORMAT, "wtns: section 2 size mismatch");
    prove_impl(p, sec[2].p, nullptr, r, s, proof, dbg);
  });
}

int nzcp_prove_witness(nzcp_prover* p, const uint8_t* witness, uint32_t n_witness, const uint8_t* r, const uint8_t* s,
                       nzcp_proof* proof, nzcp_prove_debug* dbg) {
  return api_guard([&] {
    if (!p || !witness) throw ApiError(NZCP_E_ARG, "null argument");
    if (n_witness != p->zk->n_vars)
      throw ApiError(NZCP_E_WITNESS_LEN, "Invalid witness length. Circuit: " + std::to_string(p->zk->n_vars) +
                                             ", witness: " + std::to_string(n_witness));
    prove_impl(p, witness, nullptr, r, s, proof, dbg);
  });
}

int nzcp_prove_device(nzcp_prover* p, const void* d_witness, const uint8_t* r, const uint8_t* s, nzcp_proof* proof,
                      nzcp_prove_debug* dbg) {
  return api_guard([&] {
    if (!p || !d_witness) throw ApiError(NZCP_E_ARG, "null argument");
    prove_impl(p, nullptr, reinterpret_cast<const Fr*>(d_witness), r, s, proof, dbg);
  });
}

void* nzcp_prover_witness_buffer(nzcp_prover* p) { return p ? p->d_wtns : nullptr; }

uint64_t nzcp_prover_launch_count(const nzcp_prover* p) { return p ? p->launches.load() : g_launch_count.load(); }

int nzcp_prove_batch(nzcp_zkey* zk, const uint8_t* const* wtns, const size_t* wtns_len, size_t n_proofs, const uint8_t* r,
                     const uint8_t* s, nzcp_proof* proofs, int n_provers, int* status) {
  return api_guard([&] {
    if (!zk || (n_proofs && (!wtns || !wtns_len || !proofs))) throw ApiError(NZCP_E_ARG, "null argument");
    if (n_provers < 1) n_provers = 3;
    if (n_provers > 16) n_provers = 16;   // a throughput-mode prover holds ~6 GB of scratch at the NZCP size
    if ((size_t)n_provers > n_proofs) n_provers = (int)(n_proofs ? n_proofs : 1);
    std::vector<nzcp_prover*> mine;
    {
      std::lock_guard<std::mutex> lk(zk->pool_mu);   // take provers out of the key's pool (created on first use)
      while ((int)mine.size() < n_provers && !zk->pool.empty()) {
        mine.push_back(zk->pool.back());
        zk->pool.pop_back();
      }
    }
    struct Return {
      nzcp_zkey* zk; std::vector<nzcp_prover*>* v;
      ~Return() { std::lock_guard<std::mutex> lk(zk->pool_mu); for (auto* p : *v) zk->pool.push_back(p); }
    } ret{zk, &mine};
    while ((int)mine.size() < n_provers) mine.push_back(prover_create_impl(zk, 1));   // throughput mode
    std::vector<int> codes(n_proofs, NZCP_OK);
    std::vector<std::string> msgs(n_provers);
    std::vector<std::thread> threads;
    for (int j = 0; j < n_provers; j++) {
      threads.emplace_back([&, j] {
        for (size_t i = j; i < n_proofs; i += n_provers) {
          int rc = nzcp_prove(mine[j], wtns[i], wtns_len[i], r ? r + 32 * i : nullptr, s ? s + 32 * i : nullptr, &proofs[i],
                              nullptr);
          codes[i] = rc;
          if (rc != NZCP_OK && msgs[j].empty()) msgs[j] = "proof " + std::to_string(i) + ": " + nzcp_last_error();
        }
      });
    }
    for (auto& t : threads) t.join();
    if (status) for (size_t i = 0; i < n_proofs; i++) status[i] = codes[i];
    for (size_t i = 0; i < n_proofs; i++)
      if (codes[i] != NZCP_OK) {
        std::string m;
        for (auto& x : msgs) if (!x.empty()) { m = x; break; }
        throw ApiError(codes[i], m);
      }
  });
}

}  // extern "C"
