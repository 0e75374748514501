// MSM plans: a base set made resident once, then any number of scalar vectors against it -- the stand-alone face of the
// prover's MSM machinery (msm.cu), and the per-rank half of the split MSM (BASELINE.json configs[4]).
//
// Replaces (upstream, not vendored: yarn.lock:408-416) ffjavascript src/engine_multiexp.js G1/G2.multiExpAffine.
// Two modes, same kernels:
//   fixed-base (mode 0)     the bases are expanded into the 2^(c w) window table once (what nzcp_zkey_load does for zkey
//                           sections 5-9); every run is then a single bucket problem.  Pays when the bases are reused.
//   variable-base (mode 1)  no table: entries index the raw bases, window w accumulates into its own bucket group, and
//                           the windows are folded by Horner at the end -- multiExpAffine's own contract (arbitrary
//                           bases per call), at one pass over the bases.  Building a table costs ~48 x one MSM, so a
//                           one-shot MSM belongs here.
// A run can leave its result in HBM as one XYZZ point (nzcp_msm_plan_run_partial): the ranks of a split MSM all-gather
// those 128 / 256 bytes over NCCL and nzcp_msm_sum_partials adds them on the GPU; nothing but the final affine point
// crosses to the host.
#include <chrono>
#include <memory>

#include "api_util.cuh"

using namespace nzcp;

struct nzcp_msm_plan {
  int device = 0;
  bool g2 = false;
  int mode = 0;
  size_t n_points = 0;
  void* d_bases = nullptr;    // mode 1: the raw bases stay resident; mode 0: freed after the table is built
  Fr* d_scalars = nullptr;
  cudaStream_t st = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  CudaResources res;          // st, ev0, ev1, d_scalars and the mode-1 bases
  MsmTable tab;
  MsmSort sort;
  MsmRun run;
};

namespace nzcp {

static void plan_release(nzcp_msm_plan* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  delete p;
}

static nzcp_msm_plan* plan_create_impl(const uint8_t* bases, size_t n_points, int g2, int window_bits, int mode, int device,
                                       float* build_ms) {
  if (mode != 0 && mode != 1) throw ApiError(NZCP_E_ARG, "msm plan mode must be 0 (fixed-base) or 1 (variable-base)");
  use_device(device);
  std::unique_ptr<nzcp_msm_plan, void (*)(nzcp_msm_plan*)> p(new nzcp_msm_plan(), plan_release);
  p->device = device;
  p->g2 = g2 != 0;
  p->mode = mode;
  p->n_points = n_points;
  const size_t bsz = g2 ? 128 : 64;
  const size_t np = n_points ? n_points : 1;
  int c = window_bits > 0 ? window_bits : (mode == 1 ? msm_pick_window_free(np) : msm_pick_window(np));
  if (mode == 1 && (size_t)msm_num_windows(c) << (c - 1) > ((size_t)1 << 19))
    throw ApiError(NZCP_E_ARG, "window size too large for the variable-base path (windows * 2^(c-1) must be <= 2^19)");
  p->st = p->res.stream();
  p->ev0 = p->res.event();
  p->ev1 = p->res.event();
  CudaResources staged;       // mode 0: the raw bases, freed as soon as the window table is built
  p->d_bases = (mode == 0 ? staged : p->res).device<unsigned char>(np * bsz);
  p->d_scalars = p->res.device<Fr>(np);
  const auto t0 = std::chrono::steady_clock::now();
  if (n_points) NZCP_CUDA(cudaMemcpyAsync(p->d_bases, bases, n_points * bsz, cudaMemcpyHostToDevice, p->st));
  try {
    if (mode == 0) {
      msm_table_create(&p->tab, p->d_bases, n_points, 0, p->g2, c, p->st);
      NZCP_CUDA(cudaStreamSynchronize(p->st));
      staged = CudaResources();
      p->d_bases = nullptr;
    } else {
      msm_table_view(&p->tab, p->d_bases, n_points, p->g2, c);
      NZCP_CUDA(cudaStreamSynchronize(p->st));
    }
    msm_sort_create(&p->sort, n_points, c, -1, mode == 1);
    msm_run_create(&p->run, &p->sort, p->g2);
  } catch (const CudaError&) {
    throw;
  } catch (const ApiError&) {
    throw;
  } catch (const std::runtime_error& e) {
    throw ApiError(NZCP_E_ARG, e.what());
  }
  if (build_ms) *build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return p.release();
}

// Upload the scalars, sort, accumulate, reduce; the digit sums are on their way to the host when this returns.
static void plan_enqueue(nzcp_msm_plan* p, const uint8_t* scalars, size_t n_scalars, bool finish_on_device) {
  if (n_scalars > p->n_points) throw ApiError(NZCP_E_ARG, "more scalars than bases in the plan");
  if (n_scalars && !scalars) throw ApiError(NZCP_E_ARG, "null argument");
  use_device(p->device);
  if (n_scalars) NZCP_CUDA(cudaMemcpyAsync(p->d_scalars, scalars, n_scalars * sizeof(Fr), cudaMemcpyHostToDevice, p->st));
  NZCP_CUDA(cudaEventRecord(p->ev0, p->st));
  msm_sort_launch(&p->sort, p->d_scalars, n_scalars, p->st);
  msm_run_launch(&p->run, &p->sort, &p->tab, p->st);
  if (finish_on_device) msm_run_finish_device(&p->run, p->st);
  NZCP_CUDA(cudaEventRecord(p->ev1, p->st));
}

static void plan_wait(nzcp_msm_plan* p, float* kernel_ms) {
  NZCP_CUDA(cudaStreamSynchronize(p->st));
  if (kernel_ms) NZCP_CUDA(cudaEventElapsedTime(kernel_ms, p->ev0, p->ev1));
  try {
    msm_sort_check(&p->sort);
  } catch (const std::runtime_error& e) {
    throw ApiError(NZCP_E_RANGE, e.what());
  }
}

}  // namespace nzcp

extern "C" {

int nzcp_msm_plan_create(const uint8_t* bases, size_t n_points, int g2, int window_bits, int mode, int device,
                         nzcp_msm_plan** out, float* build_ms) {
  return api_guard([&] {
    if (!out || (n_points && !bases)) throw ApiError(NZCP_E_ARG, "null argument");
    *out = nullptr;
    *out = plan_create_impl(bases, n_points, g2, window_bits, mode, device, build_ms);
  });
}

void nzcp_msm_plan_free(nzcp_msm_plan* p) { plan_release(p); }

int nzcp_msm_plan_run(nzcp_msm_plan* p, const uint8_t* scalars, size_t n_scalars, uint8_t* out, float* kernel_ms) {
  return api_guard([&] {
    if (!p || !out) throw ApiError(NZCP_E_ARG, "null argument");
    plan_enqueue(p, scalars, n_scalars, false);
    plan_wait(p, kernel_ms);
    if (p->g2) g2_to_plain_bytes(msm_run_finish_g2(&p->run), out); else g1_to_plain_bytes(msm_run_finish_g1(&p->run), out);
  });
}

/* Device time of the bucket accumulation (pair rounds + XYZZ kernel) of the plan's last run, CUDA events on its stream. */
int nzcp_msm_plan_accumulate_ms(const nzcp_msm_plan* p, float* ms) {
  return api_guard([&] {
    if (!p || !ms) throw ApiError(NZCP_E_ARG, "null argument");
    *ms = msm_run_accumulate_ms(&p->run);
  });
}

int nzcp_msm_plan_run_partial(nzcp_msm_plan* p, const uint8_t* scalars, size_t n_scalars, void* d_out, float* kernel_ms) {
  return api_guard([&] {
    if (!p || !d_out) throw ApiError(NZCP_E_ARG, "null argument");
    plan_enqueue(p, scalars, n_scalars, true);
    const size_t psz = p->g2 ? sizeof(G2XYZZ) : sizeof(G1XYZZ);
    NZCP_CUDA(cudaMemcpyAsync(d_out, p->run.result, psz, cudaMemcpyDeviceToDevice, p->st));
    plan_wait(p, kernel_ms);
  });
}

int nzcp_msm_sum_partials(const void* d_partials, size_t count, int g2, int device, uint8_t* out) {
  return api_guard([&] {
    if (!d_partials || !out || count == 0 || count > (1u << 20)) throw ApiError(NZCP_E_ARG, "bad argument");
    use_device(device);
    const size_t psz = g2 ? sizeof(G2XYZZ) : sizeof(G1XYZZ);
    CudaResources res;
    void* d_res = res.device<unsigned char>(psz);
    msm_sum_points(d_partials, (uint32_t)count, g2 != 0, d_res, 0);
    alignas(16) unsigned char host[sizeof(G2XYZZ)];
    NZCP_CUDA(cudaMemcpy(host, d_res, psz, cudaMemcpyDeviceToHost));
    if (g2) g2_to_plain_bytes(*reinterpret_cast<const G2XYZZ*>(host), out);
    else g1_to_plain_bytes(*reinterpret_cast<const G1XYZZ*>(host), out);
  });
}

/* One-shot variable-base MSM (ffjavascript multiExpAffine semantics): no window table.  ms[0] = host wall time of the
 * whole call (uploads, plan, kernels, result), ms[1] = kernel time (sort + accumulate + reduce, CUDA events). */
int nzcp_msm_var(const uint8_t* bases, const uint8_t* scalars, size_t n_points, int g2, int window_bits, int device,
                 uint8_t* out, float ms[2]) {
  return api_guard([&] {
    if (!out || (n_points && (!bases || !scalars))) throw ApiError(NZCP_E_ARG, "null argument");
    const auto t0 = std::chrono::steady_clock::now();
    std::unique_ptr<nzcp_msm_plan, void (*)(nzcp_msm_plan*)> p(plan_create_impl(bases, n_points, g2, window_bits, 1, device, nullptr),
                                                               plan_release);
    float kms = 0;
    plan_enqueue(p.get(), scalars, n_points, false);
    plan_wait(p.get(), &kms);
    if (g2) g2_to_plain_bytes(msm_run_finish_g2(&p->run), out); else g1_to_plain_bytes(msm_run_finish_g1(&p->run), out);
    if (ms) {
      ms[0] = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
      ms[1] = kms;
    }
  });
}

}  // extern "C"
