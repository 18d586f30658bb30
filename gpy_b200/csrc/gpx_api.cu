// gpx_api.cu — C ABI (include/gpx.h) and host orchestration of the exact-GP evaluation on one B200.
//
// One evaluation (= one GP.parameters_changed(), GPy/core/gp.py:269-282):
//   prep_x -> kbuild (Ky into the workspace S) -> unified blocked factor-and-invert sweep (S: lower = L, upper = U = L^-T)
//   -> t = U^T y, alpha = U t -> LAUUM K^-1 = U U^T with the fused gradient epilogue -> finalize (LML + gradient).
// Nothing of size N^2 crosses PCIe unless gpx_get asks for it.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "gpx_common.cuh"
#include "gpx_kernels.cuh"
#include "gpx_ctx.cuh"
#include "gpx_fine.cuh"

namespace gpx {
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
}  // namespace gpx

using namespace gpx;

#define GPX_CHECK(x)        \
  do {                      \
    int rc__ = (x);         \
    if (rc__ != 0) return rc__; \
  } while (0)
#define GPX_FAIL(msg)       \
  do {                      \
    gpx::set_error(msg);    \
    return -2;              \
  } while (0)


static void free_data(gpx_ctx* c) {
  double** ptrs[] = {&c->dX, &c->dXsT, &c->dsq, &c->dY, &c->dT, &c->dAlpha, &c->dUvPart, &c->S, &c->Pbuf, &c->Tm,
                     &c->Ldiag, &c->Dinv, &c->logdet_part, &c->partials, &c->Kinv, &c->staging};
  for (auto p : ptrs) {
    if (*p) cudaFree(*p);
    *p = nullptr;
  }
  c->staging_cap = 0;
  c->have_eval = false;
  c->have_kinv = false;
  for (double** mp : {&c->mXsT, &c->msq, &c->mpartials}) { if (*mp) cudaFree(*mp); *mp = nullptr; }
  c->m_cap = 0;
  c->m_pcap = 0;
  oz_planes_free(c->ozp[0]);
  oz_planes_free(c->ozp[1]);
  oz_planes_free(c->ozpA);
  oz_planes_free(c->ozpB);
  if (c->oz_tiles) cudaFree(c->oz_tiles);
  c->oz_tiles = nullptr;
  for (double** mp : {&c->dYres, &c->dTfw}) { if (*mp) cudaFree(*mp); *mp = nullptr; }
  c->oz_steps.clear();
  c->oz_ready = false;
  c->oz_lists_ready = false;
}

static long pick_nb(const gpx_ctx* c) {
  if (c->NB > 0) return std::min<long>(c->NB, c->Npad);
  const char* e = getenv("GPX_NB");
  if (e && atol(e) >= TILE && atol(e) % TILE == 0) return std::min<long>(atol(e), c->Npad);
  // measured with the chain schedule (profiles/r02s2_chain_ab.txt): N = 16384: 1024 (66.8 ms; 512: 76.3, 2048: 73.4);
  // N = 8192: 512 (12.65 vs 13.15 ms); N = 4096: 512 (3.27; 256: 3.80, 1024: 3.76); N = 512: one block (0.467 vs 0.506 ms)
  if (c->Npad > 8192) return 1024;
  if (c->Npad >= 2048) return 512;
  if (c->Npad <= 512) return c->Npad;
  return 256;
}

int gpx::fill_kp(KernParams& kp, int kind, int ard, int D, double variance, const double* ls) {
  if (kind < 0 || kind > 3) GPX_FAIL("unknown kernel kind");
  if (D < 1 || D > MAX_D) GPX_FAIL("input dimension must be in [1, 64]");
  if (!(variance > 0)) GPX_FAIL("variance must be positive");
  kp.kind = kind; kp.ard = ard ? 1 : 0; kp.D = D; kp.variance = variance;
  const int nl = ard ? D : 1;
  for (int q = 0; q < nl; q++) {
    if (!(ls[q] > 0)) GPX_FAIL("lengthscale must be positive");
    kp.ls[q] = ls[q];
  }
  for (int q = nl; q < MAX_D; q++) kp.ls[q] = 1.0;
  kp.inv_ls_iso = ard ? 1.0 : 1.0 / ls[0];
  return 0;
}

extern "C" {

const char* gpx_last_error(void) { return gpx::g_err.c_str(); }
const char* gpx_version(void) { return "gpx 0.2 (sm_100a: tcgen05 int8 digit-split GEMM + fp64 DMMA)"; }

int gpx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return -1; }
  return n;
}

int gpx_create(int device, gpx_ctx** out) {
  if (!out) GPX_FAIL("null out pointer");
  int n = 0;
  GPX_CUDA(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) GPX_FAIL("no such CUDA device");
  GPX_CUDA(cudaSetDevice(device));
  gpx_ctx* c = new gpx_ctx();
  c->device = device;
  int prio_lo = 0, prio_hi = 0;
  GPX_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  GPX_CUDA(cudaStreamCreateWithPriority(&c->st, cudaStreamNonBlocking, prio_lo));
  GPX_CUDA(cudaStreamCreateWithPriority(&c->st2, cudaStreamNonBlocking, prio_hi));
  // between the two: the big panel GEMM on st3 must not hold back the small launches of the diagonal-block chain on st2
  GPX_CUDA(cudaStreamCreateWithPriority(&c->st3, cudaStreamNonBlocking, prio_hi < prio_lo - 1 ? prio_hi + 1 : prio_hi));
  GPX_CUDA(cudaMalloc(&c->res, RES_CAP * sizeof(double)));
  GPX_CUDA(cudaMalloc(&c->info, sizeof(int)));
  GPX_CUDA(cudaMallocHost(&c->h_res, RES_CAP * sizeof(double)));
  GPX_CUDA(cudaMallocHost(&c->h_info, sizeof(int)));
  {   // keep freed temporaries of the stand-alone calls cached in the device's default pool
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t keep = 1ull << 30;   // up to 1 GiB stays cached; anything above goes back at the next synchronisation
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  GPX_CHECK(gemm_init());
  GPX_CHECK(oz_init());
  GPX_CHECK(fine_init());
  GPX_CUDA(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device));
  *out = c;
  return 0;
}

int gpx_destroy(gpx_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->st);
  dist_free(c);
  sparse_free(c);
  free_data(c);
  for (auto e : c->ev) cudaEventDestroy(e);
  for (auto e : c->sync_ev) cudaEventDestroy(e);
  if (c->st2) cudaStreamDestroy(c->st2);
  if (c->st3) cudaStreamDestroy(c->st3);
  if (c->ev_kfirst) cudaEventDestroy(c->ev_kfirst);
  if (c->res) cudaFree(c->res);
  if (c->dNoiseVec) cudaFree(c->dNoiseVec);
  if (c->dDnoise) cudaFree(c->dDnoise);
  if (c->mB) cudaFree(c->mB);
  if (c->mflag) cudaFree(c->mflag);
  if (c->info) cudaFree(c->info);
  if (c->h_res) cudaFreeHost(c->h_res);
  if (c->h_info) cudaFreeHost(c->h_info);
  cudaStreamDestroy(c->st);
  delete c;
  return 0;
}

int gpx_set_option(gpx_ctx* c, const char* name, int64_t value) {
  if (!c || !name) GPX_FAIL("null argument");
  if (!strcmp(name, "nb")) {
    if (value != 0 && (value < TILE || value % TILE)) GPX_FAIL("nb must be a multiple of 128");
    if (value != c->NB) {  // the panel buffers are sized by the block: force a re-allocation at the next gpx_set_data
      GPX_CUDA(cudaSetDevice(c->device));
      GPX_CUDA(cudaStreamSynchronize(c->st));
      free_data(c);
      c->Npad = 0;
    }
    c->NB = value;
    return 0;
  }
  if (!strcmp(name, "profile")) { c->profile = (int)value; return 0; }
  if (!strcmp(name, "ozaki")) { c->ozaki = value < 0 ? -1 : (value ? 1 : 0); return 0; }
  if (!strcmp(name, "oz_dig_up")) {
    if (value < 4 || value > OZ_S) GPX_FAIL("oz_dig_up must be in [4, 8]");
    c->oz_dig_up = (int)value;
    return 0;
  }
  if (!strcmp(name, "oz_ctas")) { c->oz_ctas = (int)std::max<int64_t>(0, value); return 0; }
  if (!strcmp(name, "oz_dbg")) { c->oz_dbg = (int)value; return 0; }
  if (!strcmp(name, "oz_tpc")) { c->oz_tpc = (int)std::max<int64_t>(0, value); return 0; }
  if (!strcmp(name, "oz_panel")) { c->oz_panel = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2)); return 0; }   // 2 = at every size
  if (!strcmp(name, "oz_sched")) { c->oz_sched = value ? 1 : 0; return 0; }
  if (!strcmp(name, "oz_u0")) { c->oz_u0 = value ? 1 : 0; return 0; }
  if (!strcmp(name, "oz_reserve")) { c->oz_reserve = (int)std::max<int64_t>(0, std::min<int64_t>(value, 64)); return 0; }
  if (!strcmp(name, "oz_wide")) {
    if ((value ? 1 : 0) != c->oz_wide && c->oz_ready) {   // the tile lists are per tile shape: rebuild at the next evaluation
      GPX_CUDA(cudaSetDevice(c->device));
      GPX_CUDA(cudaStreamSynchronize(c->st));
      if (c->oz_tiles) cudaFree(c->oz_tiles);
      c->oz_tiles = nullptr;
      c->oz_steps.clear();
      c->oz_lists_ready = false;
    }
    c->oz_wide = value ? 1 : 0;
    return 0;
  }
  if (!strcmp(name, "lookahead")) { c->lookahead = value ? 1 : 0; return 0; }
  if (!strcmp(name, "base")) { set_base_version((int)std::max<int64_t>(0, std::min<int64_t>(value, 5))); return 0; }
  if (!strcmp(name, "base_prof")) return set_base_prof((int)value);
  if (!strcmp(name, "base_pdl")) { set_base_pdl((int)value); return 0; }
  if (!strcmp(name, "fine")) { c->fine = value ? 1 : 0; return 0; }
  if (!strcmp(name, "chain")) { c->chain = value ? 1 : 0; return 0; }
  GPX_FAIL("unknown option");
}

int gpx_set_data(gpx_ctx* c, const double* X, int64_t N, int D, const double* Y, int P) {
  if (!c || !X || !Y) GPX_FAIL("null argument");
  if (N < 1) GPX_FAIL("N must be positive");
  if (D < 1 || D > MAX_D) GPX_FAIL("input dimension must be in [1, 64]");
  if (P < 1 || P > MAX_P) GPX_FAIL("number of output columns must be in [1, 8]");
  GPX_CUDA(cudaSetDevice(c->device));
  if (c->dist) return dist_set_data(c, X, N, D, Y, P);
  const long Npad = (N + TILE - 1) / TILE * TILE;
  if (Npad != c->Npad || D != c->D || P != c->P) {
    GPX_CUDA(cudaStreamSynchronize(c->st));
    free_data(c);
    c->Npad = Npad; c->D = D; c->P = P;
    const long nt = Npad / TILE;
    const long NB = pick_nb(c);
    GPX_CUDA(cudaMalloc(&c->dX, (size_t)Npad * D * 8));
    GPX_CUDA(cudaMalloc(&c->dXsT, (size_t)Npad * D * 8));
    GPX_CUDA(cudaMalloc(&c->dsq, (size_t)Npad * 8));
    GPX_CUDA(cudaMalloc(&c->dY, (size_t)Npad * P * 8));
    GPX_CUDA(cudaMalloc(&c->dT, (size_t)Npad * P * 8));
    GPX_CUDA(cudaMalloc(&c->dAlpha, (size_t)Npad * P * 8));
    GPX_CUDA(cudaMalloc(&c->dUvPart, (size_t)KSPLIT * Npad * P * 8));
    GPX_CUDA(cudaMalloc(&c->S, (size_t)Npad * Npad * 8));
    GPX_CUDA(cudaMalloc(&c->Pbuf, (size_t)2 * Npad * NB * 8));   // double-buffered for the look-ahead
    GPX_CUDA(cudaMalloc(&c->Tm, (size_t)NB * NB * 8));
    GPX_CUDA(cudaMalloc(&c->Ldiag, (size_t)Npad * TILE * 8));
    GPX_CUDA(cudaMalloc(&c->Dinv, (size_t)Npad * TILE * 8));
    GPX_CUDA(cudaMalloc(&c->logdet_part, (size_t)nt * 8));
    GPX_CUDA(cudaMalloc(&c->partials, (size_t)nt * nt * (MAX_D + 2) * 8));
  }
  c->N = N;
  c->have_eval = false;
  c->have_kinv = false;
  // X: keep the caller's row-major layout on device; Y: SoA [P][Npad] zero padded (staged through dT)
  GPX_CUDA(cudaMemcpyAsync(c->dX, X, (size_t)N * D * 8, cudaMemcpyHostToDevice, c->st));
  GPX_CUDA(cudaMemcpyAsync(c->dT, Y, (size_t)N * P * 8, cudaMemcpyHostToDevice, c->st));
  GPX_CHECK(launch_transpose_pad(c->dT, N, P, Npad, c->dY, c->st));
  c->total_launches += 1;
  GPX_CUDA(cudaStreamSynchronize(c->st));
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// event helpers for per-phase accounting on the launching stream
// ---------------------------------------------------------------------------------------------------------------
struct EvSpan { int a, b; int phase; double flops; };
enum { PH_KBUILD = 0, PH_SWEEP = 1, PH_UPDATE = 2, PH_LAUUM = 3, PH_SOLVE = 4, PH_TOTAL = 5 };

static int ev_get(gpx_ctx* c, size_t idx, cudaEvent_t* out) {
  while (c->ev.size() <= idx) {
    cudaEvent_t e;
    GPX_CUDA(cudaEventCreate(&e));
    c->ev.push_back(e);
  }
  *out = c->ev[idx];
  return 0;
}

struct Recorder {
  gpx_ctx* c;
  std::vector<EvSpan> spans;
  size_t next = 0;
  int begin(int phase, double flops = 0) {
    if (!c->profile && phase != PH_TOTAL) return -1;
    cudaEvent_t e;
    if (ev_get(c, next, &e)) return -1;
    cudaEventRecord(e, c->st);
    spans.push_back({(int)next, -1, phase, flops});
    next++;
    return (int)spans.size() - 1;
  }
  void end(int h) {
    if (h < 0) return;
    cudaEvent_t e;
    if (ev_get(c, next, &e)) return;
    cudaEventRecord(e, c->st);
    spans[h].b = (int)next;
    next++;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// the unified blocked factor-and-invert sweep
// ---------------------------------------------------------------------------------------------------------------
GemmParams gpx::gemm_defaults() {
  GemmParams p;
  memset(&p, 0, sizeof(p));
  return p;
}

static int sync_event(gpx_ctx* c, size_t idx, cudaEvent_t* out) {
  while (c->sync_ev.size() <= idx) {
    cudaEvent_t e;
    GPX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->sync_ev.push_back(e);
  }
  *out = c->sync_ev[idx];
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// tcgen05 / Ozaki path: tile lists and buffers for (Npad, NB)
// ---------------------------------------------------------------------------------------------------------------
static bool oz_wanted(const gpx_ctx* c) {
  if (c->dist) return false;
  int on = c->ozaki;
  if (on < 0) { const char* e = getenv("GPX_OZAKI"); on = e ? atoi(e) : 1; }
  if (!on) return false;
  const long NB = pick_nb(c);
  // wherever there are at least two panels (measured faster than the DMMA path from N = 700 up: 0.97 vs 1.03 ms at 700,
  // 5.3 vs 5.9 ms at 4096, 64 vs 142 ms at 16384); a single-block matrix has no panel and stays on the DMMA path
  return c->Npad >= 2 * NB && NB % OZ_KC == 0;
}

static int oz_prepare(gpx_ctx* c) {
  const long Npad = c->Npad, NB = pick_nb(c);
  const int nt = (int)(Npad / TILE);
  if (nt >= 4096) GPX_FAIL("matrix too large for the tile encoding");
  if (!c->oz_ready) {
    GPX_CHECK(oz_planes_alloc(c->ozp[0], Npad, NB));
    GPX_CHECK(oz_planes_alloc(c->ozp[1], Npad, NB));
    GPX_CHECK(oz_planes_alloc(c->ozpA, Npad, NB));
    GPX_CHECK(oz_planes_alloc(c->ozpB, NB, NB));
    if (!c->Kinv) GPX_CUDA(cudaMalloc(&c->Kinv, (size_t)Npad * Npad * 8));
    GPX_CUDA(cudaMalloc(&c->dYres, (size_t)MAX_P * Npad * 8));
    GPX_CUDA(cudaMalloc(&c->dTfw, (size_t)MAX_P * Npad * 8));
    c->oz_ready = true;
    c->oz_lists_ready = false;
  }
  if (c->oz_lists_ready) return 0;
  std::vector<uint32_t> tiles;
  oz_build_lists(Npad, NB, c->oz_wide ? 1 : 2, 1, 0, tiles, c->oz_steps);
  GPX_CUDA(cudaMalloc(&c->oz_tiles, tiles.size() * sizeof(uint32_t)));
  GPX_CUDA(cudaMemcpy(c->oz_tiles, tiles.data(), tiles.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  c->oz_lists_ready = true;
  return 0;
}

// Step k of the sweep (block column k of width nb):
//   D(k)  inner sweep of the diagonal block (128 columns at a time) + assemble of U_kk / Linv_kk      [side stream]
//   Pn(k) panel GEMM  P = S(:,block k) Linv_kk^T -> Pbuf[k&1], copied back into S                     [side stream]
//   U1(k) trailing update restricted to the columns of block k+1                                        [main stream]
//   U2(k) trailing update of the remaining columns                                                      [main stream]
// Look-ahead: D(k+1), Pn(k+1) only need U1(k), so they run on the high-priority side stream while U2(k) keeps the
// machine busy; U1(k+1) waits for Pn(k+1). Without look-ahead everything is issued on the main stream.
// oz: 0 = DMMA updates; 1 = trailing update on tcgen05 (Ozaki split); 2 = that + K^-1 = U U^T accumulated into c->Kinv
// panel by panel inside the same launches (the panel's digit planes serve both)
static int run_sweep_chain(gpx_ctx* c, Recorder& rec);

static int run_sweep(gpx_ctx* c, Recorder& rec, int oz = 0) {
  const long ld = c->Npad, Npad = c->Npad;
  const int nt = (int)(Npad / TILE);
  const long NB = pick_nb(c);
  const bool la = c->lookahead && NB < Npad;
  if (oz >= 2 && la && c->chain && !c->oz_sched) return run_sweep_chain(c, rec);
  cudaStream_t sm = c->st;
  cudaStream_t ss = la ? c->st2 : c->st;
  size_t evi = 0;
  cudaEvent_t ev, u1_done = nullptr;
  bool u1_pending = false;
  if (la) {  // side stream starts after everything queued so far on the main stream (K build)
    GPX_CHECK(sync_event(c, evi++, &ev));
    GPX_CUDA(cudaEventRecord(ev, sm));
    GPX_CUDA(cudaStreamWaitEvent(ss, ev, 0));
  }
  if (oz >= 2)   // forward substitution t = L^-1 y rides along on the side stream (see fw_block_kernel)
    GPX_CUDA(cudaMemcpyAsync(c->dYres, c->dY, (size_t)c->P * Npad * 8, cudaMemcpyDeviceToDevice, ss));
  int kblk = 0;
  for (long o = 0; o < Npad; o += NB, kblk++) {
    const long nb = std::min(NB, Npad - o);
    const int nbt = (int)(nb / TILE), kt0 = (int)(o / TILE), kt1 = kt0 + nbt;
    double* Sblk = c->S + o + o * ld;
    double* Pb = c->Pbuf + (size_t)(kblk & 1) * Npad * NB;
    // ---- D(k): inner sweep of the nb x nb diagonal block ------------------------------------------------------
    GPX_CHECK(diag_block_sweep(c, Sblk, ld, nbt, kt0, ss));
    if (nbt == nt) break;  // single block: done
    // tcgen05 schedule (option "oz_sched", default): the persistent U2(k-1) leaves a few SMs free, on which the serial
    // diagonal-block chain D(k) runs meanwhile (side stream); the panel GEMM Pn(k), which needs the whole machine for half a
    // millisecond, is queued on the MAIN stream behind U2(k-1) instead of fighting it for SM slots.
    if (u1_pending) {   // (oz_u0) the panel of this step needs ALL of its block column updated, not only the diagonal block
      GPX_CUDA(cudaStreamWaitEvent(ss, u1_done, 0));
      u1_pending = false;
    }
    const bool sched2 = oz && la && c->oz_sched;
    cudaStream_t sp = sched2 ? sm : ss;   // stream of assemble / panel / split
    if (sched2) {
      GPX_CHECK(sync_event(c, evi++, &ev));
      GPX_CUDA(cudaEventRecord(ev, ss));
      GPX_CUDA(cudaStreamWaitEvent(sm, ev, 0));
    }
    // ---- Pn(k): P = S(:, block) * Linv_kk^T; rows of the diagonal block get U_kk ------------------------------
    GPX_CHECK(launch_assemble(Sblk, ld, (int)nb, Pb + o, Npad, c->Tm, sp));
    c->eval_launches++;
    {
      GemmParams pp = gemm_defaults();
      pp.mode = GEMM_PANEL;
      pp.A = c->S + o * ld; pp.lda = ld;
      pp.B = c->Tm; pp.ldb = nb;
      pp.C = Pb; pp.ldc = Npad;
      pp.K = (int)nb; pp.nt = nt; pp.skip0 = kt0; pp.skip1 = kt1; pp.tri = 1;
      GPX_CHECK(launch_gemm(pp, dim3(nbt, nt - nbt), sp));
      c->eval_launches++;
    }
    auto copy_back = [&]() -> int {   // the panel rows take their final place in S (U block column above, L panel below)
      if (o > 0)
        GPX_CUDA(cudaMemcpy2DAsync(c->S + o * ld, ld * 8, Pb, Npad * 8, (size_t)o * 8, nb, cudaMemcpyDeviceToDevice, ss));
      if (kt1 < nt)
        GPX_CUDA(cudaMemcpy2DAsync(c->S + o * ld + (o + nb), ld * 8, Pb + (o + nb), Npad * 8,
                                   (size_t)(Npad - o - nb) * 8, nb, cudaMemcpyDeviceToDevice, ss));
      return 0;
    };
    // DMMA updates read the panel from Pb, tcgen05 updates from the digit planes: either way nothing on the main stream
    // reads block column k of S, so on the tcgen05 path the copy-back leaves the critical chain (after the hand-over)
    if (!oz) GPX_CHECK(copy_back());
    if (oz) {   // digit planes + row exponents of this panel (all rows: U block column | U_kk | Cholesky panel)
      GPX_CHECK(launch_oz_split(Pb, Npad, nb, c->ozp[kblk & 1], sp));
      c->eval_launches++;
    }
    if (sched2) {          // the side stream (copy-back, forward substitution, later D(k+1)) continues after the panel
      GPX_CHECK(sync_event(c, evi++, &ev));
      GPX_CUDA(cudaEventRecord(ev, sm));
      GPX_CUDA(cudaStreamWaitEvent(ss, ev, 0));
    } else if (la) {
      GPX_CHECK(sync_event(c, evi++, &ev));
      GPX_CUDA(cudaEventRecord(ev, ss));
      GPX_CUDA(cudaStreamWaitEvent(sm, ev, 0));
    }
    if (oz) GPX_CHECK(copy_back());
    if (oz >= 2) {   // after the hand-over to the main stream: overlaps U1(k); the panel buffer is not reused before step k+2
      GPX_CHECK(launch_fw_block(c->Tm, (int)nb, c->dYres + o, Npad, c->P, c->dTfw + o, ss));
      GPX_CHECK(launch_fw_panel(Pb + (o + nb), Npad, Npad - o - nb, (int)nb, c->dTfw + o, Npad, c->P, c->dYres + (o + nb), ss));
      c->eval_launches += 2;
    }
    // ---- trailing update: S(r,c) -= P_r P_c^T for c >= kt1, r in [0,kt1) U [c,nt), split U1 | U2 ---------------
    if (oz) {
      const gpx_ctx::OzStep& os = c->oz_steps[kblk];
      const OzPlanes& pl = c->ozp[kblk & 1];
      // U0 (next diagonal block) | U1 (rest of block column k+1) | U2 (everything else + K^-1 tiles). With option oz_u0 = 0
      // U0 and U1 are one launch (their lists are adjacent).
      const bool u0 = c->oz_u0 && la && os.u0_n > 0;
      for (int part = u0 ? -1 : 0; part < 2; part++) {
        const int off = part < 0 ? os.u0_off : (part == 0 ? (u0 ? os.u1_off : os.u0_off) : os.u2_off);
        const int ntl = part < 0 ? os.u0_n : (part == 0 ? (u0 ? os.u1_n : os.u0_n + os.u1_n) : (oz >= 2 ? os.u2_n : os.u2_upd));
        if (ntl > 0) {
          OzParams op;
          memset(&op, 0, sizeof(op));
          op.tiles = c->oz_tiles + off; op.ntiles = ntl; op.nkc = (int)(nb / OZ_KC);
          op.scale = pl.scale; op.S = c->S; op.lds = ld; op.Kinv = c->Kinv; op.ldk = ld;
          op.dig_lo = OZ_S; op.dig_up = c->oz_dig_up; op.dbg = c->oz_dbg; op.wide = c->oz_wide;
          op.tpc = c->oz_ctas > 0 ? (ntl + c->oz_ctas - 1) / c->oz_ctas : c->oz_tpc;
          if (sched2 && c->oz_ctas <= 0 && c->oz_tpc <= 0) {
            // persistent: U1 on every SM (nothing else can run before it is done), U2 on all but the reserved SMs
            const int ctas = std::max(1, c->num_sms - (part == 1 ? c->oz_reserve : 0));   // (part <= 0: every SM)
            op.tpc = (ntl + ctas - 1) / ctas;
          }
          const int tn = c->oz_wide ? 2 * OZ_TN : OZ_TN;
          const double flops = (double)ntl * 2.0 * OZ_TM * tn * (double)nb;
          const int nup = part < 0 ? 0 : (part == 0 ? os.u1_up : (oz >= 2 ? os.u2_up : os.u2_upd_up));
          const int du = c->oz_dig_up;
          c->stats.update_int8_ops += ((double)nup * (du * (du + 1) / 2) + (double)(ntl - nup) * (OZ_S * (OZ_S + 1) / 2)) * 2.0 *
                                      OZ_TM * tn * (double)nb;
          const int h = rec.begin(PH_UPDATE, flops);
          GPX_CHECK(launch_oz_gemm(pl, op, c->num_sms, sm));
          rec.end(h);
          c->eval_launches++;
          c->stats.update_launches++;
        }
        if (la && kt1 < nt && part == (u0 ? -1 : 0)) {   // the next diagonal block is final: D(k+1) may start on the side stream
          GPX_CHECK(sync_event(c, evi++, &ev));
          GPX_CUDA(cudaEventRecord(ev, sm));
          GPX_CUDA(cudaStreamWaitEvent(ss, ev, 0));
        }
        if (u0 && part == 0 && kt1 < nt) {               // block column k+1 is final: the panel GEMM of step k+1 may read it
          GPX_CHECK(sync_event(c, evi++, &u1_done));
          GPX_CUDA(cudaEventRecord(u1_done, sm));
          u1_pending = true;
        }
      }
    } else if (kt1 < nt) {
      const int next_nbt = (int)(std::min(NB, Npad - (o + nb)) / TILE);
      for (int part = 0; part < 2; part++) {
        const int cbeg = part == 0 ? kt1 : kt1 + next_nbt;
        const int cend = part == 0 ? kt1 + next_nbt : nt;
        if (cbeg < cend) {
          GemmParams pu = gemm_defaults();
          pu.mode = GEMM_UPDATE;
          pu.A = Pb; pu.lda = Npad;
          pu.B = Pb; pu.ldb = Npad;
          pu.C = c->S; pu.ldc = ld;
          pu.K = (int)nb; pu.nt = nt; pu.c0 = cbeg; pu.ncols = cend - cbeg; pu.rlow = kt1;
          double tiles = 0;
          for (int cc = cbeg; cc < cend; cc++) tiles += kt1 + (nt - cc);
          const double flops = tiles * 2.0 * TILE * TILE * (double)nb;
          const int h = rec.begin(PH_UPDATE, flops);
          GPX_CHECK(launch_gemm(pu, dim3(1, 1), sm));
          rec.end(h);
          c->eval_launches++;
          c->stats.update_launches++;
        }
        if (part == 0 && la) {  // block column k+1 is final: the side stream may start D(k+1)
          GPX_CHECK(sync_event(c, evi++, &ev));
          GPX_CUDA(cudaEventRecord(ev, sm));
          GPX_CUDA(cudaStreamWaitEvent(ss, ev, 0));
        }
      }
    }
  }
  if (la) {  // join: the main stream continues after the last side-stream work
    GPX_CHECK(sync_event(c, evi++, &ev));
    GPX_CUDA(cudaEventRecord(ev, ss));
    GPX_CUDA(cudaStreamWaitEvent(sm, ev, 0));
  }
  return 0;
}

// The tcgen05 sweep with the serial chain on its own stream (option "chain", default). Per step k:
//   side stream  ss : D(k) -> assemble -> Pc(k): panel rows of block k+1 (fine DMMA tiles) -> U0d(k): diagonal block k+1 -= Pc Pc^T
//                     (fine DMMA tiles, fp64 operands straight from the panel buffer) -> D(k+1) ...
//   third stream s3 : Pr(k): the other panel rows -> digit split of the whole panel -> copy-back -> forward substitution
//   main stream  sm : U1(k): rest of block column k+1 -> U2(k): everything else + the K^-1 tiles          (tcgen05)
// Dependences across streams (events):  Pc(k), Pr(k) read block column k: after U1(k-1);  U0d(k) touches tiles that U2(k-1)
// updates: after U2(k-1);  split(k) after Pc(k);  U1(k) after split(k);  assemble(k+1) overwrites Tm and, with Pc/Pr(k+1), the
// panel buffer of step k-1: after the forward-substitution block of step k on s3 (s3 runs in order, so everything of step
// k-1 there is done as well);  the digit planes of step k are those of step k-2: split(k) is behind Pr(k), which waits for
// U1(k-1), which is behind U2(k-2) on the main stream.
// What the next diagonal block waits for is therefore D(k) + two small launches instead of D(k) + full panel + split + a
// tcgen05 launch, and the main stream never waits for a diagonal block unless the trailing update is shorter than D.
static int run_sweep_chain(gpx_ctx* c, Recorder& rec) {
  const long ld = c->Npad, Npad = c->Npad;
  const int nt = (int)(Npad / TILE);
  const long NB = pick_nb(c);
  cudaStream_t sm = c->st, ss = c->st2, s3 = c->st3;
  size_t evi = 0;
  cudaEvent_t ev, ev_u1 = nullptr, ev_u2 = nullptr, ev_fw = nullptr;
  auto link = [&](cudaStream_t from, cudaStream_t to, cudaEvent_t* keep) -> int {   // `to` continues after what `from` holds now
    cudaEvent_t e;
    GPX_CHECK(sync_event(c, evi++, &e));
    GPX_CUDA(cudaEventRecord(e, from));
    if (to) GPX_CUDA(cudaStreamWaitEvent(to, e, 0));
    if (keep) *keep = e;
    return 0;
  };
  GPX_CHECK(link(sm, s3, &ev));                      // K build (all of it); it also stands in for "U1(-1)": block column 0 is final
  if (c->kfirst_valid) GPX_CUDA(cudaStreamWaitEvent(ss, c->ev_kfirst, 0));   // D(0) needs the first block row only
  else GPX_CUDA(cudaStreamWaitEvent(ss, ev, 0));
  ev_u1 = ev;
  GPX_CUDA(cudaMemcpyAsync(c->dYres, c->dY, (size_t)c->P * Npad * 8, cudaMemcpyDeviceToDevice, s3));
  int kblk = 0;
  for (long o = 0; o < Npad; o += NB, kblk++) {
    const long nb = std::min(NB, Npad - o);
    const int nbt = (int)(nb / TILE), kt0 = (int)(o / TILE), kt1 = kt0 + nbt;
    const int next_nbt = kt1 < nt ? (int)(std::min(NB, Npad - (o + nb)) / TILE) : 0;
    double* Sblk = c->S + o + o * ld;
    double* Pb = c->Pbuf + (size_t)(kblk & 1) * Npad * NB;
    const gpx_ctx::OzStep& os = c->oz_steps[kblk];
    const OzPlanes& pl = c->ozp[kblk & 1];
    // ---- ss: D(k), assemble ------------------------------------------------------------------------------------------
    GPX_CHECK(diag_block_sweep(c, Sblk, ld, nbt, kt0, ss));
    if (ev_fw) GPX_CUDA(cudaStreamWaitEvent(ss, ev_fw, 0));
    GPX_CHECK(launch_assemble(Sblk, ld, (int)nb, Pb + o, Npad, c->Tm, ss));
    c->eval_launches++;
    cudaEvent_t ev_asm, ev_pc = nullptr;
    GPX_CHECK(link(ss, s3, &ev_asm));
    if (ev_u1) { GPX_CUDA(cudaStreamWaitEvent(ss, ev_u1, 0)); GPX_CUDA(cudaStreamWaitEvent(s3, ev_u1, 0)); }
    // ---- ss: Pc(k), U0d(k) -------------------------------------------------------------------------------------------
    if (next_nbt > 0) {
      FineParams pc{};
      pc.mode = FINE_PANEL;
      pc.A = c->S + o * ld; pc.lda = ld;
      pc.B = c->Tm; pc.ldb = nb;
      pc.C = Pb; pc.ldc = Npad;
      pc.K = (int)nb; pc.r0 = kt1; pc.nr = next_nbt; pc.nc = nbt; pc.tri = 1;
      GPX_CHECK(launch_fine(pc, ss));
      c->eval_launches++;
      GPX_CHECK(link(ss, nullptr, &ev_pc));
      if (ev_u2) GPX_CUDA(cudaStreamWaitEvent(ss, ev_u2, 0));
      FineParams pu{};
      pu.mode = FINE_UPDATE;
      pu.A = Pb; pu.lda = Npad;
      pu.B = Pb; pu.ldb = Npad;
      pu.C = c->S; pu.ldc = ld;
      pu.K = (int)nb; pu.nt = kt1 + next_nbt; pu.c0 = kt1; pu.ncols = next_nbt; pu.rlow = 0;
      GPX_CHECK(launch_fine(pu, ss));
      c->eval_launches++;
    }
    // ---- s3: Pr(k), split, copy-back, forward substitution --------------------------------------------------------------
    // (measured, profiles/r02s2_panel_ab.txt: +3.8 % at N = 16384, +3.1 % at 8192, even at 4096, -7 % at 1300: five launches
    // instead of one only pay once the panel GEMM is a visible share of the step)
    const bool oz_pan = c->oz_panel && c->oz_wide && os.pan_n > 0 && (c->oz_panel > 1 || Npad >= 4096);
    if (oz_pan) {
      // the panel GEMM itself on the tensor cores: digit planes of block column k of the workspace (A) and of L_kk^-1 (B,
      // lower triangular: per-tile k-range), P = A B^T stored into the panel buffer. 8 digits for the Cholesky rows (they feed
      // the log-determinant), oz_dig_up for the rows above (finished block column of U: gradients only)
      GPX_CHECK(launch_oz_split(c->S + o * ld, ld, nb, c->ozpA, s3));
      GPX_CHECK(launch_oz_split(c->Tm, nb, nb, c->ozpB, s3));
      OzParams op;
      memset(&op, 0, sizeof(op));
      op.tiles = c->oz_tiles + os.pan_off; op.ntiles = os.pan_n; op.nkc = (int)(nb / OZ_KC);
      op.scale = c->ozpA.scale; op.scaleB = c->ozpB.scale; op.P = Pb; op.ldp = Npad; op.Pfinal = c->S + o * ld;
      op.S = c->S; op.lds = ld; op.Kinv = c->Kinv; op.ldk = ld;
      op.dig_lo = OZ_S; op.dig_up = c->oz_dig_up; op.dbg = c->oz_dbg; op.wide = 1;
      op.tpc = c->oz_ctas > 0 ? (os.pan_n + c->oz_ctas - 1) / c->oz_ctas : c->oz_tpc;
      GPX_CHECK(launch_oz_gemm(c->ozpA, op, c->num_sms, s3, &c->ozpB));
      c->eval_launches += 5;
    } else if (nt - nbt - next_nbt > 0) {
      GemmParams pp = gemm_defaults();
      pp.mode = GEMM_PANEL;
      pp.A = c->S + o * ld; pp.lda = ld;
      pp.B = c->Tm; pp.ldb = nb;
      pp.C = Pb; pp.ldc = Npad;
      pp.K = (int)nb; pp.nt = nt; pp.skip0 = kt0; pp.skip1 = kt1 + next_nbt; pp.tri = 1;
      GPX_CHECK(launch_gemm(pp, dim3(nbt, nt - nbt - next_nbt), s3));
      c->eval_launches++;
    }
    if (ev_pc) GPX_CUDA(cudaStreamWaitEvent(s3, ev_pc, 0));
    GPX_CHECK(launch_oz_split(Pb, Npad, nb, c->ozp[kblk & 1], s3));
    c->eval_launches++;
    GPX_CHECK(link(s3, sm, nullptr));
    if (oz_pan) {   // the tensor-core panel GEMM stored its rows into the workspace itself: only the rows of block k+1 (Pc) are left
      if (next_nbt > 0)
        GPX_CUDA(cudaMemcpy2DAsync(c->S + o * ld + (o + nb), ld * 8, Pb + (o + nb), Npad * 8, (size_t)next_nbt * TILE * 8, nb,
                                   cudaMemcpyDeviceToDevice, s3));
    } else {
      if (o > 0)
        GPX_CUDA(cudaMemcpy2DAsync(c->S + o * ld, ld * 8, Pb, Npad * 8, (size_t)o * 8, nb, cudaMemcpyDeviceToDevice, s3));
      if (kt1 < nt)
        GPX_CUDA(cudaMemcpy2DAsync(c->S + o * ld + (o + nb), ld * 8, Pb + (o + nb), Npad * 8, (size_t)(Npad - o - nb) * 8, nb,
                                   cudaMemcpyDeviceToDevice, s3));
    }
    GPX_CHECK(launch_fw_block(c->Tm, (int)nb, c->dYres + o, Npad, c->P, c->dTfw + o, s3));
    c->eval_launches++;
    GPX_CHECK(link(s3, nullptr, &ev_fw));
    GPX_CHECK(launch_fw_panel(Pb + (o + nb), Npad, Npad - o - nb, (int)nb, c->dTfw + o, Npad, c->P, c->dYres + (o + nb), s3));
    c->eval_launches++;
    // ---- sm: U1(k), U2(k) on the tcgen05 tensor cores ---------------------------------------------------------------------
    for (int part = 0; part < 2; part++) {
      const int off = part == 0 ? os.u1_off : os.u2_off;
      const int ntl = part == 0 ? os.u1_n : os.u2_n;
      if (ntl > 0) {
        OzParams op;
        memset(&op, 0, sizeof(op));
        op.tiles = c->oz_tiles + off; op.ntiles = ntl; op.nkc = (int)(nb / OZ_KC);
        op.scale = pl.scale; op.S = c->S; op.lds = ld; op.Kinv = c->Kinv; op.ldk = ld;
        op.dig_lo = OZ_S; op.dig_up = c->oz_dig_up; op.dbg = c->oz_dbg; op.wide = c->oz_wide;
        op.tpc = c->oz_ctas > 0 ? (ntl + c->oz_ctas - 1) / c->oz_ctas : c->oz_tpc;
        const int tn = c->oz_wide ? 2 * OZ_TN : OZ_TN;
        const double flops = (double)ntl * 2.0 * OZ_TM * tn * (double)nb;
        const int nup = part == 0 ? os.u1_up : os.u2_up;
        const int du = c->oz_dig_up;
        c->stats.update_int8_ops += ((double)nup * (du * (du + 1) / 2) + (double)(ntl - nup) * (OZ_S * (OZ_S + 1) / 2)) * 2.0 *
                                    OZ_TM * tn * (double)nb;
        const int h = rec.begin(PH_UPDATE, flops);
        GPX_CHECK(launch_oz_gemm(pl, op, c->num_sms, sm));
        rec.end(h);
        c->eval_launches++;
        c->stats.update_launches++;
      }
      GPX_CHECK(link(sm, nullptr, part == 0 ? &ev_u1 : &ev_u2));
    }
  }
  GPX_CHECK(link(ss, sm, nullptr));
  GPX_CHECK(link(s3, sm, nullptr));
  return 0;
}

// plain: store K^-1 (lower tiles) only, no gradient reductions (composite kernels reduce from the stored matrix)
static int run_lauum(gpx_ctx* c, double* kinv_out, Recorder* rec, bool plain = false) {
  const long ld = c->Npad;
  const int nt = (int)(c->Npad / TILE);
  const int nl = c->kp.ard ? c->D : 1;
  GPX_CUDA(cudaMemsetAsync(c->partials, 0, (size_t)nt * nt * (nl + 2) * 8, c->st));
  GemmParams pl = gemm_defaults();
  pl.mode = GEMM_LAUUM;
  pl.A = c->S; pl.lda = ld;
  pl.B = c->S; pl.ldb = ld;
  pl.C = nullptr; pl.ldc = ld;
  pl.K = (int)c->Npad; pl.nt = nt;
  pl.XsT = c->dXsT; pl.sq = c->dsq; pl.alpha = c->dAlpha; pl.ldx = c->Npad;
  pl.N = (int)c->N; pl.P = c->P;
  pl.partials = plain ? nullptr : c->partials;
  pl.kinv_out = kinv_out;
  pl.dnoise_out = (c->het && rec && !plain) ? c->dDnoise : nullptr;
  pl.kp = c->kp;
  if (plain) { pl.kp.D = 1; pl.P = 1; }
  double flops = 0;
  for (int r = 0; r < nt; r++) flops += (double)(r + 1) * 2.0 * TILE * TILE * (double)(c->Npad - (long)r * TILE);
  int h = rec ? rec->begin(PH_LAUUM, flops) : -1;
  GPX_CHECK(launch_gemm(pl, dim3(nt, nt), c->st));
  if (rec) rec->end(h);
  c->eval_launches++;
  return 0;
}

static int eval_once(gpx_ctx* c, double extra_jitter, Recorder& rec) {
  cudaStream_t st = c->st;
  const long ld = c->Npad;
  const int nt = (int)(c->Npad / TILE);
  const int nl = c->kp.ard ? c->D : 1;
  GPX_CUDA(cudaMemsetAsync(c->info, 0, sizeof(int), st));
  if (c->multi) {
    if (c->m_cap != c->Npad) {
      for (double** mp : {&c->mXsT, &c->msq}) { if (*mp) cudaFree(*mp); *mp = nullptr; }
      GPX_CUDA(cudaMalloc(&c->mXsT, (size_t)MAX_D * c->Npad * 8));
      GPX_CUDA(cudaMalloc(&c->msq, (size_t)MAX_PARTS * c->Npad * 8));
      c->m_cap = c->Npad;
    }
    size_t pneed = 0;
    for (int q = 0; q < c->mk.nparts; q++) pneed += (size_t)nt * nt * part_nred(c->mk.part[q]);
    if (c->m_pcap < pneed) {
      if (c->mpartials) cudaFree(c->mpartials);
      c->mpartials = nullptr;
      c->m_pcap = 0;
      GPX_CUDA(cudaMalloc(&c->mpartials, pneed * 8));
      c->m_pcap = pneed;
    }
    // the composite K-build is one launch: the sweep's first diagonal block must wait for all of it, not for the event a
    // previous single-kernel evaluation on this context recorded after its first block row
    c->kfirst_valid = false;
    GPX_CUDA(cudaMemsetAsync(c->mflag, 0, sizeof(int), st));
    GPX_CHECK(launch_prep_multi(c->dX, c->N, c->D, c->Npad, c->mk, c->mXsT, c->msq, c->mflag, st));
    c->eval_launches++;
    KBuildMultiParams kb;
    memset(&kb, 0, sizeof(kb));
    kb.rowsT = c->mXsT; kb.ld_rows = c->Npad; kb.sq_rows = c->msq;
    kb.colsT = c->mXsT; kb.ld_cols = c->Npad; kb.sq_cols = c->msq;
    kb.out = c->S; kb.ld = ld; kb.nrows = c->N; kb.ncols = c->N; kb.sym = 1; kb.same = 1;
    kb.diag_add = ((c->het ? 0.0 : c->noise) + c->jitter) + extra_jitter;
    kb.diag_vec = c->het ? c->dNoiseVec : nullptr;
    kb.mk = c->mk;
    const int h = rec.begin(PH_KBUILD);
    GPX_CHECK(launch_kbuild_multi(kb, nt, nt, st));
    rec.end(h);
    c->eval_launches++;
  } else {
  GPX_CHECK(launch_prep_x(c->dX, c->N, c->Npad, c->kp, c->dXsT, c->dsq, st));
  c->eval_launches++;
  {
    KBuildParams kb;
    memset(&kb, 0, sizeof(kb));
    kb.rowsT = c->dXsT; kb.ld_rows = c->Npad;
    kb.colsT = c->dXsT; kb.ld_cols = c->Npad;
    kb.sq_rows = c->dsq; kb.sq_cols = c->dsq;
    kb.out = c->S; kb.ld = ld;
    kb.nrows = c->N; kb.ncols = c->N;
    kb.sym = 1; kb.same = 1;
    kb.diag_add = ((c->het ? 0.0 : c->noise) + c->jitter) + extra_jitter;
    kb.diag_vec = c->het ? c->dNoiseVec : nullptr;
    kb.kp = c->kp;
    const int h = rec.begin(PH_KBUILD);
    // chain schedule: the first block row goes first and is announced by an event, so that the factorisation of the first
    // diagonal block runs beside the rest of the covariance build
    const int nbt0 = (int)(pick_nb(c) / TILE);
    c->kfirst_valid = false;
    if (oz_wanted(c) && c->lookahead && c->chain && !c->oz_sched && nbt0 < nt) {
      GPX_CHECK(launch_kbuild(kb, nbt0, nt, st));
      if (!c->ev_kfirst) GPX_CUDA(cudaEventCreateWithFlags(&c->ev_kfirst, cudaEventDisableTiming));
      GPX_CUDA(cudaEventRecord(c->ev_kfirst, st));
      c->kfirst_valid = true;
      kb.rt0 = nbt0;
      GPX_CHECK(launch_kbuild(kb, nt - nbt0, nt, st));
      c->eval_launches++;
    } else {
      GPX_CHECK(launch_kbuild(kb, nt, nt, st));
    }
    rec.end(h);
    c->eval_launches++;
  }
  }
  const bool oz = oz_wanted(c);
  if (oz) GPX_CHECK(oz_prepare(c));
  c->oz_last = oz;
  {
    const int h = rec.begin(PH_SWEEP);
    GPX_CHECK(run_sweep(c, rec, oz ? 2 : 0));
    rec.end(h);
  }
  {
    const int h = rec.begin(PH_SOLVE);
    // alpha = U (U^T y). On the tcgen05 path t = L^-1 y = U^T y came along with the sweep (forward substitution): one mat-vec
    if (!oz) GPX_CHECK(launch_utv(c->S, ld, c->Npad, c->P, c->dY, c->dT, st));
    GPX_CHECK(launch_uv(c->S, ld, c->Npad, c->P, oz ? c->dTfw : c->dT, KSPLIT, c->dUvPart, c->dAlpha, st));
    rec.end(h);
    c->eval_launches += oz ? 2 : 3;
  }
  if (c->multi) {
    // composite kernel: K^-1 stored (by the sweep on the tcgen05 path, else by a plain LAUUM), then one reduction pass per part
    if (!oz) {
      if (!c->Kinv) GPX_CUDA(cudaMalloc(&c->Kinv, (size_t)ld * ld * 8));
      GPX_CHECK(run_lauum(c, c->Kinv, &rec, true));
    }
    FinalizeMultiParams fm;
    memset(&fm, 0, sizeof(fm));
    const int h = rec.begin(PH_LAUUM, 0.0);
    double* part = c->mpartials;
    for (int q = 0; q < c->mk.nparts; q++) {
      const int nred = part_nred(c->mk.part[q]);
      GPX_CUDA(cudaMemsetAsync(part, 0, (size_t)nt * nt * nred * 8, st));
      GradKinvMultiParams gm;
      memset(&gm, 0, sizeof(gm));
      gm.Kinv = c->Kinv; gm.ld = ld; gm.XsT = c->mXsT; gm.sq = c->msq; gm.ldx = c->Npad; gm.alpha = c->dAlpha;
      gm.N = c->N; gm.P = c->P; gm.nt = nt; gm.part = q; gm.want_noise = q == 0; gm.partials = part; gm.mk = c->mk;
      gm.dnoise_out = (q == 0 && c->het) ? c->dDnoise : nullptr;
      GPX_CHECK(launch_grad_kinv_multi(gm, st));
      c->eval_launches++;
      fm.partials[q] = part;
      part += (size_t)nt * nt * nred;
    }
    rec.end(h);
    fm.ntiles = (long)nt * nt; fm.logdet_part = c->logdet_part; fm.nt = nt;
    fm.T = oz ? c->dTfw : c->dT; fm.ld = ld; fm.N = c->N; fm.P = c->P; fm.mk = c->mk; fm.res = c->res;
    GPX_CHECK(launch_finalize_multi(fm, st));
    c->eval_launches++;
    int nres = 4;
    for (int q = 0; q < c->mk.nparts; q++) nres += part_ngrad(c->mk.part[q]);
    GPX_CUDA(cudaMemcpyAsync(c->h_res, c->res, nres * sizeof(double), cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaMemcpyAsync(c->h_info, c->info, sizeof(int), cudaMemcpyDeviceToHost, st));
    c->oz_last = true;   // K^-1 is stored either way
    return 0;
  }
  long grad_tiles = (long)nt * nt;
  if (oz) {
    // K^-1 was accumulated panel by panel inside the sweep (tcgen05): reduce dL_dK -> gradients from the stored tiles
    const int csplit = grad_kinv_csplit(nt, nl + 2);
    grad_tiles = (long)nt * nt * csplit;
    GPX_CUDA(cudaMemsetAsync(c->partials, 0, (size_t)grad_tiles * (nl + 2) * 8, st));
    GradKinvParams gk;
    memset(&gk, 0, sizeof(gk));
    gk.csplit = csplit;
    gk.Kinv = c->Kinv; gk.ld = ld;
    gk.XsT = c->dXsT; gk.sq = c->dsq; gk.alpha = c->dAlpha; gk.ldx = c->Npad;
    gk.N = c->N; gk.P = c->P; gk.nt = nt;
    gk.partials = c->partials;
    gk.dnoise_out = c->het ? c->dDnoise : nullptr;
    gk.kp = c->kp;
    const int h = rec.begin(PH_LAUUM, 0.0);
    GPX_CHECK(launch_grad_kinv(gk, st));
    rec.end(h);
    c->eval_launches++;
  } else if (c->fine && nt <= 8 && !c->dist) {
    // small matrix on the DMMA path (one block, or tcgen05 switched off): the fused LAUUM kernel has one CTA per 128 x 128 tile
    // -- 10 CTAs for N = 512, each walking up to 512 k alone (136 us of a 0.48 ms evaluation). K^-1 = U U^T in 64 x 32 tiles
    // (80 CTAs) into the K^-1 buffer, then the gradient pass over the stored tiles, split over the columns
    if (!c->Kinv) GPX_CUDA(cudaMalloc(&c->Kinv, (size_t)ld * ld * 8));
    const int h = rec.begin(PH_LAUUM, 0.0);
    FineParams fl{};
    fl.mode = FINE_LAUUM;
    fl.A = c->S; fl.lda = ld; fl.B = c->S; fl.ldb = ld; fl.C = c->Kinv; fl.ldc = ld; fl.K = (int)c->Npad; fl.nt = nt;
    GPX_CHECK(launch_fine(fl, st));
    const int csplit = grad_kinv_csplit(nt, nl + 2);
    grad_tiles = (long)nt * nt * csplit;
    GPX_CUDA(cudaMemsetAsync(c->partials, 0, (size_t)grad_tiles * (nl + 2) * 8, st));
    GradKinvParams gk;
    memset(&gk, 0, sizeof(gk));
    gk.csplit = csplit;
    gk.Kinv = c->Kinv; gk.ld = ld;
    gk.XsT = c->dXsT; gk.sq = c->dsq; gk.alpha = c->dAlpha; gk.ldx = c->Npad;
    gk.N = c->N; gk.P = c->P; gk.nt = nt;
    gk.partials = c->partials;
    gk.dnoise_out = c->het ? c->dDnoise : nullptr;
    gk.kp = c->kp;
    GPX_CHECK(launch_grad_kinv(gk, st));
    rec.end(h);
    c->eval_launches += 2;
    c->oz_last = true;   // K^-1 is stored
  } else {
    GPX_CHECK(run_lauum(c, nullptr, &rec));
  }
  {
    FinalizeParams f;
    memset(&f, 0, sizeof(f));
    f.partials = c->partials; f.ntiles = grad_tiles; f.nl = nl;
    f.logdet_part = c->logdet_part; f.nt = nt;
    f.T = oz ? c->dTfw : c->dT; f.ld = ld; f.N = c->N; f.P = c->P;
    f.kp = c->kp;
    f.res = c->res;
    GPX_CHECK(launch_finalize(f, st));
    c->eval_launches++;
  }
  GPX_CUDA(cudaMemcpyAsync(c->h_res, c->res, (nl + 5) * sizeof(double), cudaMemcpyDeviceToHost, st));
  GPX_CUDA(cudaMemcpyAsync(c->h_info, c->info, sizeof(int), cudaMemcpyDeviceToHost, st));
  return 0;
}

extern "C" {

}  // extern "C"

// coreg: one gpx_coreg per GPX_COREGIONALIZE part (null: no such part allowed). *kdiag_total = Kdiag of the composite kernel
// when it is the same at every point (no coregionalization part), else unused (composite_kdiag per point)
static int fill_multi(gpx_ctx* c, const gpx_kern_part* parts, int nparts, const gpx_coreg* coreg, double* kdiag_total) {
  if (!parts || nparts < 1 || nparts > MAX_PARTS) GPX_FAIL("number of kernel parts must be in [1, 8]");
  MultiKern& mk = c->mk;
  memset(&mk, 0, sizeof(mk));
  mk.nparts = nparts;
  c->m_coreg = false;
  int off = 0, nco = 0;
  double total = 0.0, prod = 1.0;
  for (int p = 0; p < nparts; p++) {
    const gpx_kern_part& in = parts[p];
    PartDev& pd = mk.part[p];
    if (in.kind < 0 || in.kind > GPX_COREGIONALIZE) GPX_FAIL("unknown kernel kind");
    if (p > 0 && in.term < parts[p - 1].term) GPX_FAIL("kernel parts must be ordered by term");
    if (in.kind == GPX_COREGIONALIZE) {
      if (!coreg) GPX_FAIL("a coregionalization part needs gpx_exact_eval_coreg and its B");
      const gpx_coreg& cg = coreg[nco++];
      if (cg.output_dim < 1 || cg.output_dim > MAX_O) GPX_FAIL("output_dim of a coregionalization part must be in [1, 16]");
      if (!cg.B) GPX_FAIL("null B of a coregionalization part");
      if (in.ndims != 1 || !in.dims) GPX_FAIL("a coregionalization part has exactly one active dim (the output index)");
      if (in.dims[0] < 0 || in.dims[0] >= c->D) GPX_FAIL("active dim outside the data");
      if (off + 1 > MAX_D) GPX_FAIL("the parts' active dims add up to more than 64");
      pd.kind = GPX_COREGIONALIZE; pd.term = in.term; pd.D = 1; pd.xoff = off; pd.odim = cg.output_dim;
      pd.variance = 1.0; pd.inv_ls_iso = 1.0;
      mk.dims[off] = in.dims[0];
      mk.ls[off] = 1.0;
      const int O = cg.output_dim;
      if (c->hB.size() != (size_t)MAX_PARTS * MAX_O * MAX_O) c->hB.assign((size_t)MAX_PARTS * MAX_O * MAX_O, 0.0);
      // only the lower tiles of K are built and an off-diagonal tile stands for its mirror in the S reduction: B must be
      // exactly symmetric, as W W^T + diag(kappa) is
      for (int a = 0; a < O; a++)
        for (int b = 0; b < O; b++) {
          if (!std::isfinite(cg.B[a * O + b])) GPX_FAIL("B of a coregionalization part must be finite");
          if (cg.B[a * O + b] != cg.B[b * O + a]) GPX_FAIL("B of a coregionalization part must be symmetric");
          c->hB[(size_t)p * MAX_O * MAX_O + a * O + b] = cg.B[a * O + b];
        }
      c->m_coreg = true;
      off += 1;
      if (p > 0 && in.term != parts[p - 1].term) { total += prod; prod = 1.0; }
      continue;
    }
    if (!(in.variance > 0)) GPX_FAIL("variance must be positive");
    const bool stat = in.kind >= GPX_WHITE;
    if (!stat && (in.ndims < 1 || !in.dims || !in.lengthscale)) GPX_FAIL("a stationary part needs active dims and a lengthscale");
    pd.kind = in.kind; pd.ard = (!stat && in.ard) ? 1 : 0; pd.term = in.term; pd.D = stat ? 0 : in.ndims; pd.xoff = off;
    pd.variance = in.variance; pd.inv_ls_iso = 1.0;
    if (off + pd.D > MAX_D) GPX_FAIL("the parts' active dims add up to more than 64");
    for (int q = 0; q < pd.D; q++) {
      if (in.dims[q] < 0 || in.dims[q] >= c->D) GPX_FAIL("active dim outside the data");
      const double l = in.lengthscale[pd.ard ? q : 0];
      if (!(l > 0)) GPX_FAIL("lengthscale must be positive");
      mk.dims[off + q] = in.dims[q];
      mk.ls[off + q] = l;
    }
    if (!stat && !pd.ard) pd.inv_ls_iso = 1.0 / in.lengthscale[0];
    off += pd.D;
    if (p > 0 && in.term != parts[p - 1].term) { total += prod; prod = 1.0; }
    prod *= in.variance;                      // every kind has Kdiag = variance (stationary.py:170-173, static.py:30-33)
  }
  total += prod;
  mk.sumD = off;
  *kdiag_total = total;
  if (c->m_coreg) {
    if (!c->mB) GPX_CUDA(cudaMalloc(&c->mB, (size_t)MAX_PARTS * MAX_O * MAX_O * 8));
    GPX_CUDA(cudaMemcpyAsync(c->mB, c->hB.data(), (size_t)MAX_PARTS * MAX_O * MAX_O * 8, cudaMemcpyHostToDevice, c->st));
  }
  if (!c->mflag) GPX_CUDA(cudaMalloc(&c->mflag, sizeof(int)));
  mk.B = c->mB;
  return 0;
}

// Kdiag of the composite kernel at one point x (D columns, output indices already checked): sum over the terms of the
// product of the parts' Kdiag (add.py:74-79, prod.py:68-76): variance for the stationary / static kinds (stationary.py:170-173,
// static.py:30-33), B[idx, idx] for a coregionalization part (coregionalize.py:107-108)
static double composite_kdiag(const gpx_ctx* c, const double* x) {
  const MultiKern& mk = c->mk;
  double total = 0.0, prod = 1.0;
  for (int p = 0; p < mk.nparts; p++) {
    const PartDev& pd = mk.part[p];
    if (p > 0 && pd.term != mk.part[p - 1].term) { total += prod; prod = 1.0; }
    if (pd.kind == GPX_COREGIONALIZE) {
      const int a = (int)x[mk.dims[pd.xoff]];
      prod *= c->hB[(size_t)p * MAX_O * MAX_O + (size_t)a * pd.odim + a];
    } else {
      prod *= pd.variance;
    }
  }
  return total + prod;
}

// every output index of the coregionalization parts in the M x D host points X lies in [0, O)
static bool coreg_indices_ok(const gpx_ctx* c, const double* X, long M) {
  for (int p = 0; p < c->mk.nparts; p++) {
    const PartDev& pd = c->mk.part[p];
    if (pd.kind != GPX_COREGIONALIZE) continue;
    for (long m = 0; m < M; m++) {
      const double v = X[m * c->D + c->mk.dims[pd.xoff]];
      if (!(v > -1.0 && v < (double)pd.odim)) return false;
    }
  }
  return true;
}

static int exact_eval_impl(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale, double noise,
                           const double* noise_vec, double jitter, int max_tries, double* lml, double* grad,
                           double* dnoise, double* jitter_used, const gpx_kern_part* parts = nullptr, int nparts = 0,
                           const gpx_coreg* coreg = nullptr) {
  if (!c || !lml || !grad || (!parts && !lengthscale)) GPX_FAIL("null argument");
  if (!c->S) GPX_FAIL("gpx_set_data has not been called");
  if (!(noise >= 0)) GPX_FAIL("noise variance must be non-negative");
  GPX_CUDA(cudaSetDevice(c->device));
  // the kernel description is rewritten below: a call rejected half-way must not leave the previous posterior usable
  // with a half-filled kernel (gpx_get(K) / gpx_predict)
  c->have_eval = false;
  c->have_kinv = false;
  c->multi = parts != nullptr;
  if (c->multi) {
    if (c->dist) GPX_FAIL("composite kernels are single-GPU");
    GPX_CHECK(fill_multi(c, parts, nparts, coreg, &variance));   // `variance` = Kdiag of the composite kernel (jitter ladder)
    c->kp.variance = variance;
  } else
  GPX_CHECK(fill_kp(c->kp, kind, ard, c->D, variance, lengthscale));
  c->het = noise_vec != nullptr;
  if (c->het) {
    if (c->dist) GPX_FAIL("heteroscedastic evaluation is single-GPU");
    if (!dnoise) GPX_FAIL("null argument");
    if (c->het_cap < c->Npad) {
      if (c->dNoiseVec) cudaFree(c->dNoiseVec);
      if (c->dDnoise) cudaFree(c->dDnoise);
      c->dNoiseVec = c->dDnoise = nullptr;
      GPX_CUDA(cudaMalloc(&c->dNoiseVec, (size_t)c->Npad * 8));
      GPX_CUDA(cudaMalloc(&c->dDnoise, (size_t)c->Npad * 8));
      c->het_cap = c->Npad;
    }
    GPX_CUDA(cudaMemcpyAsync(c->dNoiseVec, noise_vec, (size_t)c->N * 8, cudaMemcpyHostToDevice, c->st));
  }
  c->noise = noise;
  c->jitter = jitter;
  c->have_eval = false;
  c->have_kinv = false;
  const int nl = ard ? c->D : 1;
  memset(&c->stats, 0, sizeof(c->stats));
  c->eval_launches = 0;
  Recorder rec{c};
  const int htot = rec.begin(PH_TOTAL);
  double extra = 0.0;
  int tries = 0;
  int info = 0;
  for (;;) {
    tries++;
    if (c->dist) {
      GPX_CHECK(dist_exact_eval(c, extra));
    } else {
      GPX_CHECK(eval_once(c, extra, rec));
      GPX_CUDA(cudaStreamSynchronize(c->st));
    }
    if (c->multi && c->m_coreg) {
      int bad = 0;
      GPX_CUDA(cudaMemcpy(&bad, c->mflag, sizeof(int), cudaMemcpyDeviceToHost));
      if (bad) GPX_FAIL("output index of a coregionalization part outside [0, output_dim)");
    }
    info = *c->h_info;
    if (info == 0) break;
    if (tries == 1 && c->multi && c->m_coreg) {
      // the ladder's mean diagonal (util/linalg.py:66-74) with a per-point Kdiag: its mean over the training points
      std::vector<double> hx((size_t)c->N * c->D);
      GPX_CUDA(cudaMemcpy(hx.data(), c->dX, hx.size() * 8, cudaMemcpyDeviceToHost));
      double s = 0.0;
      for (long i = 0; i < c->N; i++) s += composite_kdiag(c, hx.data() + (size_t)i * c->D);
      variance = s / (double)std::max<long>(c->N, 1);
    }
    // jitchol ladder (GPy/util/linalg.py:61-75): the diagonal of Ky is variance + noise + jitter (> 0 here),
    // extra jitter = mean(diag) * 1e-6 * 10^k for k = 0 .. max_tries-1
    if (tries > max_tries) break;
    const double mean_diag = variance + (noise + jitter);
    extra = mean_diag * 1e-6 * pow(10.0, tries - 1);
    if (!std::isfinite(extra)) break;
  }
  rec.end(htot);
  GPX_CUDA(cudaStreamSynchronize(c->st));
  c->jitter_extra = extra;
  c->stats.tries = tries;
  // accounting
  for (auto& s : rec.spans) {
    if (s.b < 0) continue;
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev[s.a], c->ev[s.b]);
    switch (s.phase) {
      case PH_KBUILD: c->stats.kbuild_ms += ms; break;
      case PH_SWEEP: c->stats.sweep_ms += ms; break;
      case PH_UPDATE: c->stats.update_ms += ms; c->stats.update_flops += s.flops; break;
      case PH_LAUUM: c->stats.lauum_ms += ms; c->stats.lauum_flops += s.flops; break;
      case PH_SOLVE: c->stats.solve_ms += ms; break;
      case PH_TOTAL: c->stats.total_ms += ms; break;
    }
  }
  c->stats.kbuild_bytes = 8.0 * (double)c->N * c->N + 8.0 * (double)c->N * c->D;
  c->stats.launches = c->eval_launches;
  c->total_launches += c->eval_launches;
  if (jitter_used) *jitter_used = extra;
  if (info != 0) {
    gpx::set_error("not positive definite, even with jitter.");
    return info;
  }
  *lml = c->h_res[0];
  if (c->multi) {
    int n = 0;
    for (int p = 0; p < c->mk.nparts; p++) n += part_ngrad(c->mk.part[p]);
    for (int q = 0; q < n; q++) grad[q] = c->h_res[4 + q];
    grad[n] = c->h_res[3];
  } else
  for (int q = 0; q < nl + 2; q++) grad[q] = c->h_res[1 + q];
  if (c->het) {
    GPX_CUDA(cudaMemcpyAsync(dnoise, c->dDnoise, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->st));
    GPX_CUDA(cudaStreamSynchronize(c->st));
  }
  c->have_eval = true;
  c->have_kinv = c->oz_last;   // the Ozaki path leaves K^-1 (lower tiles) in c->Kinv
  return 0;
}

extern "C" {

int gpx_exact_eval(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale, double noise,
                   double jitter, int max_tries, double* lml, double* grad, double* jitter_used) {
  return exact_eval_impl(c, kind, ard, variance, lengthscale, noise, nullptr, jitter, max_tries, lml, grad, nullptr,
                         jitter_used);
}

int gpx_exact_eval_multi(gpx_ctx* c, const gpx_kern_part* parts, int nparts, double noise, double jitter, int max_tries,
                         double* lml, double* grad, double* jitter_used) {
  if (!parts) GPX_FAIL("null argument");
  return exact_eval_impl(c, 0, 0, 1.0, nullptr, noise, nullptr, jitter, max_tries, lml, grad, nullptr, jitter_used, parts,
                         nparts);
}

int gpx_exact_eval_coreg(gpx_ctx* c, const gpx_kern_part* parts, int nparts, const gpx_coreg* coreg, double noise,
                         const double* noise_variances, double jitter, int max_tries, double* lml, double* grad,
                         double* dnoise, double* jitter_used) {
  if (!c || !parts) GPX_FAIL("null argument");
  if (!noise_variances) return exact_eval_impl(c, 0, 0, 1.0, nullptr, noise, nullptr, jitter, max_tries, lml, grad, nullptr,
                                               jitter_used, parts, nparts, coreg);
  double mean = 0.0;
  for (int64_t i = 0; i < c->N; i++) {
    if (!(noise_variances[i] >= 0)) GPX_FAIL("noise variances must be non-negative");
    mean += noise_variances[i];
  }
  mean /= (double)std::max<int64_t>(c->N, 1);
  return exact_eval_impl(c, 0, 0, 1.0, nullptr, mean, noise_variances, jitter, max_tries, lml, grad, dnoise, jitter_used,
                         parts, nparts, coreg);
}

int gpx_exact_eval_het(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale,
                       const double* noise_variances, double jitter, int max_tries, double* lml, double* grad,
                       double* dnoise, double* jitter_used) {
  if (!c || !noise_variances) GPX_FAIL("null argument");
  double mean = 0.0;
  for (int64_t i = 0; i < c->N; i++) {
    if (!(noise_variances[i] >= 0)) GPX_FAIL("noise variances must be non-negative");
    mean += noise_variances[i];
  }
  mean /= (double)std::max<int64_t>(c->N, 1);
  return exact_eval_impl(c, kind, ard, variance, lengthscale, mean, noise_variances, jitter, max_tries, lml, grad, dnoise,
                         jitter_used);
}

int gpx_measure_fp64_peak(gpx_ctx* c, double* tflops) {
  if (!c || !tflops) GPX_FAIL("null argument");
  GPX_CUDA(cudaSetDevice(c->device));
  return measure_dmma_peak(c->st, tflops);
}

int gpx_get_stats(gpx_ctx* c, gpx_stats* out) {
  if (!c || !out) GPX_FAIL("null argument");
  *out = c->stats;
  return 0;
}
int64_t gpx_total_launches(gpx_ctx* c) { return c ? c->total_launches : -1; }

static int ensure_staging(gpx_ctx* c) {
  const size_t need = (size_t)c->N * c->N * 8;
  if (c->staging && c->staging_cap < need) { cudaFree(c->staging); c->staging = nullptr; }
  if (!c->staging) { GPX_CUDA(cudaMalloc(&c->staging, need)); c->staging_cap = need; }
  return 0;
}

int gpx_get(gpx_ctx* c, int which, double* out) {
  if (!c || !out) GPX_FAIL("null argument");
  if (!c->have_eval) GPX_FAIL("no successful gpx_exact_eval to fetch results from");
  GPX_CUDA(cudaSetDevice(c->device));
  if (c->dist && which == GPX_GET_L) {   // collective: every rank calls it and receives the whole factor
    memset(out, 0, (size_t)c->N * c->N * 8);
    return dist_get_L(c, out);
  }
  if (c->dist && which != GPX_GET_ALPHA)
    GPX_FAIL("sharded mode: alpha and L (collective) can be fetched; K^-1 / dL_dK / K stay distributed or are rebuilt by the caller");
  cudaStream_t st = c->st;
  const long N = c->N, ld = c->Npad;
  if (which == GPX_GET_ALPHA) {
    GPX_CHECK(launch_untranspose(c->dAlpha, N, c->P, ld, c->dUvPart, st));
    c->total_launches++;
    GPX_CUDA(cudaMemcpyAsync(out, c->dUvPart, (size_t)N * c->P * 8, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  GPX_CHECK(ensure_staging(c));
  if (which == GPX_GET_K && c->multi) {
    KBuildMultiParams kb;
    memset(&kb, 0, sizeof(kb));
    kb.rowsT = c->mXsT; kb.ld_rows = ld; kb.sq_rows = c->msq; kb.colsT = c->mXsT; kb.ld_cols = ld; kb.sq_cols = c->msq;
    kb.out = c->staging; kb.ld = N; kb.nrows = N; kb.ncols = N; kb.sym = 0; kb.same = 1; kb.mk = c->mk;
    GPX_CHECK(launch_kbuild_multi(kb, (int)(ld / TILE), (int)(ld / TILE), st));
    c->total_launches++;
  } else if (which == GPX_GET_K) {
    KBuildParams kb;
    memset(&kb, 0, sizeof(kb));
    kb.rowsT = c->dXsT; kb.ld_rows = ld; kb.colsT = c->dXsT; kb.ld_cols = ld;
    kb.sq_rows = c->dsq; kb.sq_cols = c->dsq;
    kb.out = c->staging; kb.ld = N; kb.nrows = N; kb.ncols = N; kb.sym = 0; kb.same = 1; kb.kp = c->kp;
    GPX_CHECK(launch_kbuild(kb, (int)(ld / TILE), (int)(ld / TILE), st));
    c->total_launches++;
  } else if (which == GPX_GET_L || which == GPX_GET_LINV) {
    GPX_CHECK(launch_extract(which, c->S, ld, c->Ldiag, nullptr, nullptr, 0, N, c->staging, st));
    c->total_launches++;
  } else if (which == GPX_GET_KINV || which == GPX_GET_DLDK) {
    if (!c->have_kinv) {
      if (!c->Kinv) GPX_CUDA(cudaMalloc(&c->Kinv, (size_t)ld * ld * 8));
      const int64_t keep = c->eval_launches;
      GPX_CHECK(run_lauum(c, c->Kinv, nullptr));
      c->total_launches += c->eval_launches - keep;
      c->eval_launches = keep;
      c->have_kinv = true;
    }
    GPX_CHECK(launch_extract(which, c->S, ld, c->Ldiag, c->Kinv, c->dAlpha, c->P, N, c->staging, st));
    c->total_launches++;
  } else {
    GPX_FAIL("unknown gpx_get selector");
  }
  GPX_CUDA(cudaMemcpyAsync(out, c->staging, (size_t)N * N * 8, cudaMemcpyDeviceToHost, st));
  GPX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// standalone kernel-plugin calls
// ---------------------------------------------------------------------------------------------------------------
static std::mutex g_scratch_mu;
static gpx_ctx* g_scratch = nullptr;
static int scratch_ctx(gpx_ctx** out) {
  std::lock_guard<std::mutex> lk(g_scratch_mu);
  if (!g_scratch) {
    int dev = 0;
    cudaGetDevice(&dev);
    GPX_CHECK(gpx_create(dev, &g_scratch));
  }
  *out = g_scratch;
  return 0;
}

// Temporaries of the stand-alone kernel calls and of gpx_predict: stream-ordered allocations from the device's default memory
// pool (cudaMallocAsync / cudaFreeAsync on the context's stream; gpx_create raises the pool's release threshold so that freed
// blocks stay cached). A plain cudaMalloc / cudaFree pair per call is a device-wide synchronisation point inside any
// optimiser loop that uses foreign inference (round-1 review).
#define GPX_TMP_ALLOC(ptr, bytes, st) GPX_CUDA(cudaMallocAsync((void**)(ptr), (bytes), (st)))
#define GPX_TMP_FREE(p, st) do { if (p) cudaFreeAsync((p), (st)); } while (0)

struct PointSet {
  double* raw = nullptr; double* xT = nullptr; double* sq = nullptr; long n = 0, ld = 0;
  cudaStream_t st = nullptr;
  ~PointSet() { GPX_TMP_FREE(raw, st); GPX_TMP_FREE(xT, st); GPX_TMP_FREE(sq, st); }
};
static int upload_points(gpx_ctx* c, const double* X, long n, const KernParams& kp, PointSet& ps) {
  ps.n = n; ps.ld = (n + TILE - 1) / TILE * TILE; ps.st = c->st;
  GPX_TMP_ALLOC(&ps.raw, (size_t)n * kp.D * 8, c->st);
  GPX_TMP_ALLOC(&ps.xT, (size_t)ps.ld * kp.D * 8, c->st);
  GPX_TMP_ALLOC(&ps.sq, (size_t)ps.ld * 8, c->st);
  GPX_CUDA(cudaMemcpyAsync(ps.raw, X, (size_t)n * kp.D * 8, cudaMemcpyHostToDevice, c->st));
  GPX_CHECK(launch_prep_x(ps.raw, n, ps.ld, kp, ps.xT, ps.sq, c->st));
  c->total_launches++;
  return 0;
}

int gpx_kern_K(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale, const double* X, int64_t N,
               const double* X2, int64_t M, int D, double* out) {
  if (!X || !lengthscale) GPX_FAIL("null argument");
  if (!c) GPX_CHECK(scratch_ctx(&c));
  GPX_CUDA(cudaSetDevice(c->device));
  KernParams kp;
  GPX_CHECK(fill_kp(kp, kind, ard, D, variance, lengthscale));
  if (!X2) M = N;
  if (N < 1 || M < 1) GPX_FAIL("empty input");
  PointSet p1, p2;
  GPX_CHECK(upload_points(c, X, N, kp, p1));
  if (X2) GPX_CHECK(upload_points(c, X2, M, kp, p2));
  PointSet& pj = X2 ? p2 : p1;   // thread-mapped operand = X2 points (contiguous index of the row-major output)
  double* dout = nullptr;
  GPX_TMP_ALLOC(&dout, (size_t)N * M * 8, c->st);
  KBuildParams kb;
  memset(&kb, 0, sizeof(kb));
  kb.rowsT = pj.xT; kb.ld_rows = pj.ld; kb.sq_rows = pj.sq;
  kb.colsT = p1.xT; kb.ld_cols = p1.ld; kb.sq_cols = p1.sq;
  kb.out = dout; kb.ld = M; kb.nrows = M; kb.ncols = N; kb.sym = 0; kb.same = X2 ? 0 : 1; kb.kp = kp;
  // out == NULL: build on the device only (the result is dropped) and report the kernel time through gpx_get_stats
  // (kbuild_ms / kbuild_bytes) — used to measure the rectangular K(X, Z) build of the sparse model at full size.
  cudaEvent_t e0, e1;
  int rc = ev_get(c, 0, &e0) || ev_get(c, 1, &e1);
  if (rc == 0) {
    cudaEventRecord(e0, c->st);
    rc = launch_kbuild(kb, (int)(pj.ld / TILE), (int)(p1.ld / TILE), c->st);
    cudaEventRecord(e1, c->st);
  }
  c->total_launches++;
  if (rc == 0 && out && cudaMemcpyAsync(out, dout, (size_t)N * M * 8, cudaMemcpyDeviceToHost, c->st) != cudaSuccess) rc = -1;
  if (cudaStreamSynchronize(c->st) != cudaSuccess) { gpx::set_error("gpx_kern_K: device failure"); rc = -1; }
  if (rc == 0) {
    cudaEventElapsedTime(&c->stats.kbuild_ms, e0, e1);
    c->stats.kbuild_bytes = 8.0 * (double)N * M + 8.0 * (double)(N + M) * D;
  }
  GPX_TMP_FREE(dout, c->st);
  return rc;
}

int gpx_kern_Kdiag(int kind, double variance, int64_t N, double* out) {
  (void)kind;
  if (!out) GPX_FAIL("null argument");
  for (int64_t i = 0; i < N; i++) out[i] = variance;   // stationary.py:170-173
  return 0;
}

int gpx_kern_grad_full(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale, const double* X,
                       int64_t N, const double* X2, int64_t M, int D, const double* dL_dK, double* dvariance,
                       double* dlengthscale) {
  if (!X || !dL_dK || !lengthscale || !dvariance || !dlengthscale) GPX_FAIL("null argument");
  if (!c) GPX_CHECK(scratch_ctx(&c));
  GPX_CUDA(cudaSetDevice(c->device));
  KernParams kp;
  GPX_CHECK(fill_kp(kp, kind, ard, D, variance, lengthscale));
  if (!X2) M = N;
  PointSet p1, p2;
  GPX_CHECK(upload_points(c, X, N, kp, p1));
  if (X2) GPX_CHECK(upload_points(c, X2, M, kp, p2));
  PointSet& pj = X2 ? p2 : p1;
  double* dd = nullptr; double* dpart = nullptr;
  const int tj = (int)(pj.ld / TILE), ti = (int)(p1.ld / TILE);
  const int nl = ard ? D : 1, nred = nl + 1;
  GPX_TMP_ALLOC(&dd, (size_t)N * M * 8, c->st);
  GPX_TMP_ALLOC(&dpart, (size_t)tj * ti * nred * 8, c->st);
  GPX_CUDA(cudaMemcpyAsync(dd, dL_dK, (size_t)N * M * 8, cudaMemcpyHostToDevice, c->st));
  GradFullParams gp;
  memset(&gp, 0, sizeof(gp));
  gp.x1T = p1.xT; gp.ld1 = p1.ld; gp.sq1 = p1.sq; gp.N = N;
  gp.x2T = pj.xT; gp.ld2 = pj.ld; gp.sq2 = pj.sq; gp.M = M;
  gp.dL_dK = dd; gp.same = X2 ? 0 : 1; gp.partials = dpart; gp.kp = kp;
  int rc = launch_grad_full(gp, tj, ti, c->st);
  c->total_launches++;
  std::vector<double> hp((size_t)tj * ti * nred);
  if (rc == 0 && cudaMemcpyAsync(hp.data(), dpart, hp.size() * 8, cudaMemcpyDeviceToHost, c->st) != cudaSuccess) rc = -1;
  if (cudaStreamSynchronize(c->st) != cudaSuccess) { gpx::set_error("gpx_kern_grad_full: device failure"); rc = -1; }
  GPX_TMP_FREE(dd, c->st); GPX_TMP_FREE(dpart, c->st);
  if (rc) return rc;
  std::vector<double> tot(nred, 0.0);
  for (size_t t = 0; t < (size_t)tj * ti; t++)
    for (int q = 0; q < nred; q++) tot[q] += hp[t * nred + q];
  *dvariance = tot[0];
  for (int q = 0; q < nl; q++) dlengthscale[q] = -tot[1 + q] / lengthscale[q];
  return 0;
}

int gpx_kern_grad_X(gpx_ctx* c, int kind, int ard, double variance, const double* lengthscale, const double* X, int64_t N,
                    const double* X2, int64_t M, int D, const double* dL_dK, double* grad) {
  if (!X || !dL_dK || !lengthscale || !grad) GPX_FAIL("null argument");
  if (!c) GPX_CHECK(scratch_ctx(&c));
  GPX_CUDA(cudaSetDevice(c->device));
  KernParams kp;
  GPX_CHECK(fill_kp(kp, kind, ard, D, variance, lengthscale));
  if (!X2) M = N;
  PointSet p1, p2;
  GPX_CHECK(upload_points(c, X, N, kp, p1));
  if (X2) GPX_CHECK(upload_points(c, X2, M, kp, p2));
  PointSet& pj = X2 ? p2 : p1;
  // m is split into chunks so that ~4 waves of CTAs are in flight; partials are reduced in fixed order
  const long ntile = (N + TILE - 1) / TILE;
  int nchunk = (int)std::max<long>(1, std::min<long>((M + 31) / 32, (4 * 148 + ntile - 1) / ntile));
  const long mchunk = ((M + nchunk - 1) / nchunk + 31) / 32 * 32;
  nchunk = (int)((M + mchunk - 1) / mchunk);
  double *dd = nullptr, *dpart = nullptr, *dout = nullptr;
  GPX_TMP_ALLOC(&dd, (size_t)N * M * 8, c->st);
  GPX_TMP_ALLOC(&dpart, (size_t)nchunk * N * D * 8, c->st);
  GPX_TMP_ALLOC(&dout, (size_t)N * D * 8, c->st);
  GPX_CUDA(cudaMemcpyAsync(dd, dL_dK, (size_t)N * M * 8, cudaMemcpyHostToDevice, c->st));
  GradFullParams gp;
  memset(&gp, 0, sizeof(gp));
  gp.x1T = p1.xT; gp.ld1 = p1.ld; gp.sq1 = p1.sq; gp.N = N;
  gp.x2T = pj.xT; gp.ld2 = pj.ld; gp.sq2 = pj.sq; gp.M = M;
  gp.dL_dK = dd; gp.same = X2 ? 0 : 1; gp.kp = kp;
  int rc = launch_gradx(gp, nchunk, mchunk, dpart, dout, c->st);
  c->total_launches += 2;
  if (rc == 0 && cudaMemcpyAsync(grad, dout, (size_t)N * D * 8, cudaMemcpyDeviceToHost, c->st) != cudaSuccess) rc = -1;
  if (cudaStreamSynchronize(c->st) != cudaSuccess) { gpx::set_error("gpx_kern_grad_X: device failure"); rc = -1; }
  GPX_TMP_FREE(dd, c->st); GPX_TMP_FREE(dpart, c->st); GPX_TMP_FREE(dout, c->st);
  return rc;
}

// ---------------------------------------------------------------------------------------------------------------
// stand-alone pdinv / jitchol for a caller-supplied symmetric matrix (GPy/util/linalg.py:56-75,193-214)
// ---------------------------------------------------------------------------------------------------------------
}  // extern "C"

// Factor-and-invert a dense symmetric matrix that already lives on the device (dA, leading dimension lda, order N) into
// the workspace of context c (lower = L, upper = U = L^-T), with jitchol's ladder (GPy/util/linalg.py:56-75):
// jitter0 is always added; on failure mean(diag)*1e-6*10^k. Returns 0, or the failing minor (>0) / an error (<0).
int gpx::factor_device(gpx_ctx* c, const double* dA, long lda, long N, double jitter0, int max_tries, double* logdet,
                       double* jitter_used) {
  {
    std::vector<double> zx((size_t)N, 0.0);
    if (c->N != N || c->D != 1 || c->P != 1 || !c->S) GPX_CHECK(gpx_set_data(c, zx.data(), N, 1, zx.data(), 1));
  }
  c->have_eval = false;
  c->have_kinv = false;
  cudaStream_t st = c->st;
  const long ld = c->Npad;
  Recorder rec{c};
  double extra = 0.0;
  int tries = 0, info = 0;
  const int64_t l0 = c->eval_launches;
  for (;;) {
    tries++;
    GPX_CUDA(cudaMemsetAsync(c->info, 0, sizeof(int), st));
    GPX_CHECK(launch_load_sym(dA, lda, N, c->S, ld, jitter0 + extra, st));
    c->eval_launches++;
    GPX_CHECK(run_sweep(c, rec));
    GPX_CUDA(cudaMemcpyAsync(c->h_info, c->info, sizeof(int), cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
    info = *c->h_info;
    if (info == 0) break;
    // jitchol's rules need the diagonal: fetch it only on this (rare) path
    std::vector<double> dg((size_t)N);
    GPX_CUDA(cudaMemcpy2DAsync(dg.data(), 8, dA, (size_t)(lda + 1) * 8, 8, (size_t)N, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
    double dsum = 0.0;
    bool nonpos = false;
    for (long i = 0; i < N; i++) { dsum += dg[i] + jitter0; if (!(dg[i] + jitter0 > 0.0)) nonpos = true; }
    if (nonpos) { gpx::set_error("not pd: non-positive diagonal elements"); c->total_launches += c->eval_launches - l0; return info; }
    if (tries > max_tries) break;
    extra = dsum / (double)N * 1e-6 * pow(10.0, tries - 1);     // linalg.py:66-72
    if (!std::isfinite(extra)) break;
  }
  c->total_launches += c->eval_launches - l0;
  if (jitter_used) *jitter_used = extra;
  if (info != 0) { gpx::set_error("not positive definite, even with jitter."); return info; }
  if (logdet) {   // 2 sum log diag(L) (linalg.py:208): per-tile partials summed in fixed order
    const int nt = (int)(ld / TILE);
    std::vector<double> parts(nt);
    GPX_CUDA(cudaMemcpyAsync(parts.data(), c->logdet_part, (size_t)nt * 8, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
    double s = 0.0;
    for (int i = 0; i < nt; i++) s += parts[i];
    *logdet = s;
  }
  return 0;
}

extern "C" {

int gpx_pdinv(gpx_ctx* c, const double* A, int64_t N, int max_tries, double* Ai, double* L, double* Li, double* logdet,
              double* jitter_used) {
  if (!A || !logdet) GPX_FAIL("null argument");
  if (!c) GPX_CHECK(scratch_ctx(&c));
  if (c->dist) GPX_FAIL("gpx_pdinv is single-GPU");
  if (N < 1) GPX_FAIL("N must be positive");
  GPX_CUDA(cudaSetDevice(c->device));
  {
    std::vector<double> zx((size_t)N, 0.0);
    if (c->N != N || c->D != 1 || c->P != 1 || !c->S) GPX_CHECK(gpx_set_data(c, zx.data(), N, 1, zx.data(), 1));
  }
  cudaStream_t st = c->st;
  const long ld = c->Npad;
  GPX_CHECK(ensure_staging(c));
  GPX_CUDA(cudaMemcpyAsync(c->staging, A, (size_t)N * N * 8, cudaMemcpyHostToDevice, st));
  if (!c->Kinv) GPX_CUDA(cudaMalloc(&c->Kinv, (size_t)ld * ld * 8));
  // the factorisation reads the staged copy; the staging buffer is reused for the results afterwards
  double* dA = c->Kinv;   // park A in the K^-1 buffer (same size class) so that staging stays free for extraction
  GPX_CUDA(cudaMemcpyAsync(dA, c->staging, (size_t)N * N * 8, cudaMemcpyDeviceToDevice, st));
  {
    const int rc = factor_device(c, dA, N, N, 0.0, max_tries, logdet, jitter_used);
    if (rc != 0) return rc;
  }
  const int64_t l0 = c->eval_launches;
  if (Ai) {
    const long ntl = ld / TILE;
    GemmParams pl = gemm_defaults();
    pl.mode = GEMM_LAUUM;
    pl.A = c->S; pl.lda = ld; pl.B = c->S; pl.ldb = ld; pl.ldc = ld;
    pl.K = (int)ld; pl.nt = (int)ntl; pl.N = (int)N; pl.P = 1;
    pl.partials = nullptr; pl.kinv_out = c->Kinv;
    pl.kp.D = 1;
    GPX_CHECK(launch_gemm(pl, dim3(1, 1), st));
    c->eval_launches++;
    GPX_CHECK(launch_extract(GPX_GET_KINV, c->S, ld, c->Ldiag, c->Kinv, nullptr, 0, N, c->staging, st));
    c->eval_launches++;
    GPX_CUDA(cudaMemcpyAsync(Ai, c->staging, (size_t)N * N * 8, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
  }
  if (L) {
    GPX_CHECK(launch_extract(GPX_GET_L, c->S, ld, c->Ldiag, nullptr, nullptr, 0, N, c->staging, st));
    c->eval_launches++;
    GPX_CUDA(cudaMemcpyAsync(L, c->staging, (size_t)N * N * 8, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
  }
  if (Li) {
    GPX_CHECK(launch_extract(GPX_GET_LINV, c->S, ld, c->Ldiag, nullptr, nullptr, 0, N, c->staging, st));
    c->eval_launches++;
    GPX_CUDA(cudaMemcpyAsync(Li, c->staging, (size_t)N * N * 8, cudaMemcpyDeviceToHost, st));
    GPX_CUDA(cudaStreamSynchronize(st));
  }
  c->total_launches += c->eval_launches - l0;
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// prediction with the factor of the last evaluation (posterior.py:273-302)
// ---------------------------------------------------------------------------------------------------------------
int gpx_predict(gpx_ctx* c, const double* Xnew, int64_t M, int full_cov, double* mu, double* var) {
  if (!c || !Xnew || !mu || !var) GPX_FAIL("null argument");
  if (!c->have_eval) GPX_FAIL("no successful gpx_exact_eval to predict from");
  if (M < 1) GPX_FAIL("empty Xnew");
  // sharded factor: U = L^-T is column-distributed (block columns dealt round-robin), X / Y / alpha are replicated.
  // Every rank forms K(X, Xnew) and the mean; the variance term sum_i (U^T Kx)_i^2 splits over the owned columns and is
  // all-reduced. All ranks must call gpx_predict together (it contains a collective).
  int drank = 0, dG = 1;
  dist_world(c, &drank, &dG);
  const long dNB = dist_block(c);
  GPX_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->st;
  const long ld = c->Npad, N = c->N;
  PointSet pn;
  if (c->multi && !coreg_indices_ok(c, Xnew, M)) GPX_FAIL("output index of a coregionalization part outside [0, output_dim)");
  if (c->multi) {   // composite kernel: stacked per-part scaled coordinates of the new points
    pn.n = M; pn.ld = (M + TILE - 1) / TILE * TILE; pn.st = c->st;
    GPX_TMP_ALLOC(&pn.raw, (size_t)M * c->D * 8, c->st);
    GPX_TMP_ALLOC(&pn.xT, (size_t)pn.ld * std::max(1, c->mk.sumD) * 8, c->st);
    GPX_TMP_ALLOC(&pn.sq, (size_t)pn.ld * c->mk.nparts * 8, c->st);
    GPX_CUDA(cudaMemcpyAsync(pn.raw, Xnew, (size_t)M * c->D * 8, cudaMemcpyHostToDevice, st));
    GPX_CHECK(launch_prep_multi(pn.raw, M, c->D, pn.ld, c->mk, pn.xT, pn.sq, c->mflag, st));
    c->total_launches++;
  } else
  GPX_CHECK(upload_points(c, Xnew, M, c->kp, pn));
  // Kx as [M][ld] (each new point one zero-padded column of length ld): thread-mapped operand = training points
  double* Kx = nullptr; double* Tx = nullptr;
  GPX_TMP_ALLOC(&Kx, (size_t)pn.ld * ld * 8, c->st);
  GPX_TMP_ALLOC(&Tx, (size_t)pn.ld * ld * 8, c->st);
  GPX_CUDA(cudaMemsetAsync(Kx, 0, (size_t)pn.ld * ld * 8, st));
  if (dG > 1) GPX_CUDA(cudaMemsetAsync(Tx, 0, (size_t)pn.ld * ld * 8, st));   // columns of other ranks stay zero
  KBuildParams kb;
  memset(&kb, 0, sizeof(kb));
  kb.rowsT = c->dXsT; kb.ld_rows = ld; kb.sq_rows = c->dsq;
  kb.colsT = pn.xT; kb.ld_cols = pn.ld; kb.sq_cols = pn.sq;
  kb.out = Kx; kb.ld = ld; kb.nrows = N; kb.ncols = M; kb.sym = 0; kb.same = 0; kb.kp = c->kp;
  int rc;
  if (c->multi) {
    KBuildMultiParams km;
    memset(&km, 0, sizeof(km));
    km.rowsT = c->mXsT; km.ld_rows = ld; km.sq_rows = c->msq; km.colsT = pn.xT; km.ld_cols = pn.ld; km.sq_cols = pn.sq;
    km.out = Kx; km.ld = ld; km.nrows = N; km.ncols = M; km.sym = 0; km.same = 0; km.mk = c->mk;
    rc = launch_kbuild_multi(km, (int)(ld / TILE), (int)(pn.ld / TILE), st);
  } else
  rc = launch_kbuild(kb, (int)(ld / TILE), (int)(pn.ld / TILE), st);
  c->total_launches++;
  // tmp = L^-1 Kx = U^T Kx, MAX_P columns per pass
  for (long m0 = 0; rc == 0 && m0 < M; m0 += MAX_P) {
    const int pc = (int)std::min<long>(MAX_P, M - m0);
    long ldu = ld;
    const double* Ud = c->dist ? dist_U(c, &ldu) : nullptr;   // sharded: the column-owned U storage (local column slots)
    rc = Ud ? launch_utv(Ud, ldu, c->Npad, pc, Kx + m0 * ld, Tx + m0 * ld, st, dG, drank, dNB, 1)
            : launch_utv(c->S, ld, c->Npad, pc, Kx + m0 * ld, Tx + m0 * ld, st);
    c->total_launches++;
  }
  if (!full_cov) {
    // diagonal variance: everything reduces on the device; only M (P + 1) doubles come back
    double* red = nullptr;   // [P][M] means, then [M] sums of squares
    if (rc == 0 && cudaMallocAsync((void**)&red, (size_t)(c->P + 1) * M * 8, c->st) != cudaSuccess) { gpx::set_error("gpx_predict: out of memory"); rc = -1; }
    if (rc == 0) rc = launch_col_dot(Kx, ld, N, M, c->P, c->dAlpha, ld, red, M, st);              // mu = Kx^T alpha
    if (rc == 0) rc = launch_col_sqnorm(Tx, ld, c->Npad, M, red + (size_t)c->P * M, st);          // sum_i tmp_i^2
    if (rc == 0 && dG > 1) rc = dist_allreduce_sum(c, red + (size_t)c->P * M, (size_t)M, st);
    c->total_launches += 2;
    std::vector<double> h((size_t)(c->P + 1) * M);
    if (rc == 0 && cudaMemcpyAsync(h.data(), red, h.size() * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) { gpx::set_error("gpx_predict: device failure"); rc = -1; }
    GPX_TMP_FREE(Kx, c->st); GPX_TMP_FREE(Tx, c->st);
    GPX_TMP_FREE(red, c->st);
    if (rc) return rc;
    for (long m = 0; m < M; m++) {
      for (int q = 0; q < c->P; q++) mu[m * c->P + q] = h[(size_t)q * M + m];
      // per-point Kdiag of the composite kernel with coregionalization parts, else the one Kdiag of every point
      var[m] = (c->multi && c->m_coreg ? composite_kdiag(c, Xnew + m * c->D) : c->kp.variance) - h[(size_t)c->P * M + m];
    }
    return 0;
  }
  std::vector<double> hK, hT;
  if (rc == 0) {
    hK.resize((size_t)M * ld); hT.resize((size_t)M * ld);
    if (cudaMemcpyAsync(hK.data(), Kx, hK.size() * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
    if (cudaMemcpyAsync(hT.data(), Tx, hT.size() * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
  }
  std::vector<double> hA((size_t)c->P * ld);
  if (rc == 0 && cudaMemcpyAsync(hA.data(), c->dAlpha, hA.size() * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
  if (cudaStreamSynchronize(st) != cudaSuccess) { gpx::set_error("gpx_predict: device failure"); rc = -1; }
  // sums over the training index of this rank's part, completed over the ranks below
  std::vector<double> ssq((size_t)M * M, 0.0);
  if (rc == 0) {
    for (long a = 0; a < M; a++)
      for (long b = 0; b < M; b++) {
        double s = 0.0;
        for (long i = 0; i < N; i++) s += hT[a * ld + i] * hT[b * ld + i];
        ssq[a + b * M] = s;
      }
    if (dG > 1) {
      if ((size_t)pn.ld * ld < ssq.size()) { gpx::set_error("gpx_predict: internal buffer size"); rc = -2; }
      if (rc == 0 && cudaMemcpyAsync(Kx, ssq.data(), ssq.size() * 8, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = -1;
      if (rc == 0) rc = dist_allreduce_sum(c, Kx, ssq.size(), st);
      if (rc == 0 && cudaMemcpyAsync(ssq.data(), Kx, ssq.size() * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
      if (cudaStreamSynchronize(st) != cudaSuccess) { gpx::set_error("gpx_predict: device failure"); rc = -1; }
    }
  }
  GPX_TMP_FREE(Kx, c->st); GPX_TMP_FREE(Tx, c->st);
  if (rc) return rc;
  // full covariance (small M): host epilogue mu = Kx^T alpha, var = Kxx - tmp^T tmp
  for (long m = 0; m < M; m++)
    for (int q = 0; q < c->P; q++) {
      double s = 0.0;
      for (long i = 0; i < N; i++) s += hK[m * ld + i] * hA[(size_t)q * ld + i];
      mu[m * c->P + q] = s;
    }
  std::vector<double> kxx((size_t)M * M);
  double lsv[MAX_D];
  for (int q = 0; q < MAX_D; q++) lsv[q] = c->kp.ls[q];
  if (c->multi) {   // K(Xnew, Xnew) of the composite kernel, built on the device
    PointSet pm;
    pm.n = M; pm.ld = (M + TILE - 1) / TILE * TILE; pm.st = c->st;
    double* dk = nullptr;
    GPX_TMP_ALLOC(&pm.raw, (size_t)M * c->D * 8, c->st);
    GPX_TMP_ALLOC(&pm.xT, (size_t)pm.ld * std::max(1, c->mk.sumD) * 8, c->st);
    GPX_TMP_ALLOC(&pm.sq, (size_t)pm.ld * c->mk.nparts * 8, c->st);
    GPX_TMP_ALLOC(&dk, (size_t)M * M * 8, c->st);
    GPX_CUDA(cudaMemcpyAsync(pm.raw, Xnew, (size_t)M * c->D * 8, cudaMemcpyHostToDevice, st));
    rc = launch_prep_multi(pm.raw, M, c->D, pm.ld, c->mk, pm.xT, pm.sq, c->mflag, st);
    KBuildMultiParams km;
    memset(&km, 0, sizeof(km));
    km.rowsT = pm.xT; km.ld_rows = pm.ld; km.sq_rows = pm.sq; km.colsT = pm.xT; km.ld_cols = pm.ld; km.sq_cols = pm.sq;
    km.out = dk; km.ld = M; km.nrows = M; km.ncols = M; km.sym = 0; km.same = 1; km.mk = c->mk;
    if (rc == 0) rc = launch_kbuild_multi(km, (int)(pm.ld / TILE), (int)(pm.ld / TILE), st);
    c->total_launches += 2;
    if (rc == 0 && cudaMemcpyAsync(kxx.data(), dk, (size_t)M * M * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) { gpx::set_error("gpx_predict: device failure"); rc = -1; }
    GPX_TMP_FREE(dk, c->st);
  } else
  rc = gpx_kern_K(c, c->kp.kind, c->kp.ard, c->kp.variance, lsv, Xnew, M, nullptr, M, c->D, kxx.data());
  if (rc) return rc;
  for (long a = 0; a < M; a++)
    for (long b = 0; b < M; b++) var[a + b * M] = kxx[a * M + b] - ssq[a + b * M];
  return 0;
}

}  // extern "C"
