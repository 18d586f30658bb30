// gpx_ctx.cuh — the device context behind the opaque gpx_ctx of include/gpx.h (internal).
#pragma once
#include <vector>

#include "gpx_common.cuh"
#include "gpx_ozaki.cuh"
#include "gpx_multi.cuh"

struct DistState;
struct SparseState;

struct gpx_ctx {
  int device = 0;
  cudaStream_t st = nullptr;
  cudaStream_t st2 = nullptr;   // high-priority side stream: diagonal-block work + panel of the NEXT step (look-ahead)
  cudaStream_t st3 = nullptr;   // high-priority third stream (option "chain"): rest of the panel, digit split, copy-back, forward
                                // substitution -- everything of step k that the NEXT diagonal block does not wait for
  cudaEvent_t ev_kfirst = nullptr;   // chain schedule: the first block row of the covariance build is done (D(0) may start)
  bool kfirst_valid = false;
  int lookahead = 1;
  int fine = 1;                 // option "fine": 64 x 64-tile DMMA kernels in the diagonal-block chain (gpx_fine.cu); 0 = 128 x 128 tiles
  int chain = 1;                // option "chain": tcgen05 path: the chain D(k) -> panel rows of block k+1 -> update of diagonal block k+1
                                // (fp64 DMMA, fine tiles) -> D(k+1) runs alone on the side stream; 0 = round-2 schedule
  std::vector<cudaEvent_t> sync_ev;
  // data
  long N = 0, Npad = 0;
  int D = 0, P = 0;
  double* dX = nullptr;      // N x D row-major (as given)
  double* dXsT = nullptr;    // [D][Npad] scaled SoA
  double* dsq = nullptr;     // [Npad]
  double* dY = nullptr;      // [P][Npad]
  double* dT = nullptr;      // [P][Npad]  L^-1 y
  double* dAlpha = nullptr;  // [P][Npad]
  double* dUvPart = nullptr; // [KSPLIT][P][Npad]
  // workspace
  double* S = nullptr;       // Npad x Npad column-major: lower L, upper U
  double* Pbuf = nullptr;    // Npad x NB
  double* Tm = nullptr;      // NB x NB
  double* Ldiag = nullptr;   // nt tiles of 128x128
  double* Dinv = nullptr;    // nt tiles of 128x128
  double* logdet_part = nullptr;
  double* partials = nullptr;
  int* info = nullptr;
  double* res = nullptr;     // device result vector
  double* h_res = nullptr;   // pinned
  int* h_info = nullptr;     // pinned
  double* Kinv = nullptr;    // lazy, Npad x Npad (lower tiles)
  double* staging = nullptr; // lazy, N x N dense
  size_t staging_cap = 0;
  long NB = 0;               // outer block (0 = auto)
  // last evaluation
  bool have_eval = false;
  bool have_kinv = false;
  gpx::KernParams kp{};
  double noise = 0, jitter = 0, jitter_extra = 0;
  // heteroscedastic evaluation (gpx_exact_eval_het): per-point noise variances in, diag(dL_dK) out
  bool het = false;
  double* dNoiseVec = nullptr; double* dDnoise = nullptr; long het_cap = 0;
  // accounting
  gpx_stats stats{};
  int64_t total_launches = 0;
  int64_t eval_launches = 0;
  std::vector<cudaEvent_t> ev;
  int profile = 1;
  // ---- tcgen05 / Ozaki path (gpx_ozaki.cu): trailing update and K^-1 on the INT8 tensor cores ------------------------
  int ozaki = -1;              // option "ozaki": -1 = default (env GPX_OZAKI, else on), 0 = DMMA only, 1 = on where applicable
  int oz_dig_up = 7;           // digits per operand for the inverse-part / K^-1 tiles, which feed only the gradients
                               // (option "oz_dig_up"; 7 -> 28 digit pairs instead of 36, gradient error ~6e-10 at N = 16384)
  int oz_ctas = 0;             // option "oz_ctas": >0 = that many CTAs sharing the tile list evenly (persistent-style); 0 = default chunking
  int oz_tpc = 0;              // option "oz_tpc": consecutive tiles per CTA (0 = default 4)
  int oz_dbg = 0;              // measurement-only kernel variants (OzParams::dbg)
  int oz_u0 = 1;               // option "oz_u0": update the NEXT diagonal block first (own small launch) so that its factorisation starts
                               // before the rest of block column k+1 is updated
  int oz_sched = 0;            // option "oz_sched": 1 = panel GEMM on the main stream + persistent U2 leaving oz_reserve SMs to the
                               // diagonal-block chain; 0 = everything of step k+1 on the side stream, U launches in chunks of tiles
  int oz_reserve = 4;          // SMs left free by the persistent U2 launch for the side stream
  int oz_wide = 1;             // option "oz_wide": 1 = two-pass kernel with 128 x 128 tiles, 0 = one-pass kernel with 128 x 64 tiles
  int num_sms = 148;
  bool oz_ready = false;       // planes and K^-1 buffer allocated for (Npad, NB)
  bool oz_lists_ready = false; // tile lists built for (Npad, NB, oz_wide)
  gpx::OzPlanes ozp[2];        // digit planes of the current / next panel (look-ahead double buffer)
  int oz_panel = 1;            // option "oz_panel": the panel GEMM P = S(:, block) L_kk^-T outside the chain rows on the tensor cores too
                               // (digit planes of the block column and of L_kk^-1); 0 = fp64 DMMA panel GEMM
  gpx::OzPlanes ozpA, ozpB;    // its operands: block column of the workspace (Npad x NB), L_kk^-1 (NB x NB)
  uint32_t* oz_tiles = nullptr;
  double* dYres = nullptr;     // [P][Npad] running right-hand side of the forward substitution carried along the sweep
  double* dTfw = nullptr;      // [P][Npad] t = L^-1 y from that substitution (quadratic form of the LML)
  using OzStep = gpx::OzStep;
  std::vector<OzStep> oz_steps;
  bool oz_last = false;        // the last evaluation went through the Ozaki path (K^-1 already stored)
  // ---- composite kernels (gpx_multi.cu): the last evaluation used gpx_exact_eval_multi --------------------------------
  bool multi = false;
  gpx::MultiKern mk{};
  double* mXsT = nullptr;      // [sumD][Npad] stacked scaled inputs of the parts
  double* msq = nullptr;       // [nparts][Npad]
  double* mpartials = nullptr; // per part [nt*nt][part_nred], parts back to back
  long m_cap = 0;              // Npad the XsT / sq buffers were sized for
  size_t m_pcap = 0;           // doubles in mpartials: nt*nt * sum over the parts of part_nred
  bool m_coreg = false;        // the kernel has coregionalization parts (gpx_exact_eval_coreg)
  double* mB = nullptr;        // [MAX_PARTS][MAX_O * MAX_O] B of the coregionalization parts (MultiKern::B)
  std::vector<double> hB;      // host copy of mB (composite Kdiag of the jitter ladder and of gpx_predict)
  int* mflag = nullptr;        // set by prep_multi: an output index outside [0, O)
  struct DistState* dist = nullptr;   // multi-GPU state (gpx_dist.cu), null on a single GPU
  struct SparseState* sparse = nullptr;   // sparse-GP (VarDTC) state (gpx_sparse.cu)
};


namespace gpx {
constexpr int KSPLIT = 32;
GemmParams gemm_defaults();
// multi-GPU hooks implemented in gpx_dist.cu
int dist_set_data(gpx_ctx* c, const double* X, int64_t N, int D, const double* Y, int P);
int dist_exact_eval(gpx_ctx* c, double extra_jitter);
void dist_free(gpx_ctx* c);
int dist_get_L(gpx_ctx* c, double* out);                                       // collective: sharded woodbury_chol
long dist_block(const gpx_ctx* c);
const double* dist_U(const gpx_ctx* c, long* ld);                               // sharded: column-owned U storage                                             // NB of the sharded layout (0: none)
int dist_world(const gpx_ctx* c, int* rank, int* nranks);                       // (0, 1) without a communicator
int dist_allreduce_sum(gpx_ctx* c, double* buf, size_t count, cudaStream_t st);   // in place, on stream st
void sparse_free(gpx_ctx* c);
int factor_device(gpx_ctx* c, const double* dA, long lda, long N, double jitter0, int max_tries, double* logdet,
                  double* jitter_used);
int fill_kp(KernParams& kp, int kind, int ard, int D, double variance, const double* ls);
}  // namespace gpx
