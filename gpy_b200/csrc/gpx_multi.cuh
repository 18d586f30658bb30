// gpx_multi.cuh — composite kernels on the device (internal): K = sum over terms of products of parts, each part a
// stationary kernel on its own active dims, a White or a Bias kernel. Mirrors GPy/kern/src/add.py:60-99 (Add.K /
// update_gradients_full), prod.py:59-68,377-396 (Prod.K; each factor's gradient sees dL_dK times the other factors) and
// static.py:63-185 (White, Bias) and coregionalize.py:82-137 (Coregionalize: B[idx_i, idx_j] on the output-index column).
#pragma once
#include <algorithm>

#include "gpx_common.cuh"

namespace gpx {

constexpr int MAX_PARTS = 8;
constexpr int MAX_O = 16;          // outputs of a coregionalization part; its B lives at MultiKern::B + part * MAX_O * MAX_O

struct PartDev {
  int kind;          // GPX_RBF .. GPX_MATERN52, GPX_WHITE, GPX_BIAS, GPX_COREGIONALIZE
  int ard;
  int term;          // parts with equal `term` are multiplied, terms are summed (parts sorted by term)
  int D;             // active dims (0 for the static kinds)
  int xoff;          // first row of this part inside the stacked scaled-input SoA [sumD][ld]
  int odim;          // coregionalization: number of outputs O (B is O x O, row stride O); 0 otherwise
  double variance;   // 1 for a coregionalization part
  double inv_ls_iso;
};

struct MultiKern {
  int nparts;
  int sumD;
  PartDev part[MAX_PARTS];
  int dims[MAX_D];       // column of X behind stacked row (xoff + q)
  double ls[MAX_D];      // its lengthscale (ARD: per dim; iso: the part's single lengthscale repeated)
  const double* B;       // device, [MAX_PARTS][MAX_O * MAX_O]: B of every coregionalization part (uploaded per evaluation)
};

struct KBuildMultiParams {
  const double* rowsT; long ld_rows; const double* sq_rows;    // stacked SoA [sumD][ld] and [nparts][ld] of the ROW points
  const double* colsT; long ld_cols; const double* sq_cols;
  double* out; long ld;                                        // out[rowidx + colidx * ld]
  long nrows, ncols;
  int sym, same;                                               // as KBuildParams
  double diag_add;
  const double* diag_vec;                                      // sym mode: per-point noise added on the diagonal, or null
  MultiKern mk;
};

struct GradKinvMultiParams {
  const double* Kinv; long ld;
  const double* XsT; const double* sq; long ldx;               // stacked SoA of the training points
  const double* alpha;
  long N; int P; int nt;
  int part;                                                    // the part whose parameter sums are reduced by this launch
  int want_noise;                                              // also reduce tr(dL_dK) (done by the first launch only)
  double* partials;                                            // [nt*nt][nred] of THIS part (part_nred), zeroed by the caller
  double* dnoise_out;                                          // with want_noise: diag(dL_dK) per point, or null
  MultiKern mk;
};

struct FinalizeMultiParams {
  const double* partials[MAX_PARTS]; long ntiles;
  const double* logdet_part; long nt;
  const double* T; long ld; long N; int P;
  MultiKern mk;
  double* res;   // [0] lml, [1] logdet, [2] quad, [3] d/d noise, then per part [d/d variance, d/d lengthscale(s)] (static: variance
                 // only; coregionalization: the O x O sums S, row-major)
};

// bad: set to 1 when an output index of a coregionalization part lies outside [0, O) (that entry is then read as 0)
int launch_prep_multi(const double* X, long N, int Dfull, long ld, const MultiKern& mk, double* XsT, double* sq, int* bad,
                      cudaStream_t st);
int launch_kbuild_multi(const KBuildMultiParams& p, int row_tiles, int col_tiles, cudaStream_t st);
int launch_grad_kinv_multi(const GradKinvMultiParams& p, cudaStream_t st);
int launch_finalize_multi(const FinalizeMultiParams& f, cudaStream_t st);

inline int part_nl(const PartDev& pd) { return pd.kind >= GPX_WHITE ? 0 : (pd.ard ? pd.D : 1); }
// gradient entries of one part in the result vector, and reduction slots per tile ([variance, lengthscale(s) or S, noise])
inline int part_ngrad(const PartDev& pd) { return pd.kind == GPX_COREGIONALIZE ? pd.odim * pd.odim : 1 + part_nl(pd); }
inline int part_nred(const PartDev& pd) {
  return pd.kind == GPX_COREGIONALIZE ? pd.odim * pd.odim + 2 : std::max(1, part_nl(pd)) + 2;
}
// 8 + MAX_D + MAX_PARTS * (MAX_O^2 + 2) doubles hold every result layout
constexpr int RES_CAP = 8 + MAX_D + MAX_PARTS * (MAX_O * MAX_O + 2);

}  // namespace gpx
