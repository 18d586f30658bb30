// gpx_multi.cu — composite kernels (sums of products of stationary / White / Bias parts) evaluated on the device:
// covariance build, gradient reductions from the stored K^-1 and the final assembly. See gpx_multi.cuh for the references.
#include <algorithm>
#include <cstring>

#include "gpx_common.cuh"
#include "gpx_multi.cuh"

namespace gpx {

// ---------------------------------------------------------------------------------------------------------------
// prep: every part's active dims scaled the way its own Stationary._scaled_dist does (stationary.py:151-168: ARD divides
// by the lengthscale before the expansion, iso afterwards), stacked as SoA rows, plus per-part squared norms. A
// coregionalization part stores its output index truncated to an integer (coregionalize.py:88: np.asarray(X, dtype=int));
// an index outside [0, O) raises `bad` and is stored as 0, so that no later kernel reads outside B
// ---------------------------------------------------------------------------------------------------------------
__global__ void prep_multi_kernel(const double* __restrict__ X, long N, int Dfull, long ld, MultiKern mk,
                                  double* __restrict__ XsT, double* __restrict__ sq, int* __restrict__ bad) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ld) return;
  for (int p = 0; p < mk.nparts; p++) {
    const PartDev& pd = mk.part[p];
    double s = 0.0;
    for (int q = 0; q < pd.D; q++) {
      double v = 0.0;
      if (i < N) {
        v = X[i * Dfull + mk.dims[pd.xoff + q]];
        if (pd.ard) v = v / mk.ls[pd.xoff + q];
        if (pd.kind == GPX_COREGIONALIZE) {
          if (v > -1.0 && v < (double)pd.odim) {
            v = trunc(v);
          } else {
            *bad = 1;
            v = 0.0;
          }
        }
      }
      XsT[(long)(pd.xoff + q) * ld + i] = v;
      s += v * v;
    }
    sq[(long)p * ld + i] = s;
  }
}

int launch_prep_multi(const double* X, long N, int Dfull, long ld, const MultiKern& mk, double* XsT, double* sq, int* bad,
                      cudaStream_t st) {
  prep_multi_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, st>>>(X, N, Dfull, ld, mk, XsT, sq, bad);
  GPX_CUDA(cudaGetLastError());
  return 0;
}

// value of one part at a pair of points held in shared-memory tiles (row point il, column point jl), unit handling of the
// static kinds: White = variance on coincident points of the SAME set (static.py:75-79), Bias = variance (static.py:155-157);
// coregionalization: B[idx_i, idx_j] (coregionalize.py:88-108)
__device__ __forceinline__ double part_value(const MultiKern& mk, int p, const double* sR, const double* sC, const double* sSr,
                                             const double* sSc, int il, int jl, bool samept, double* r_out, double* dk_out) {
  const PartDev& pd = mk.part[p];
  if (pd.kind == GPX_COREGIONALIZE) {
    if (r_out) { *r_out = 0.0; *dk_out = 0.0; }
    const int a = (int)sR[pd.xoff * TILE + il], b = (int)sC[pd.xoff * TILE + jl];
    return mk.B[p * MAX_O * MAX_O + a * pd.odim + b];
  }
  if (pd.kind == GPX_BIAS) { if (r_out) { *r_out = 0.0; *dk_out = 0.0; } return 1.0; }
  if (pd.kind == GPX_WHITE) { if (r_out) { *r_out = 0.0; *dk_out = 0.0; } return samept ? 1.0 : 0.0; }
  double dot = 0.0;
  for (int q = 0; q < pd.D; q++) dot = fma(sR[(pd.xoff + q) * TILE + il], sC[(pd.xoff + q) * TILE + jl], dot);
  double r2 = sSr[p * TILE + il] + sSc[p * TILE + jl] - 2.0 * dot;
  if (samept) r2 = 0.0;
  r2 = fmax(r2, 0.0);
  const double rr = sqrt(r2) * pd.inv_ls_iso;
  if (r_out) {
    double k, dk;
    k_dk_of_r_unit(pd.kind, rr, k, dk);
    *r_out = rr; *dk_out = dk;
    return k;
  }
  return k_of_r_unit(pd.kind, rr);
}

__device__ __forceinline__ void load_tiles(const MultiKern& mk, const double* rowsT, long ld_rows, const double* sq_rows, int rt,
                                           const double* colsT, long ld_cols, const double* sq_cols, int ct, double* sR,
                                           double* sC, double* sSr, double* sSc) {
  for (int idx = threadIdx.x; idx < mk.sumD * TILE; idx += blockDim.x) {
    const int q = idx / TILE, m = idx % TILE;
    sR[idx] = rowsT[(long)q * ld_rows + (long)rt * TILE + m];
    sC[idx] = colsT[(long)q * ld_cols + (long)ct * TILE + m];
  }
  for (int idx = threadIdx.x; idx < mk.nparts * TILE; idx += blockDim.x) {
    const int q = idx / TILE, m = idx % TILE;
    sSr[idx] = sq_rows[(long)q * ld_rows + (long)rt * TILE + m];
    sSc[idx] = sq_cols[(long)q * ld_cols + (long)ct * TILE + m];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// covariance build: K = sum_t prod_{p in t} k_p (add.py:60-74, prod.py:59-68), `sym` mode = factor workspace image
// (lower tiles, zero upper tiles, identity padding, + (noise + jitter) on the diagonal: exact_gaussian_inference.py:55-56)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kbuild_multi_kernel(KBuildMultiParams p) {
  extern __shared__ __align__(128) unsigned char km_smem[];
  const MultiKern& mk = p.mk;
  double* sR = reinterpret_cast<double*>(km_smem);
  double* sC = sR + (size_t)mk.sumD * TILE;
  double* sSr = sC + (size_t)mk.sumD * TILE;
  double* sSc = sSr + (size_t)mk.nparts * TILE;
  const int ct = blockIdx.x, rt = blockIdx.y;
  const int tid = threadIdx.x, il = tid & (TILE - 1), half = tid >> 7;
  const long gi = (long)rt * TILE + il;
  double* outp = p.out + gi + ((long)ct * TILE + half * 64) * p.ld;
  if (p.sym && rt < ct) {
#pragma unroll 8
    for (int j = 0; j < 64; j++) outp[(long)j * p.ld] = 0.0;
    return;
  }
  load_tiles(mk, p.rowsT, p.ld_rows, p.sq_rows, rt, p.colsT, p.ld_cols, p.sq_cols, ct, sR, sC, sSr, sSc);
  __syncthreads();
  const bool row_valid = gi < p.nrows;
  for (int j = 0; j < 64; j++) {
    const int jl = half * 64 + j;
    const long gj = (long)ct * TILE + jl;
    const bool samept = p.same && gi == gj;
    double val = 0.0, prod = 1.0;
    int cur = mk.part[0].term;
    for (int q = 0; q < mk.nparts; q++) {
      if (mk.part[q].term != cur) { val += prod; prod = 1.0; cur = mk.part[q].term; }
      prod *= mk.part[q].variance * part_value(mk, q, sR, sC, sSr, sSc, il, jl, samept, nullptr, nullptr);
    }
    val += prod;
    if (p.sym) {
      if (gi == gj) val += p.diag_add + (p.diag_vec && row_valid ? p.diag_vec[gi] : 0.0);
      if (!row_valid || gj >= p.ncols) val = (gi == gj) ? 1.0 : 0.0;
      outp[(long)j * p.ld] = val;
    } else if (row_valid && gj < p.ncols) {
      outp[(long)j * p.ld] = val;
    }
  }
}

static size_t multi_tile_smem(const MultiKern& mk) { return (size_t)(2 * mk.sumD + 2 * mk.nparts) * TILE * 8 + 8 * (MAX_D + 2) * 8; }
// the gradient pass of a coregionalization part also bins every thread's row into O columns: [O][256] doubles, [256] ints
constexpr size_t COREG_SMEM = (size_t)MAX_O * 256 * 8 + 256 * 4;
constexpr int MULTI_SMEM_MAX = (2 * MAX_D + 2 * MAX_PARTS) * TILE * 8 + 8 * (MAX_D + 2) * 8;

int launch_kbuild_multi(const KBuildMultiParams& p, int row_tiles, int col_tiles, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    GPX_CUDA(cudaFuncSetAttribute(kbuild_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MULTI_SMEM_MAX));
    attr_set = true;
  }
  kbuild_multi_kernel<<<dim3(col_tiles, row_tiles), 256, multi_tile_smem(p.mk), st>>>(p);
  GPX_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// gradient reductions of ONE part from the stored K^-1: with dL_dK = 1/2 (alpha alpha^T - P K^-1) the part sees
// dL_dK o prod(other factors of its term) (prod.py:377-396; add.py:76-99 passes dL_dK through unchanged) and reduces it
// exactly like Stationary.update_gradients_full (stationary.py:193-243), White (static.py:88-92: trace) or Bias
// (static.py:172-173: sum). One CTA per lower 128 x 128 tile, thread-mapped index = row (contiguous in K^-1).
// A coregionalization part reduces to the O x O matrix S (coregionalize.py:130-137): every thread bins the columns of its row
// by idx_j in shared memory, then thread (a, b) sums, in thread order, the bins b of the threads whose row has idx_i = a; an
// off-diagonal tile also stands for its mirror tile, so it adds the bins a of the threads with idx_i = b (S + S^T of the
// tile). No atomics: every sum has a fixed order. The launch with want_noise also writes diag(dL_dK) to dnoise_out.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void grad_coreg_tile(const GradKinvMultiParams& p, const double* sR, const double* sC,
                                                const double* sSr, const double* sSc, double* sRed, int r, int c) {
  const MultiKern& mk = p.mk;
  const PartDev& me = mk.part[p.part];
  const int O = me.odim, nred = O * O + 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int il = tid & (TILE - 1), half = tid >> 7;
  const long gi = (long)r * TILE + il;
  double* sBin = sRed + 8 * (MAX_D + 2);                 // [O][256]
  int* sIdx = reinterpret_cast<int*>(sBin + MAX_O * 256);  // [256] idx_i of each thread's row, -1 = padding row
  for (int b = 0; b < O; b++) sBin[b * 256 + tid] = 0.0;
  sIdx[tid] = gi < p.N ? (int)sR[me.xoff * TILE + il] : -1;
  double gnoise = 0.0;
  const double* kcol = p.Kinv + gi + ((long)c * TILE + half * 64) * p.ld;
  if (gi < p.N) {
    for (int jj = 0; jj < 64; jj++) {
      const int jl = half * 64 + jj;
      const long gj = (long)c * TILE + jl;
      if (gj >= p.N) break;
      const bool samept = gi == gj;
      const double kinv = kcol[(long)jj * p.ld];
      double aa = 0.0;
      for (int q = 0; q < p.P; q++) aa = fma(p.alpha[(long)q * p.ldx + gi], p.alpha[(long)q * p.ldx + gj], aa);
      double dl = 0.5 * (aa - (double)p.P * kinv);
      if (samept) {
        gnoise += dl;
        if (p.dnoise_out) p.dnoise_out[gi] = dl;
      }
      for (int q = 0; q < mk.nparts; q++)
        if (q != p.part && mk.part[q].term == me.term)
          dl *= mk.part[q].variance * part_value(mk, q, sR, sC, sSr, sSc, il, jl, samept, nullptr, nullptr);
      sBin[(int)sC[me.xoff * TILE + jl] * 256 + tid] += dl;
    }
  }
  gnoise = warp_sum(gnoise);
  if (lane == 0) sRed[warp] = gnoise;
  __syncthreads();
  const bool mirror = r > c;
  if (tid < O * O) {
    const int a = tid / O, b = tid % O;
    double s = 0.0;
    for (int t = 0; t < 256; t++) {
      const int at = sIdx[t];
      if (at == a) s += sBin[b * 256 + t];
      if (mirror && at == b) s += sBin[a * 256 + t];
    }
    p.partials[((long)r * p.nt + c) * nred + 1 + tid] = s;
  }
  if (tid == 0) {
    double s = 0.0;
#pragma unroll
    for (int wdx = 0; wdx < 8; wdx++) s += sRed[wdx];
    p.partials[((long)r * p.nt + c) * nred] = 0.0;
    p.partials[((long)r * p.nt + c) * nred + nred - 1] = p.want_noise ? s : 0.0;
  }
}

template <int DREG>
__global__ void __launch_bounds__(256) grad_kinv_multi_kernel(GradKinvMultiParams p) {
  extern __shared__ __align__(128) unsigned char gm_smem[];
  const MultiKern& mk = p.mk;
  const int P = p.P;
  double* sR = reinterpret_cast<double*>(gm_smem);
  double* sC = sR + (size_t)mk.sumD * TILE;
  double* sSr = sC + (size_t)mk.sumD * TILE;
  double* sSc = sSr + (size_t)mk.nparts * TILE;
  double* sRed = sSc + (size_t)mk.nparts * TILE;      // [8 warps][nred]
  int r = (int)((sqrtf(8.f * (float)blockIdx.x + 1.f) - 1.f) * 0.5f);
  while (r * (r + 1) / 2 > (int)blockIdx.x) --r;
  while ((r + 1) * (r + 2) / 2 <= (int)blockIdx.x) ++r;
  const int c = blockIdx.x - r * (r + 1) / 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  load_tiles(mk, p.XsT, p.ldx, p.sq, r, p.XsT, p.ldx, p.sq, c, sR, sC, sSr, sSc);
  __syncthreads();
  if (mk.part[p.part].kind == GPX_COREGIONALIZE) {
    grad_coreg_tile(p, sR, sC, sSr, sSc, sRed, r, c);
    return;
  }
  const PartDev me = mk.part[p.part];
  const int D = me.D;
  const bool ard = me.ard != 0 && me.kind < GPX_WHITE;
  const int nl = me.kind >= GPX_WHITE ? 1 : (ard ? D : 1), nred = nl + 2;
  const int il = tid & (TILE - 1), half = tid >> 7;
  const long gi = (long)r * TILE + il;
  double xi[DREG], gq[DREG];
#pragma unroll
  for (int q = 0; q < DREG; q++) { gq[q] = 0.0; xi[q] = q < D ? sR[(me.xoff + q) * TILE + il] : 0.0; }
  const double w = (r > c) ? 2.0 : 1.0;
  double gvar = 0.0, giso = 0.0, gnoise = 0.0;
  const double* kcol = p.Kinv + gi + ((long)c * TILE + half * 64) * p.ld;
  if (gi < p.N) {
    for (int jj = 0; jj < 64; jj++) {
      const int jl = half * 64 + jj;
      const long gj = (long)c * TILE + jl;
      if (gj >= p.N) break;
      const bool samept = gi == gj;
      const double kinv = kcol[(long)jj * p.ld];
      double aa = 0.0;
      for (int q = 0; q < P; q++) aa = fma(p.alpha[(long)q * p.ldx + gi], p.alpha[(long)q * p.ldx + gj], aa);
      double dl = 0.5 * (aa - (double)P * kinv);
      if (samept) {
        gnoise += dl;
        if (p.dnoise_out) p.dnoise_out[gi] = dl;
      }
      for (int q = 0; q < mk.nparts; q++)       // the other factors of this part's term
        if (q != p.part && mk.part[q].term == me.term)
          dl *= mk.part[q].variance * part_value(mk, q, sR, sC, sSr, sSc, il, jl, samept, nullptr, nullptr);
      double rr, dk;
      const double k = part_value(mk, p.part, sR, sC, sSr, sSc, il, jl, samept, &rr, &dk);
      gvar = fma(w * k, dl, gvar);
      const double G = me.variance * dk * dl;
      if (ard) {
        const double tmpv = (rr != 0.0) ? w * G / rr : 0.0;     // stationary.py:205,225-232: 1/r with 1/0 := 0
#pragma unroll
        for (int q = 0; q < DREG; q++)
          if (q < D) {
            const double df = xi[q] - sC[(me.xoff + q) * TILE + jl];
            gq[q] = fma(tmpv, df * df, gq[q]);
          }
      } else {
        giso = fma(w * G, rr, giso);
      }
    }
  }
  gvar = warp_sum(gvar);
  gnoise = warp_sum(gnoise);
  if (lane == 0) { sRed[warp * nred] = gvar; sRed[warp * nred + nred - 1] = p.want_noise ? gnoise : 0.0; }
  if (ard) {
#pragma unroll
    for (int q = 0; q < DREG; q++)
      if (q < D) {
        const double s = warp_sum(gq[q]);
        if (lane == 0) sRed[warp * nred + 1 + q] = s;
      }
  } else {
    giso = warp_sum(giso);
    if (lane == 0) sRed[warp * nred + 1] = giso;
  }
  __syncthreads();
  if (tid < nred) {
    double s = 0.0;
#pragma unroll
    for (int wdx = 0; wdx < 8; wdx++) s += sRed[wdx * nred + tid];
    p.partials[((long)r * p.nt + c) * nred + tid] = s;
  }
}

template <int DREG>
static int launch_gkm_t(const GradKinvMultiParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    GPX_CUDA(cudaFuncSetAttribute(grad_kinv_multi_kernel<DREG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(MULTI_SMEM_MAX + COREG_SMEM)));
    attr_set = true;
  }
  grad_kinv_multi_kernel<DREG><<<grid, 256, smem, st>>>(p);
  GPX_CUDA(cudaGetLastError());
  return 0;
}

int launch_grad_kinv_multi(const GradKinvMultiParams& p, cudaStream_t st) {
  const int D = p.mk.part[p.part].D;
  const unsigned grid = (unsigned)(p.nt * (p.nt + 1) / 2);
  const size_t smem = multi_tile_smem(p.mk) + (p.mk.part[p.part].kind == GPX_COREGIONALIZE ? COREG_SMEM : 0);
  if (D <= 8) return launch_gkm_t<8>(p, grid, smem, st);
  if (D <= 16) return launch_gkm_t<16>(p, grid, smem, st);
  if (D <= 32) return launch_gkm_t<32>(p, grid, smem, st);
  return launch_gkm_t<64>(p, grid, smem, st);
}

// ---------------------------------------------------------------------------------------------------------------
// final assembly: fixed-order sums of the per-tile partials of every part, log-determinant, quadratic form
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) finalize_multi_kernel(FinalizeMultiParams f) {
  __shared__ double sh[256];
  const int tid = threadIdx.x;
  auto block_sum = [&](double s) {
    sh[tid] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) sh[tid] += sh[tid + o]; __syncthreads(); }
    const double tot = sh[0];
    __syncthreads();
    return tot;
  };
  double s = 0.0;
  for (long i = tid; i < f.nt; i += 256) s += f.logdet_part[i];
  const double logdet = block_sum(s);
  s = 0.0;
  for (int q = 0; q < f.P; q++)
    for (long i = tid; i < f.N; i += 256) { const double x = f.T[(long)q * f.ld + i]; s = fma(x, x, s); }
  const double quad = block_sum(s);
  if (tid == 0) {
    const double log2pi = 1.8378770664093453;
    f.res[0] = 0.5 * (-(double)f.N * f.P * log2pi - (double)f.P * logdet - quad);
    f.res[1] = logdet;
    f.res[2] = quad;
  }
  int off = 4;
  for (int p = 0; p < f.mk.nparts; p++) {
    const PartDev& pd = f.mk.part[p];
    const bool co = pd.kind == GPX_COREGIONALIZE;
    const bool stat = pd.kind >= GPX_WHITE;
    const int nl = co ? pd.odim * pd.odim : (stat ? 1 : (pd.ard ? pd.D : 1)), nred = nl + 2;
    for (int t = 0; t < nred; t++) {
      if (co && t == 0) continue;                                                      // no variance of its own
      s = 0.0;
      for (long i = tid; i < f.ntiles; i += 256) s += f.partials[p][i * nred + t];
      const double tot = block_sum(s);
      if (tid == 0) {
        if (t == nred - 1) { if (p == 0) f.res[3] = tot; }                             // tr(dL_dK) -> noise (gaussian.py:78-79)
        else if (co) f.res[off + t - 1] = tot;                                         // S (coregionalize.py:130-137)
        else if (t == 0) f.res[off] = tot;                                             // d/d variance (stationary.py:199)
        else if (!stat) f.res[off + t] = -tot / f.mk.ls[pd.xoff + (pd.ard ? t - 1 : 0)];   // stationary.py:210,213
      }
    }
    off += co ? nl : 1 + (stat ? 0 : nl);
  }
}

int launch_finalize_multi(const FinalizeMultiParams& f, cudaStream_t st) {
  finalize_multi_kernel<<<1, 256, 0, st>>>(f);
  GPX_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace gpx
