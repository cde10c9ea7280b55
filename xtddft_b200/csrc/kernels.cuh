// Streaming (HBM-bound) kernels of the sigma path: layout pack/unpack, transposes, the grid f_xc weighting
// with warp-shuffle reductions, density-fitted Coulomb blocks, rank-1 / diagonal local terms and the
// Davidson vector primitives.  All fp64, coalesced along the contiguous index, grids sized from the data.
#pragma once
#include "common.cuh"

namespace xtd {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum; result valid in thread 0 (and broadcast through smem to all when bcast)
template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double* sm) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sm[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = (l < THREADS / 32) ? sm[l] : 0.0;
    r = warp_sum(r);
    if (l == 0) sm[0] = r;
  }
  __syncthreads();
  r = sm[0];
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------------
// layout: external vector <-> padded internal block  (sparse maps built by the host plan)
// ------------------------------------------------------------------------------------------------------
// Z[x][i][a] (ld) = sum_k val[k] * zext[x][col[k]],  rows r = i*nv + a
__global__ void pack_kernel(double* __restrict__ Z, long ldz, long z_vec_stride, int nv, long nrows,
                            const long* __restrict__ indptr, const long* __restrict__ cols, const double* __restrict__ vals,
                            const double* __restrict__ zext, long ext_dim, int nvec) {
  const long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (r >= nrows || x >= nvec) return;
  const long k0 = indptr[r], k1 = indptr[r + 1];
  double acc = 0.0;
  const double* zx = zext + (long)x * ext_dim;
  for (long k = k0; k < k1; ++k) acc += vals[k] * zx[cols[k]];
  const long i = r / nv, a = r - i * nv;
  Z[(long)x * z_vec_stride + i * ldz + a] = acc;
}

// the same gather, also writing the transposed copy ZT[x][a][i] (small problems: one launch instead of pack + transpose)
__global__ void pack_t_kernel(double* __restrict__ Z, long ldz, long z_vec_stride, double* __restrict__ ZT, long ldzt, long zt_vec_stride, int nv,
                              long nrows, const long* __restrict__ indptr, const long* __restrict__ cols, const double* __restrict__ vals,
                              const double* __restrict__ zext, long ext_dim, int nvec) {
  const long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (r >= nrows || x >= nvec) return;
  const long k0 = indptr[r], k1 = indptr[r + 1];
  double acc = 0.0;
  const double* zx = zext + (long)x * ext_dim;
  for (long k = k0; k < k1; ++k) acc += vals[k] * zx[cols[k]];
  const long i = r / nv, a = r - i * nv;
  Z[(long)x * z_vec_stride + i * ldz + a] = acc;
  ZT[(long)x * zt_vec_stride + a * ldzt + i] = acc;
}

// hz[x][e] = sum_k val[k] * SIG[ chan_base[ch[k]] + x*chan_vec_stride[ch[k]] + off[k] ]
struct UnpackChan {
  long base[2];
  long vec_stride[2];
};
__global__ void unpack_kernel(double* __restrict__ hz, long ext_dim, int nvec, const long* __restrict__ indptr,
                              const long* __restrict__ offs, const signed char* __restrict__ chans,
                              const double* __restrict__ vals, const double* __restrict__ sig, UnpackChan uc) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (e >= ext_dim || x >= nvec) return;
  double acc = 0.0;
  for (long k = indptr[e]; k < indptr[e + 1]; ++k) {
    const int c = chans[k];
    acc += vals[k] * sig[uc.base[c] + (long)x * uc.vec_stride[c] + offs[k]];
  }
  hz[(long)x * ext_dim + e] = acc;
}

// dst[b][c][r] = src[b][r][c]   (32x32 tiles through shared memory)
__global__ void transpose_kernel(double* __restrict__ dst, long ldd, long dst_batch, const double* __restrict__ src, long lds,
                                 long src_batch, int rows, int cols) {
  __shared__ double tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const double* s = src + (long)b * src_batch;
  double* d = dst + (long)b * dst_batch;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int r = r0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < rows && c < cols) ? s[(long)r * lds + c] : 0.0;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int c = c0 + j, r = r0 + threadIdx.x;
    if (c < cols && r < rows) d[(long)c * ldd + r] = tile[threadIdx.x][j];
  }
}

// ZTs[x][a][j] = w[jblk(j)][bblk(a)] * ZT[x][a][j]   (block weights of the exchange build)
struct BlockSplit {
  int o2off;   // start of the 2nd occ block (>= no means single block)
  int v2off;
  double w[2][2];  // [jblk][bblk]
};
__global__ void scale_blocks_kernel(double* __restrict__ dst, const double* __restrict__ src, long ld, long batch, int nv, int no,
                                    BlockSplit bs) {
  const int x = blockIdx.z;
  const int a = blockIdx.y;
  const int bb = a >= bs.v2off ? 1 : 0;
  const double* s = src + (long)x * batch + (long)a * ld;
  double* d = dst + (long)x * batch + (long)a * ld;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < no; j += gridDim.x * blockDim.x)
    d[j] = s[j] * bs.w[j >= bs.o2off ? 1 : 0][bb];
}

// dst[r][c] (ldd) = src[r][c] (lds), optional lower-triangular packed source (PySCF cderi rows)
__global__ void pad_copy_kernel(double* __restrict__ dst, long ldd, long dst_batch, const double* __restrict__ src, long lds,
                                long src_batch, int rows, int cols) {
  const int b = blockIdx.z;
  const int r = blockIdx.y;
  const double* s = src + (long)b * src_batch + (long)r * lds;
  double* d = dst + (long)b * dst_batch + (long)r * ldd;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x) d[c] = s[c];
}
__global__ void unpack_tril_kernel(double* __restrict__ dst, long ldd, long dst_batch, const double* __restrict__ src,
                                   long src_batch, int n) {
  const int b = blockIdx.z;
  const int r = blockIdx.y;
  const double* s = src + (long)b * src_batch;
  double* d = dst + (long)b * dst_batch + (long)r * ldd;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n; c += gridDim.x * blockDim.x) {
    const long hi = r > c ? r : c, lo = r > c ? c : r;
    d[c] = s[hi * (hi + 1) / 2 + lo];
  }
}

// dst[i][p] = (idx[p] >= 0) ? C[i][idx[p]] : 0   (gather MO columns; zero pad orbitals)
__global__ void gather_cols_kernel(double* __restrict__ dst, long ldd, const double* __restrict__ C, long ldc, int nao,
                                   const int* __restrict__ idx, int n) {
  const int i = blockIdx.y;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const int k = idx[p];
    dst[(long)i * ldd + p] = k >= 0 ? C[(long)i * ldc + k] : 0.0;
  }
}

// ------------------------------------------------------------------------------------------------------
// grid kernel weighting: Y (half-transformed trial density on the grid) -> A (weighted occupied values)
//   rho^s_c(g,x) = sum_o Y^s_c[g,x,o] phi^s_0[g,o] (+ Y^s_0 phi^s_c for gradient components)   warp-shuffle reduction
//   wv = f_xc . rho  (kernel kind), A^s_0 = wv_0 phi_0 + sum_k wv_k phi_k,  A^s_k = wv_k phi_0
// One warp per grid point, lanes over the occupied index, loop over trial vectors.  In place (A overwrites Y).
// ------------------------------------------------------------------------------------------------------
enum { XC_KIND_UKS = 1, XC_KIND_ALDA0 = 2, XC_KIND_MCOL = 3 };

struct XcArgs {
  int nch, nvec, gb;
  long g0;                 // first grid point of this chunk (index into phi / kernel arrays)
  double* Y[2];            // [nvar][gb][ldY]
  long ldY[2];
  long y_comp[2];          // component stride of Y
  const double* phi[2];    // [nvar][ng][ldphi]
  long ldphi[2];
  long phi_comp[2];
  int no[2];
  const double* wf;        // per-point kernel data: UKS [ng][(2 nvar)^2] (weighted), ALDA0 [ng], MCOL [ng][nvar^2] (2 w f)
};

// XU trial vectors are processed together (independent loads in flight before the first shuffle reduction: the kernel
// is latency-bound otherwise); W = 2 uses 16-byte accesses (needs an even occupied count so that every
// (vector, component) row segment stays 16-byte aligned).
template <int W>
struct XcVec;
template <>
struct XcVec<1> {
  double v[1];
  __device__ __forceinline__ void load(const double* p) { v[0] = *p; }
  __device__ __forceinline__ void store(double* p) const { *p = v[0]; }
};
template <>
struct XcVec<2> {
  double v[2];
  __device__ __forceinline__ void load(const double* p) {
    const double2 t = *reinterpret_cast<const double2*>(p);
    v[0] = t.x; v[1] = t.y;
  }
  __device__ __forceinline__ void store(double* p) const { *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]); }
};

// TAU (value + gradient AO components only): the kernel tables carry a fifth component, the kinetic-energy density
//   tau(g,x) = 1/2 sum_k sum_o Y_k phi_k,   and its potential adds  A_k += 1/2 wv_tau phi_k   (meta-GGA, no Laplacian).
template <int NVAR, int KIND, int XU, int W, bool TAU = false>
__global__ void __launch_bounds__(256) xc_weight_kernel(const XcArgs a) {
  static_assert(!TAU || NVAR == 4, "the tau component needs value + gradient AO components");
  const int lane = threadIdx.x & 31;
  const long g = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (g >= a.gb) return;
  constexpr int NCH = (KIND == XC_KIND_UKS) ? 2 : 1;
  constexpr int NK = TAU ? 5 : NVAR;          // components of the response density / kernel tables
  constexpr int NR = NCH * NK;
  // kernel row for this grid point (kept in registers across the vector loop)
  double fk[(KIND == XC_KIND_UKS) ? NR : (KIND == XC_KIND_MCOL ? NK : 1)];
  if (KIND == XC_KIND_UKS) {
    // lane l < NR owns output component l = t*NK + d and needs wf[g][l][*]
    const double* row = a.wf + (a.g0 + g) * (long)(NR * NR);
#pragma unroll
    for (int q = 0; q < NR; ++q) fk[q] = (lane < NR) ? row[lane * NR + q] : 0.0;
  } else if (KIND == XC_KIND_MCOL) {
    const double* row = a.wf + (a.g0 + g) * (long)(NK * NK);
#pragma unroll
    for (int q = 0; q < NK; ++q) fk[q] = (lane < NK) ? row[lane * NK + q] : 0.0;
  } else {
    fk[0] = a.wf[a.g0 + g];
  }
  for (int x0 = 0; x0 < a.nvec; x0 += XU) {
    double rho[XU][NR];
#pragma unroll
    for (int u = 0; u < XU; ++u)
#pragma unroll
      for (int q = 0; q < NR; ++q) rho[u][q] = 0.0;
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s];
      const double* yb = a.Y[s] + g * a.ldY[s] + (long)x0 * no;
      const double* p = a.phi[s] + (a.g0 + g) * a.ldphi[s];
      for (int o = lane * W; o < no; o += 32 * W) {
        XcVec<W> pc[NVAR];
#pragma unroll
        for (int k = 0; k < NVAR; ++k) pc[k].load(p + k * a.phi_comp[s] + o);
        XcVec<W> yc[XU][NVAR];
#pragma unroll
        for (int u = 0; u < XU; ++u)
          if (x0 + u < a.nvec) {
#pragma unroll
            for (int k = 0; k < NVAR; ++k) yc[u][k].load(yb + (long)u * no + k * a.y_comp[s] + o);
          }
#pragma unroll
        for (int u = 0; u < XU; ++u)
          if (x0 + u < a.nvec) {
#pragma unroll
            for (int e = 0; e < W; ++e) {
              rho[u][s * NK] += yc[u][0].v[e] * pc[0].v[e];
#pragma unroll
              for (int k = 1; k < NVAR; ++k) {
                rho[u][s * NK + k] += yc[u][k].v[e] * pc[0].v[e] + yc[u][0].v[e] * pc[k].v[e];
                if (TAU) rho[u][s * NK + 4] += 0.5 * yc[u][k].v[e] * pc[k].v[e];
              }
            }
          }
      }
    }
#pragma unroll
    for (int u = 0; u < XU; ++u)
#pragma unroll
      for (int q = 0; q < NR; ++q) rho[u][q] = warp_sum(rho[u][q]);
    double wv[XU][NR];
#pragma unroll
    for (int u = 0; u < XU; ++u) {
      if (KIND == XC_KIND_UKS) {
        double mine = 0.0;
#pragma unroll
        for (int q = 0; q < NR; ++q) mine += fk[q] * rho[u][q];      // wv[t,d] = sum_{s,c} wf[g][t,d][s,c] rho[s,c]
#pragma unroll
        for (int q = 0; q < NR; ++q) wv[u][q] = __shfl_sync(0xffffffffu, mine, q);
      } else if (KIND == XC_KIND_MCOL) {
        double mine = 0.0;
#pragma unroll
        for (int q = 0; q < NK; ++q) mine += fk[q] * rho[u][q];      // wv[a] = sum_b (2 w f[b,a]) rho[b]
#pragma unroll
        for (int q = 0; q < NK; ++q) wv[u][q] = __shfl_sync(0xffffffffu, mine, q);
      } else {
        wv[u][0] = rho[u][0] * fk[0];
      }
    }
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s];
      double* yb = a.Y[s] + g * a.ldY[s] + (long)x0 * no;
      const double* p = a.phi[s] + (a.g0 + g) * a.ldphi[s];
      for (int o = lane * W; o < no; o += 32 * W) {
        XcVec<W> pc[NVAR];
        pc[0].load(p + o);
        if (KIND != XC_KIND_ALDA0) {
#pragma unroll
          for (int k = 1; k < NVAR; ++k) pc[k].load(p + k * a.phi_comp[s] + o);
        }
#pragma unroll
        for (int u = 0; u < XU; ++u)
          if (x0 + u < a.nvec) {
            XcVec<W> out;
#pragma unroll
            for (int e = 0; e < W; ++e) out.v[e] = wv[u][s * NK] * pc[0].v[e];
            if (KIND != XC_KIND_ALDA0) {
#pragma unroll
              for (int k = 1; k < NVAR; ++k) {
                XcVec<W> ok;
#pragma unroll
                for (int e = 0; e < W; ++e) {
                  out.v[e] += wv[u][s * NK + k] * pc[k].v[e];
                  ok.v[e] = wv[u][s * NK + k] * pc[0].v[e];
                  if (TAU) ok.v[e] += 0.5 * wv[u][s * NK + 4] * pc[k].v[e];
                }
                ok.store(yb + (long)u * no + k * a.y_comp[s] + o);
              }
            }
            out.store(yb + (long)u * no + o);
          }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// Value + gradient kernels with two GEMMs per direction instead of four ("split gradient" form):
//   Y0[g,x,o] = sum_v phiv_0[g,v] z[x,o,v]      T[g,x,v] = sum_o phi_0[g,o] z[x,o,v]          (the two forward GEMMs)
//   rho_0 = sum_o Y0 phi_0      rho_k = sum_o Y0 phi_k + sum_v T phiv_k                        (k = x, y, z)
//   wv = f_xc . rho
//   A[g,x,o] = wv_0 phi_0 + sum_k wv_k phi_k   (over Y0)       B[g,x,v] = sum_k wv_k phiv_k    (over T)
//   sigma[x,o,v] += sum_g A[g,x,o] phiv_0[g,v] + sum_g phi_0[g,o] B[g,x,v]                     (the two backward GEMMs)
// The gradient of the orbital product is split as (grad phi_o) phi_v + phi_o (grad phi_v); the second half is carried
// by the virtual-side buffers T / B, which this kernel streams once (read T, write B in place).  One warp per grid
// point, lanes over the orbital index, XU trial vectors in flight.
// ------------------------------------------------------------------------------------------------------
struct XcArgs2 {
  int nch, nvec, gb;
  long g0;
  double* Y[2];            // [gb][ldY]          Y0 in, A out
  long ldY[2];
  double* T[2];            // [nvec][t_rows][ldT]    T in, B out   (t_rows >= gb: rows per trial vector, 0 = gb)
  long ldT[2];
  long t_rows = 0;
  const double* phi[2];    // [4][ng][ldphi]
  long ldphi[2], phi_comp[2];
  const double* phiv[2];   // [4][ng][ldphiv]
  long ldphiv[2], phiv_comp[2];
  int no[2], nv[2];
  const double* wf;        // UKS [ng][64] (weighted), MCOL [ng][16] (2 w f)
};

// One CTA per grid point, one warp per trial vector: the orbital values of the point (4 occupied components, 3 virtual
// gradient components per channel) are staged in shared memory once and shared by all vectors, so every byte of Y0 / T
// and of the MO values is read from HBM exactly once.
__host__ __device__ inline long xc_split_smem_doubles(int nch, const int* no, const int* nv) {
  long n = 0;
  for (int s = 0; s < nch; ++s) n += 4L * ((no[s] + 1) & ~1) + 3L * ((nv[s] + 1) & ~1);
  return n;
}

template <int KIND, int W>
__global__ void __launch_bounds__(512, 2) xc_weight_split_kernel(const XcArgs2 a) {
  constexpr int NVAR = 4;
  constexpr int NCH = (KIND == XC_KIND_UKS) ? 2 : 1;
  constexpr int NR = NCH * NVAR;
  extern __shared__ __align__(16) double xc_sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const long g = blockIdx.x;
  // ---- stage the MO values of this point ----------------------------------------------------------------
  double* sphi[NCH];
  double* sphiv[NCH];
  int nop[NCH], nvp[NCH];
  {
    double* cur = xc_sm;
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      nop[s] = (a.no[s] + 1) & ~1;
      nvp[s] = (a.nv[s] + 1) & ~1;
      sphi[s] = cur; cur += 4 * nop[s];
      sphiv[s] = cur; cur += 3 * nvp[s];
      const double* p = a.phi[s] + (a.g0 + g) * a.ldphi[s];
      const double* pv = a.phiv[s] + (a.g0 + g) * a.ldphiv[s];
      // 16-byte loads, one independent load per component in flight (the rows are padded with zeros past an odd orbital count)
#pragma unroll
      for (int k = 0; k < 4; ++k)
        for (int o = threadIdx.x * 2; o < nop[s]; o += blockDim.x * 2)
          *reinterpret_cast<double2*>(sphi[s] + k * nop[s] + o) = *reinterpret_cast<const double2*>(p + k * a.phi_comp[s] + o);
#pragma unroll
      for (int k = 0; k < 3; ++k)
        for (int v = threadIdx.x * 2; v < nvp[s]; v += blockDim.x * 2)
          *reinterpret_cast<double2*>(sphiv[s] + k * nvp[s] + v) = *reinterpret_cast<const double2*>(pv + (k + 1) * a.phiv_comp[s] + v);
    }
  }
  double fk[(KIND == XC_KIND_UKS) ? NR : NVAR];
  if (KIND == XC_KIND_UKS) {
    const double* row = a.wf + (a.g0 + g) * (long)(NR * NR);
#pragma unroll
    for (int q = 0; q < NR; ++q) fk[q] = (lane < NR) ? row[lane * NR + q] : 0.0;
  } else {
    const double* row = a.wf + (a.g0 + g) * (long)(NVAR * NVAR);
#pragma unroll
    for (int q = 0; q < NVAR; ++q) fk[q] = (lane < NVAR) ? row[lane * NVAR + q] : 0.0;
  }
  __syncthreads();
  for (int x = warp; x < a.nvec; x += nwarps) {
    double rho[NR];
#pragma unroll
    for (int q = 0; q < NR; ++q) rho[q] = 0.0;
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s], nv = a.nv[s];
      const double* yb = a.Y[s] + g * a.ldY[s] + (long)x * no;
#pragma unroll 2
      for (int o = lane * W; o < no; o += 32 * W) {
        XcVec<W> y;
        y.load(yb + o);
#pragma unroll
        for (int e = 0; e < W; ++e)
#pragma unroll
          for (int k = 0; k < NVAR; ++k) rho[s * NVAR + k] += y.v[e] * sphi[s][k * nop[s] + o + e];
      }
      const double* tb = a.T[s] + ((long)x * (a.t_rows ? a.t_rows : a.gb) + g) * a.ldT[s];
#pragma unroll 2
      for (int v = lane * 2; v < nv; v += 64) {
        XcVec<2> t;
        t.load(tb + v);
        const double t1 = (v + 1 < nv) ? t.v[1] : 0.0;       // past an odd nv the buffer holds no data
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double2 pv = *reinterpret_cast<const double2*>(sphiv[s] + k * nvp[s] + v);
          rho[s * NVAR + 1 + k] += t.v[0] * pv.x + t1 * pv.y;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < NR; ++q) rho[q] = warp_sum(rho[q]);
    double wv[NR];
    {
      double mine = 0.0;
      constexpr int NQ = (KIND == XC_KIND_UKS) ? NR : NVAR;
#pragma unroll
      for (int q = 0; q < NQ; ++q) mine += fk[q] * rho[q];
#pragma unroll
      for (int q = 0; q < NQ; ++q) wv[q] = __shfl_sync(0xffffffffu, mine, q);
    }
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s], nv = a.nv[s];
      double* yb = a.Y[s] + g * a.ldY[s] + (long)x * no;
#pragma unroll 2
      for (int o = lane * W; o < no; o += 32 * W) {
        XcVec<W> out;
#pragma unroll
        for (int e = 0; e < W; ++e) {
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < NVAR; ++k) acc += wv[s * NVAR + k] * sphi[s][k * nop[s] + o + e];
          out.v[e] = acc;
        }
        out.store(yb + o);
      }
      double* tb = a.T[s] + ((long)x * (a.t_rows ? a.t_rows : a.gb) + g) * a.ldT[s];
#pragma unroll 2
      for (int v = lane * 2; v < nv; v += 64) {
        double2 acc = make_double2(0.0, 0.0);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double2 pv = *reinterpret_cast<const double2*>(sphiv[s] + k * nvp[s] + v);
          acc.x += wv[s * NVAR + 1 + k] * pv.x;
          acc.y += wv[s * NVAR + 1 + k] * pv.y;
        }
        *reinterpret_cast<double2*>(tb + v) = acc;           // the staged value past an odd nv is 0
      }
    }
  }
}

// The same step for SMALL batches of trial vectors (a Z-vector solve applies the operator to one vector at a time, the last Davidson
// cycles to a few): with one warp per trial vector a CTA would be one or two warps, each staging ~50 KB of MO values by itself and
// four of them resident per SM -- latency-bound (config 4, one vector: 84 ms against 8 ms of HBM time).  Here the eight warps of a
// CTA share the grid point by ORBITAL range: all 256 threads stage the point, every warp accumulates the partial densities of its
// slice for XB vectors at a time, one shared-memory reduction (double-buffered: one barrier per batch) combines them, every warp
// forms the potentials and writes its slice back.  Each byte of Y0 / T and of the MO values is still read from HBM exactly once.
template <int KIND, int W, int XB>
__global__ void __launch_bounds__(256, (XB >= 4 ? 2 : 3)) xc_weight_split_op_kernel(const XcArgs2 a) {
  constexpr int NVAR = 4;
  constexpr int NCH = (KIND == XC_KIND_UKS) ? 2 : 1;
  constexpr int NR = NCH * NVAR;
  constexpr int NWARPS = 8;
  extern __shared__ __align__(16) double xc_sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long g = blockIdx.x;
  double* sphi[NCH];
  double* sphiv[NCH];
  int nop[NCH], nvp[NCH];
  double* cur = xc_sm;
#pragma unroll
  for (int s = 0; s < NCH; ++s) {
    nop[s] = (a.no[s] + 1) & ~1;
    nvp[s] = (a.nv[s] + 1) & ~1;
    sphi[s] = cur; cur += 4 * nop[s];
    sphiv[s] = cur; cur += 3 * nvp[s];
    const double* p = a.phi[s] + (a.g0 + g) * a.ldphi[s];
    const double* pv = a.phiv[s] + (a.g0 + g) * a.ldphiv[s];
    // 16-byte loads, one independent load per component in flight (the rows are padded with zeros past an odd orbital count)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      for (int o = threadIdx.x * 2; o < nop[s]; o += blockDim.x * 2)
        *reinterpret_cast<double2*>(sphi[s] + k * nop[s] + o) = *reinterpret_cast<const double2*>(p + k * a.phi_comp[s] + o);
#pragma unroll
    for (int k = 0; k < 3; ++k)
      for (int v = threadIdx.x * 2; v < nvp[s]; v += blockDim.x * 2)
        *reinterpret_cast<double2*>(sphiv[s] + k * nvp[s] + v) = *reinterpret_cast<const double2*>(pv + (k + 1) * a.phiv_comp[s] + v);
  }
  double* red = cur;                     // [2][NWARPS][XB][NR] partial densities
  double fk[NR];
  {
    const double* row = a.wf + (a.g0 + g) * (long)(NR * NR);
#pragma unroll
    for (int q = 0; q < NR; ++q) fk[q] = (lane < NR) ? row[lane * NR + q] : 0.0;
  }
  __syncthreads();
  const long t_rows = a.t_rows ? a.t_rows : a.gb;
  int buf = 0;
  for (int x0 = 0; x0 < a.nvec; x0 += XB, buf ^= 1) {
    double rho[XB][NR];
#pragma unroll
    for (int xi = 0; xi < XB; ++xi)
#pragma unroll
      for (int q = 0; q < NR; ++q) rho[xi][q] = 0.0;
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s], nv = a.nv[s];
      const double* yb = a.Y[s] + g * a.ldY[s];
      for (int o = (warp * 32 + lane) * W; o < no; o += NWARPS * 32 * W) {
        double ph[NVAR][W];
#pragma unroll
        for (int k = 0; k < NVAR; ++k)
#pragma unroll
          for (int e = 0; e < W; ++e) ph[k][e] = sphi[s][k * nop[s] + o + e];
#pragma unroll
        for (int xi = 0; xi < XB; ++xi) {
          if (x0 + xi < a.nvec) {
            XcVec<W> y;
            y.load(yb + (long)(x0 + xi) * no + o);
#pragma unroll
            for (int e = 0; e < W; ++e)
#pragma unroll
              for (int k = 0; k < NVAR; ++k) rho[xi][s * NVAR + k] += y.v[e] * ph[k][e];
          }
        }
      }
      for (int v = (warp * 32 + lane) * 2; v < nv; v += NWARPS * 64) {
        double2 pv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) pv[k] = *reinterpret_cast<const double2*>(sphiv[s] + k * nvp[s] + v);
#pragma unroll
        for (int xi = 0; xi < XB; ++xi) {
          if (x0 + xi < a.nvec) {
            XcVec<2> t;
            t.load(a.T[s] + ((long)(x0 + xi) * t_rows + g) * a.ldT[s] + v);
            const double t1 = (v + 1 < nv) ? t.v[1] : 0.0;       // past an odd nv the buffer holds no data
#pragma unroll
            for (int k = 0; k < 3; ++k) rho[xi][s * NVAR + 1 + k] += t.v[0] * pv[k].x + t1 * pv[k].y;
          }
        }
      }
    }
    double* rb = red + (long)buf * NWARPS * XB * NR;
#pragma unroll
    for (int xi = 0; xi < XB; ++xi)
#pragma unroll
      for (int q = 0; q < NR; ++q) {
        const double v = warp_sum(rho[xi][q]);
        if (lane == 0) rb[(warp * XB + xi) * NR + q] = v;
      }
    __syncthreads();
    double wv[XB][NR];
#pragma unroll
    for (int xi = 0; xi < XB; ++xi) {
      // lane q < NR: total density component q of vector xi, then mine = sum_q' fk[q'] rho[q'] and a broadcast of the results
      double tot = 0.0;
      if (lane < NR)
#pragma unroll
        for (int w = 0; w < NWARPS; ++w) tot += rb[(w * XB + xi) * NR + lane];
      double mine = 0.0;
#pragma unroll
      for (int q = 0; q < NR; ++q) mine += fk[q] * __shfl_sync(0xffffffffu, tot, q);
#pragma unroll
      for (int q = 0; q < NR; ++q) wv[xi][q] = __shfl_sync(0xffffffffu, mine, q);
    }
#pragma unroll
    for (int s = 0; s < NCH; ++s) {
      const int no = a.no[s], nv = a.nv[s];
      double* yb = a.Y[s] + g * a.ldY[s];
      for (int o = (warp * 32 + lane) * W; o < no; o += NWARPS * 32 * W) {
        double ph[NVAR][W];
#pragma unroll
        for (int k = 0; k < NVAR; ++k)
#pragma unroll
          for (int e = 0; e < W; ++e) ph[k][e] = sphi[s][k * nop[s] + o + e];
#pragma unroll
        for (int xi = 0; xi < XB; ++xi) {
          if (x0 + xi < a.nvec) {
            XcVec<W> out;
#pragma unroll
            for (int e = 0; e < W; ++e) {
              double acc = 0.0;
#pragma unroll
              for (int k = 0; k < NVAR; ++k) acc += wv[xi][s * NVAR + k] * ph[k][e];
              out.v[e] = acc;
            }
            out.store(yb + (long)(x0 + xi) * no + o);
          }
        }
      }
      for (int v = (warp * 32 + lane) * 2; v < nv; v += NWARPS * 64) {
        double2 pv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) pv[k] = *reinterpret_cast<const double2*>(sphiv[s] + k * nvp[s] + v);
#pragma unroll
        for (int xi = 0; xi < XB; ++xi) {
          if (x0 + xi < a.nvec) {
            double2 acc = make_double2(0.0, 0.0);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              acc.x += wv[xi][s * NVAR + 1 + k] * pv[k].x;
              acc.y += wv[xi][s * NVAR + 1 + k] * pv[k].y;
            }
            *reinterpret_cast<double2*>(a.T[s] + ((long)(x0 + xi) * t_rows + g) * a.ldT[s] + v) = acc;   // the staged value past an odd nv is 0
          }
        }
      }
    }
  }
}

// per-point kernel tables (once per solve)
// UKS: wf[g][t*nvar+d][s*nvar+c] = w[g] * fxc[s,c,t,d,g]
__global__ void build_wf_uks_kernel(double* __restrict__ wf, const double* __restrict__ fxc, const double* __restrict__ w, long ng,
                                    int nvar) {
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  const int nr = 2 * nvar;
  for (int td = 0; td < nr; ++td)
    for (int sc = 0; sc < nr; ++sc) wf[g * nr * nr + td * nr + sc] = w[g] * fxc[((long)sc * nr + td) * ng + g];
}
// MCOL: wf[g][a][b] = 2 w[g] fxc[b,a,g]
__global__ void build_wf_mcol_kernel(double* __restrict__ wf, const double* __restrict__ fxc, const double* __restrict__ w, long ng,
                                     int nvar) {
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  for (int a = 0; a < nvar; ++a)
    for (int b = 0; b < nvar; ++b) wf[g * nvar * nvar + a * nvar + b] = 2.0 * w[g] * fxc[((long)b * nvar + a) * ng + g];
}

// ------------------------------------------------------------------------------------------------------
// Grid kernel weighting of a SYMMETRIC MO-block density (xtd_block_response), UKS kernel tables, both channels:
//   Wo[c][g,i] = sum_p phi_c[g,p] D[p,i]  (p over the channel's occupied and virtual positions),  Wv[c][g,a] likewise
//   rho_0 = sum_i phi_0 Wo_0 + sum_a phiv_0 Wv_0      rho_k = 2 (sum_i phi_k Wo_0 + sum_a phiv_k Wv_0)
//   tau   = 1/2 sum_k (sum_i phi_k Wo_k + sum_a phiv_k Wv_k)                              (TAU: Wo_k, Wv_k of k = 1..3 given)
//   wv = f_xc . rho,   Bo_0 = wv_0 phi_0 + sum_k wv_k phi_k,   Bo_k = wv_k phi_0 + 1/2 wv_tau phi_k   (written over Wo)
// so that the response blocks are  V_oo = sum_c Bo_c^T phi_c  and  V_ov = sum_c Bo_c^T phiv_c.  One warp per grid point.
// ------------------------------------------------------------------------------------------------------
struct XcBlockArgs {
  int gb;
  long g0;
  double* Wo[2];           // [nvar][gb][ldWo]
  const double* Wv[2];     // [nvar][gb][ldWv]
  long ldWo[2], ldWv[2];
  const double* phi[2];    // [nvar][ng][ldphi]
  const double* phiv[2];
  long ldphi[2], ldphiv[2], phi_comp[2], phiv_comp[2];
  int no[2], nv[2];
  const double* wf;        // UKS [ng][(2 nk)^2], weighted
};

template <int NVAR, bool TAU>
__global__ void __launch_bounds__(256) xc_block_weight_kernel(const XcBlockArgs a) {
  static_assert(!TAU || NVAR == 4, "the tau component needs value + gradient AO components");
  const int lane = threadIdx.x & 31;
  const long g = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (g >= a.gb) return;
  constexpr int NK = TAU ? 5 : NVAR;
  constexpr int NR = 2 * NK;
  double fk[NR];
  const double* row = a.wf + (a.g0 + g) * (long)(NR * NR);
#pragma unroll
  for (int q = 0; q < NR; ++q) fk[q] = (lane < NR) ? row[lane * NR + q] : 0.0;
  double rho[NR];
#pragma unroll
  for (int q = 0; q < NR; ++q) rho[q] = 0.0;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const long wcmp_o = (long)a.gb * a.ldWo[s], wcmp_v = (long)a.gb * a.ldWv[s];
    for (int side = 0; side < 2; ++side) {
      const int n = side ? a.nv[s] : a.no[s];
      const double* p = side ? a.phiv[s] + (a.g0 + g) * a.ldphiv[s] : a.phi[s] + (a.g0 + g) * a.ldphi[s];
      const long pc = side ? a.phiv_comp[s] : a.phi_comp[s];
      const double* w = side ? a.Wv[s] + g * a.ldWv[s] : a.Wo[s] + g * a.ldWo[s];
      const long wc = side ? wcmp_v : wcmp_o;
      for (int o = lane; o < n; o += 32) {
        const double w0 = w[o];
        rho[s * NK] += p[o] * w0;
#pragma unroll
        for (int k = 1; k < NVAR; ++k) {
          const double pk = p[k * pc + o];
          rho[s * NK + k] += 2.0 * pk * w0;
          if (TAU) rho[s * NK + 4] += 0.5 * pk * w[k * wc + o];
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < NR; ++q) rho[q] = warp_sum(rho[q]);
  double mine = 0.0;
#pragma unroll
  for (int q = 0; q < NR; ++q) mine += fk[q] * rho[q];      // wv[t,d] = sum_{s,c} wf[g][t,d][s,c] rho[s,c]
  double wv[NR];
#pragma unroll
  for (int q = 0; q < NR; ++q) wv[q] = __shfl_sync(0xffffffffu, mine, q);
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    double* w = a.Wo[s] + g * a.ldWo[s];
    const long wc = (long)a.gb * a.ldWo[s];
    const double* p = a.phi[s] + (a.g0 + g) * a.ldphi[s];
    for (int o = lane; o < a.no[s]; o += 32) {
      const double p0 = p[o];
      double b0 = wv[s * NK] * p0;
#pragma unroll
      for (int k = 1; k < NVAR; ++k) {
        const double pk = p[k * a.phi_comp[s] + o];
        b0 += wv[s * NK + k] * pk;
        w[k * wc + o] = wv[s * NK + k] * p0 + (TAU ? 0.5 * wv[s * NK + 4] * pk : 0.0);
      }
      w[o] = b0;
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// density-fitted Coulomb blocks
// ------------------------------------------------------------------------------------------------------
// R[x][P] = sum_{i,a in block} L[P][i][a] * Z[x][r0+i][c0+a]        one CTA per aux function
template <int XC>
__global__ void __launch_bounds__(256) j_rho_kernel(double* __restrict__ R, long r_vec_stride, const double* __restrict__ L, long ldl,
                                                    long l_slice, const double* __restrict__ Z, long ldz, long z_vec_stride, int nr,
                                                    int nc, int nvec) {
  __shared__ double sm[8];
  const long P = blockIdx.x;
  const double* lp = L + P * l_slice;
  for (int x0 = 0; x0 < nvec; x0 += XC) {
    double acc[XC];
#pragma unroll
    for (int q = 0; q < XC; ++q) acc[q] = 0.0;
    for (long e = threadIdx.x; e < (long)nr * nc; e += blockDim.x) {
      const long i = e / nc, c = e - i * nc;
      const double l = lp[i * ldl + c];
#pragma unroll
      for (int q = 0; q < XC; ++q)
        if (x0 + q < nvec) acc[q] += l * Z[(long)(x0 + q) * z_vec_stride + i * ldz + c];
    }
#pragma unroll
    for (int q = 0; q < XC; ++q) {
      const double t = block_sum<256>(acc[q], sm);
      if (threadIdx.x == 0 && x0 + q < nvec) R[(long)(x0 + q) * r_vec_stride + P] = t;
    }
  }
}

// Rm[x][t][P] = sum_s mix[t][s] R[x][s][P]
__global__ void j_mix_kernel(double* __restrict__ Rm, const double* __restrict__ R, const double* __restrict__ mix, int njb, long naux,
                             long ldr, int nvec) {
  const long P = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (P >= naux || x >= nvec) return;
  for (int t = 0; t < njb; ++t) {
    double acc = 0.0;
    for (int s = 0; s < njb; ++s) acc += mix[t * njb + s] * R[((long)x * njb + s) * ldr + P];
    Rm[((long)x * njb + t) * ldr + P] = acc;
  }
}

// rho[P] = sum_r w[r] R[r][P]   (the per-block densities of xtd_block_response -> one fitted density)
struct RhoWeights {
  double w[6];
};
__global__ void rho_combine_kernel(double* __restrict__ rho, const double* __restrict__ R, long ldr, int nrows, long n, const RhoWeights w) {
  const long P = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= n) return;
  double acc = 0.0;
  for (int r = 0; r < nrows; ++r) acc += w.w[r] * R[r * ldr + P];
  rho[P] = acc;
}

// S[x][r0+i][c0+a] += sum_P Rm[x][P] * L[P][i][a]      each thread owns one block element, XC vectors at a time
template <int XC>
__global__ void __launch_bounds__(256) j_apply_kernel(double* __restrict__ S, long lds, long s_vec_stride, const double* __restrict__ L,
                                                      long ldl, long l_slice, const double* __restrict__ Rm, long r_vec_stride, long naux,
                                                      int nr, int nc, int nvec) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int x0 = blockIdx.y * XC;
  if (e >= (long)nr * nc) return;
  const long i = e / nc, c = e - i * nc;
  double acc[XC];
#pragma unroll
  for (int q = 0; q < XC; ++q) acc[q] = 0.0;
  const double* lp = L + i * ldl + c;
  for (long P = 0; P < naux; ++P) {
    const double l = lp[P * l_slice];
#pragma unroll
    for (int q = 0; q < XC; ++q)
      if (x0 + q < nvec) acc[q] += l * Rm[(long)(x0 + q) * r_vec_stride + P];
  }
#pragma unroll
  for (int q = 0; q < XC; ++q)
    if (x0 + q < nvec) S[(long)(x0 + q) * s_vec_stride + i * lds + c] += acc[q];
}

// out[i][a] = sum_P L[P][i][a]^2   (Coulomb diagonals (ia|ia) for the XSF preconditioner)
__global__ void jblock_diag_kernel(double* __restrict__ out, const double* __restrict__ L, long ldl, long l_slice, long naux, int nr,
                                   int nc, int accumulate) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)nr * nc) return;
  const long i = e / nc, c = e - i * nc;
  double acc = 0.0;
  for (long P = 0; P < naux; ++P) {
    const double l = L[P * l_slice + i * ldl + c];
    acc += l * l;
  }
  out[e] = acc + (accumulate ? out[e] : 0.0);
}

// ------------------------------------------------------------------------------------------------------
// local terms
// ------------------------------------------------------------------------------------------------------
// d[x] = <V, Zsrc[x]>   over a dense [no][nv] block (ld shared)
__global__ void __launch_bounds__(256) block_dot_kernel(double* __restrict__ d, const double* __restrict__ V, const double* __restrict__ Z,
                                                        long ld, long z_vec_stride, int no, int nv) {
  __shared__ double sm[8];
  const int x = blockIdx.x;
  double acc = 0.0;
  for (long e = threadIdx.x; e < (long)no * nv; e += blockDim.x) {
    const long i = e / nv, a = e - i * nv;
    acc += V[i * ld + a] * Z[(long)x * z_vec_stride + i * ld + a];
  }
  const double t = block_sum<256>(acc, sm);
  if (threadIdx.x == 0) d[x] = t;
}
// S[x] += d[x] * U
__global__ void block_axpy_kernel(double* __restrict__ S, const double* __restrict__ U, const double* __restrict__ d, long ld,
                                  long s_vec_stride, int no, int nv) {
  const int x = blockIdx.y;
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)no * nv) return;
  const long i = e / nv, a = e - i * nv;
  S[(long)x * s_vec_stride + i * ld + a] += d[x] * U[i * ld + a];
}
// S[x] += D o Z[x]
__global__ void block_diag_kernel(double* __restrict__ S, const double* __restrict__ D, const double* __restrict__ Z, long ld,
                                  long vec_stride, int no, int nv) {
  const int x = blockIdx.y;
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)no * nv) return;
  const long i = e / nv, a = e - i * nv;
  const long o = (long)x * vec_stride + i * ld + a;
  S[o] += D[i * ld + a] * Z[o];
}

// All local GEMM terms and diagonal terms of a SMALL problem in ONE launch (launch-bound molecules: a dozen tiny GEMM launches
// otherwise).  One thread per destination element (channel, vector, i, a): it walks the term list and adds every contribution
// that covers its element -- deterministic, no atomics.
struct LocalTermDev {
  int side, dch, r0, nr, c0, nc, sch, sr0, sc0, k;   // k: contraction length
  long ldm;
  double alpha;
  const double* M;
};
struct LocalSmallArgs {
  const LocalTermDev* terms;
  int nterms;
  const LocalTermDev* diags;   // diagonal terms reuse the record: dch = channel, M = D[no][ld]
  int ndiags;
  double* sig;
  const double* z[2];
  long sig_base[2], ldz[2], vec_stride[2];
  int no[2], nv[2];
};
__global__ void local_small_kernel(const LocalSmallArgs a) {
  const int ch = blockIdx.z, x = blockIdx.y;
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long)a.no[ch] * a.nv[ch]) return;
  const int i = (int)(e / a.nv[ch]), c = (int)(e - (long)i * a.nv[ch]);
  double acc = 0.0;
  for (int t = 0; t < a.nterms; ++t) {
    const LocalTermDev& l = a.terms[t];
    if (l.dch != ch || i < l.r0 || i >= l.r0 + l.nr || c < l.c0 || c >= l.c0 + l.nc) continue;
    const double* src = a.z[l.sch] + (long)x * a.vec_stride[l.sch];
    const long lds = a.ldz[l.sch];
    double v = 0.0;
    if (l.side == 0) {        // RIGHT: dst[r][c] += alpha sum_b src[sr0 + r][sc0 + b] M[b][c]
      const double* sr = src + (long)(l.sr0 + i - l.r0) * lds + l.sc0;
      const double* m = l.M + (c - l.c0);
      for (int b = 0; b < l.k; ++b) v = fma(sr[b], m[(long)b * l.ldm], v);
    } else if (l.side == 1) { // LEFT: dst[r][c] += alpha sum_j M[r][j] src[sr0 + j][sc0 + c]
      const double* m = l.M + (long)(i - l.r0) * l.ldm;
      const double* sc = src + (long)l.sr0 * lds + l.sc0 + (c - l.c0);
      for (int j = 0; j < l.k; ++j) v = fma(m[j], sc[(long)j * lds], v);
    } else if (l.side == 2) { // LEFT_T: dst[r][c] += alpha sum_k M[r][k] src[sr0 + c][sc0 + k]
      const double* m = l.M + (long)(i - l.r0) * l.ldm;
      const double* sr = src + (long)(l.sr0 + c - l.c0) * lds + l.sc0;
      for (int k = 0; k < l.k; ++k) v = fma(m[k], sr[k], v);
    } else {                  // RIGHT_T: dst[r][c] += alpha sum_j src[sr0 + j][sc0 + r] M[j][c]
      const double* sc = src + (long)l.sr0 * lds + l.sc0 + (i - l.r0);
      const double* m = l.M + (c - l.c0);
      for (int j = 0; j < l.k; ++j) v = fma(sc[(long)j * lds], m[(long)j * l.ldm], v);
    }
    acc = fma(l.alpha, v, acc);
  }
  const long o = (long)x * a.vec_stride[ch] + (long)i * a.ldz[ch] + c;
  for (int t = 0; t < a.ndiags; ++t)
    if (a.diags[t].dch == ch) acc = fma(a.diags[t].M[(long)i * a.ldz[ch] + c], a.z[ch][o], acc);
  a.sig[a.sig_base[ch] + o] += acc;
}

// ------------------------------------------------------------------------------------------------------
// Davidson vector primitives (subspace orthogonalisation, projected matrix, Ritz vectors, residuals)
// ------------------------------------------------------------------------------------------------------
// G[i][j] = <A_i, B_j>    one CTA per (i, j) pair
__global__ void __launch_bounds__(512) vec_dots_kernel(double* __restrict__ G, int ldg, const double* __restrict__ A, long lda,
                                                       const double* __restrict__ B, long ldb, long n) {
  __shared__ double sm[16];
  const double* a = A + (long)blockIdx.y * lda;
  const double* b = B + (long)blockIdx.x * ldb;
  double acc0 = 0.0, acc1 = 0.0;
  long e = threadIdx.x;
  for (; e + 512 < n; e += 1024) {
    acc0 += a[e] * b[e];
    acc1 += a[e + 512] * b[e + 512];
  }
  for (; e < n; e += 512) acc0 += a[e] * b[e];
  const double t = block_sum<512>(acc0 + acc1, sm);
  if (threadIdx.x == 0) G[blockIdx.y * ldg + blockIdx.x] = t;
}

// Y[i] = beta*Y[i] + sum_j C[i][j] X[j]   (m outputs, k inputs)
template <int MB>
__global__ void __launch_bounds__(256) vec_lincomb_kernel(double* __restrict__ Y, long ldy, const double* __restrict__ X, long ldx,
                                                          const double* __restrict__ C, int ldc, int m, int k, long n, double beta) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int i0 = blockIdx.y * MB;
  if (e >= n) return;
  double acc[MB];
#pragma unroll
  for (int q = 0; q < MB; ++q) acc[q] = 0.0;
  for (int j = 0; j < k; ++j) {
    const double xv = X[(long)j * ldx + e];
#pragma unroll
    for (int q = 0; q < MB; ++q)
      if (i0 + q < m) acc[q] += C[(i0 + q) * ldc + j] * xv;
  }
#pragma unroll
  for (int q = 0; q < MB; ++q)
    if (i0 + q < m) {
      double* y = Y + (long)(i0 + q) * ldy + e;
      *y = (beta != 0.0 ? beta * *y : 0.0) + acc[q];
    }
}

// r[k] = ax[k] - e[k]*x[k];  nrm2[k] = |r[k]|^2
__global__ void __launch_bounds__(512) vec_residual_kernel(double* __restrict__ R, const double* __restrict__ AX, const double* __restrict__ X,
                                                           long ld, const double* __restrict__ e, double* __restrict__ nrm2, long n) {
  __shared__ double sm[16];
  const int k = blockIdx.x;
  const double ek = e[k];
  double acc = 0.0;
  for (long i = threadIdx.x; i < n; i += 512) {
    const double r = AX[(long)k * ld + i] - ek * X[(long)k * ld + i];
    R[(long)k * ld + i] = r;
    acc += r * r;
  }
  const double t = block_sum<512>(acc, sm);
  if (threadIdx.x == 0) nrm2[k] = t;
}

// x[k] = x[k] / clamp(hdiag - shift[k]);  nrm2[k] = |x[k]|^2   (diagonal preconditioner, make_diag_precond)
__global__ void __launch_bounds__(512) vec_precond_kernel(double* __restrict__ X, long ld, const double* __restrict__ hdiag,
                                                          const double* __restrict__ shift, double* __restrict__ nrm2, long n) {
  __shared__ double sm[16];
  const int k = blockIdx.x;
  const double sh = shift[k];
  double acc = 0.0;
  for (long i = threadIdx.x; i < n; i += 512) {
    double d = hdiag[i] - sh;
    if (fabs(d) < 1e-8) d = 1e-8;
    const double v = X[(long)k * ld + i] / d;
    X[(long)k * ld + i] = v;
    acc += v * v;
  }
  const double t = block_sum<512>(acc, sm);
  if (threadIdx.x == 0) nrm2[k] = t;
}

// x[k] *= s[k]
__global__ void vec_scale_kernel(double* __restrict__ X, long ld, const double* __restrict__ s, long n) {
  const int k = blockIdx.y;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) X[(long)k * ld + i] *= s[k];
}

}  // namespace xtd
