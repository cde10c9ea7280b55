// FP64 contraction emulated on the INT8 tensor cores of sm_100a (Ozaki splitting):
//
//   C[m][n] (+)= alpha * sum_q sum_k A[q][m][k] * B[q][n][k]                      (fp64 in, fp64 out)
//
// tcgen05 has no f64 kind, and the warp-level DMMA pipe tops out at 37 TFLOP/s.  Here every fp64 operand row is scaled by a
// power of two per (row, group of `group` q-slices) and cut into S balanced radix-256 digits (signed 8-bit planes):
//   x = scale * sum_l d_l 2^(-8 l),  d_0 in [-64, 64],  d_l in [-128, 127] (l >= 1)                 -> 8 S - 2 bits below the row scale
// (floor digits first, then a carry pass from the least significant digit turns [0, 255] into [-128, 127]: balanced digits keep
// the dropped products zero-mean, so their sum over a long contraction grows like sqrt(K), not K), so that
//   A.B = sa sb sum_{i+j < S} 2^(-8(i+j)) (A_i . B_j)   with every A_i . B_j an EXACT int8 x int8 -> int32 product on
// `tcgen05.mma.kind::i8`; the S(S+1)/2 plane products are accumulated per level l = i + j in S separate TMEM accumulators
// (128 lanes x 64 columns each, S <= 8 fills the 512 columns) over one group, then read back with tcgen05.ld, recombined in
// fp64 (Horner in 2^-8), scaled and added to fp64 register accumulators.  Terms with i + j >= S (below 2^(-8S) of the row
// scale) are dropped.  int32 never overflows: |d_i d_j| <= 2^14, at most S products per level and k, `group` bounded accordingly.
//
// Sliced operands live in HBM pre-tiled as shared-memory images, so a pipeline stage is two plain bulk copies
// (cp.async.bulk, no tensor map), in the canonical no-swizzle K-major UMMA layout (core matrix 8 rows x 16 B, SBO 128 B):
//   A  [q][row tile][k block of 32][plane][2 chunks][128 rows][16 B]          one descriptor per plane, LBO 2 KB
//   B  [q][row tile][k block of 32][2 chunks][plane][ 64 rows][16 B]          planes stacked along N, LBO S KB
// With the planes of B stacked along N, ONE instruction multiplies plane A_i with planes B_0 .. B_{S-1-i} (N = 64 (S - i),
// in pieces of <= 256) and lands in the contiguous TMEM columns of levels i .. S-1: 8 (S = 6) instead of 21 MMAs per k-step,
// and A_i is read from shared memory once or twice instead of S - i times (an N = 64 instruction re-reads 4 KB of A for 2 KB
// of B: 192 B/clk of shared-memory reads against the 128 B/clk the SM has).
//
// Warp roles in a CTA of 192 threads: warp 0 bulk-copy producer, warp 1 MMA issuer (+ TMEM allocation), warps 2-5 epilogue
// (TMEM lane quadrant = warp % 4).  One CTA per (128 x 64 output tile, split of the group range); partial tiles go to a
// workspace and are reduced deterministically.
#pragma once
#include "common.cuh"

namespace xtd {

constexpr int OZ_BM = 128, OZ_BN = 64, OZ_KB = 32, OZ_STAGES = 4, OZ_MAX_S = 8, OZ_MIN_S = 3;
constexpr int OZ_THREADS = 192;
constexpr int OZ_K1_THREADS = 320;     // producer + MMA issuer + 8 epilogue warps

__device__ __forceinline__ uint32_t oz_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- packed rows ----------------------------------------------------------------------------------------------------------
// The A operand of the fused half-transform packs the rows (P, i) of G aux functions into one q-slice, so a 128-row tile spans aux
// functions instead of padding every aux function's `no` rows to a multiple of 128.  Rows are ordered (occupied row block, P, i)
// with the row blocks [0, o2) and [o2, no), so a pass over one row block of a block-weighted term reads a contiguous row range:
//   r < G o2:  P = r / o2,  i = r % o2;     else  r' = r - G o2,  P = r' / (no - o2),  i = o2 + r' % (no - o2)     (r' < G (no - o2))
__host__ __device__ __forceinline__ bool oz_unpack_row(int r, int G, int o2, int no, int& P, int& i) {
  if (r < G * o2) {
    P = r / o2;
    i = r - P * o2;
    return true;
  }
  const int n1 = no - o2, r1 = r - G * o2;
  if (r1 >= G * n1) return false;
  P = r1 / n1;
  i = o2 + (r1 - P * n1);
  return true;
}
// first and one-past-last packed row of a pass over the orbitals [i_lo, i_hi) (exact when the range is a row block or all rows)
inline int oz_packed_row_lo(int i_lo, int G, int o2) { return i_lo >= o2 ? G * o2 : 0; }
inline int oz_packed_row_hi(int i_hi, int G, int o2, int no) { return i_hi <= o2 ? G * o2 : G * no; }

// Source of a packed-row slicing (OzRowPack::G > 0): row r of q-slice q is aux function q G + P (valid while < np), orbital i, at
// X[q * sq + P * sp + i * ld].  G = 0: plain rows.
struct OzRowPack {
  int G = 0, o2 = 0, no = 0, np = 0;
  long sp = 0;
};
// offset of row `row` of q-slice q relative to X + q * sq, or -1 for a row with no source (zero)
__device__ __forceinline__ long oz_src_row(const OzRowPack& pk, int q, int row, int rows, long ld) {
  if (pk.G == 0) return row < rows ? (long)row * ld : -1L;
  int P, i;
  if (!oz_unpack_row(row, pk.G, pk.o2, pk.no, P, i) || q * pk.G + P >= pk.np) return -1L;
  return (long)P * pk.sp + (long)i * ld;
}

// ---- slicing ------------------------------------------------------------------------------------------------------------
// Source element (q, row, k):  X[q * sq + row * ld + k]   (K-contiguous rows; X[q * sq + oz_src_row(..) + k] with packed rows),
// or for a TRANSPOSED source (the contraction index is the row index of the array, e.g. grid points)  X[q * sq + k * ld + row].
// Only k with q * K + k < k_valid are read (a ragged last q-slice); everything else is zero.
__device__ __forceinline__ double oz_scale_of(double m) {
  if (!(m > 1e-280 && m < 1e280)) return 0.0;
  int e;
  frexp(m, &e);                 // m = f 2^e, f in [0.5, 1)
  return ldexp(1.0, e - 6);
}

// transposed source: block (32 rows, 32 k-lanes); grid (rows_pad / 32, ngroups)
__global__ void oz_rowmax_t_kernel(double* __restrict__ scale, int rows_pad, const double* __restrict__ X, long ld, long sq, int rows, int K,
                                   int nq, int group, long k_valid) {
  const int row = blockIdx.x * 32 + threadIdx.x, g = blockIdx.y;
  double m = 0.0;
  if (row < rows) {
    const int q1 = min(nq, (g + 1) * group);
    for (int q = g * group; q < q1; ++q) {
      const long kmax = min((long)K, k_valid - (long)q * K);
      const double* x = X + (long)q * sq + row;
      for (long k = threadIdx.y; k < kmax; k += 32) m = fmax(m, fabs(x[k * ld]));
    }
  }
  __shared__ double red[32][33];
  red[threadIdx.y][threadIdx.x] = m;
  __syncthreads();
  if (threadIdx.y == 0) {
    for (int w = 1; w < 32; ++w) m = fmax(m, red[w][threadIdx.x]);
    if (row < rows_pad) scale[(long)g * rows_pad + row] = oz_scale_of(m);
  }
}

// scale[g][row] = 2^(e - 6) with max |x| over the row's group < 2^e (0 for an all-zero / padding row)
__global__ void oz_rowmax_kernel(double* __restrict__ scale, int rows_pad, const double* __restrict__ X, long ld, long sq, int rows, int K,
                                 int nq, int group, long k_valid, const OzRowPack pack) {
  const int row = blockIdx.x, g = blockIdx.y;
  double m = 0.0;
  const int q1 = min(nq, (g + 1) * group);
  for (int q = g * group; q < q1; ++q) {
    const long off = oz_src_row(pack, q, row, rows, ld);
    if (off < 0) continue;
    const int kmax = (int)min((long)K, k_valid - (long)q * K);
    const double* x = X + (long)q * sq + off;
    for (int k = threadIdx.x; k < kmax; k += blockDim.x) m = fmax(m, fabs(x[k]));
  }
  __shared__ double red[8];
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, red[w]);
    scale[(long)g * rows_pad + row] = oz_scale_of(m);
  }
}

// one thread: 16 consecutive k of one row -> S 16-byte chunks.  grid (2 nkb, rows_pad / 128, nq), block 128 (lane <-> row)
// 16 consecutive elements t[k] (already divided by the row scale: |t| < 64) -> S balanced radix-256 digit planes, packed as the
// 16-byte row chunk of every plane: x = sum_l d_l 2^(-8l), d_0 in [-64, 64], d_l in [-128, 127].
// S <= 6: in integer arithmetic.  q = floor(t 2^(8(S-1))) lands in the low mantissa bits of RD(t 2^(8(S-1)) + 1.5 2^52) (one FMA;
// |q| < 2^46), and adding 128 at every lower byte position turns the bytes of q into the balanced digits,
//   q + B = d_0 2^(8(S-1)) + sum_{l>=1} (d_l + 128) 2^(8(S-1-l)),
// the same digits as floor-then-carry (the representation is unique); (d_l + 128) ^ 0x80 is the int8 pattern of d_l.  One FMA, one
// 64-bit add and a few byte permutes per element instead of three fp64 operations and a carry step per digit (the fused
// half-transform's epilogue was bound by exactly that arithmetic: two warps per scheduler, ~85 dependent instructions per element).
// S = 7, 8 (q would not fit 51 bits): digit by digit, MSB first with round-down, then the carry pass.
template <int S>
__device__ __forceinline__ void oz_digits16(const double (&t)[16], uint32_t (&pk)[S][4]) {
  const double magic = 6755399441055744.0;   // 1.5 * 2^52: RD(x + magic) has floor(x) in its low mantissa bits (two's complement)
  if constexpr (S <= 6) {
    constexpr double SCL = (double)(1ull << (8 * (S - 1)));
    constexpr unsigned long long BAL = 128ull * (((1ull << (8 * (S - 1))) - 1ull) / 255ull);
    constexpr unsigned long long CADD = BAL - 0x4338000000000000ull;      // minus the bit pattern of 1.5 * 2^52
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      uint32_t lo[4], hi[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned long long q = (unsigned long long)__double_as_longlong(__fma_rd(t[4 * w + j], SCL, magic)) + CADD;
        lo[j] = (uint32_t)q;
        hi[j] = (uint32_t)(q >> 32);
      }
#pragma unroll
      for (int pos = 0; pos < S; ++pos) {                 // byte position from the least significant digit
        const uint32_t* src = pos < 4 ? lo : hi;
        const uint32_t sel = (uint32_t)(pos & 3) | ((uint32_t)(4 + (pos & 3)) << 4);
        const uint32_t t01 = __byte_perm(src[0], src[1], sel), t23 = __byte_perm(src[2], src[3], sel);
        pk[S - 1 - pos][w] = __byte_perm(t01, t23, 0x5410) ^ (pos < S - 1 ? 0x80808080u : 0u);
      }
    }
  } else {
#pragma unroll
    for (int sl = 0; sl < S; ++sl)
#pragma unroll
      for (int w = 0; w < 4; ++w) pk[sl][w] = 0u;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      double tt = t[k];
      int dg[S];
#pragma unroll
      for (int sl = 0; sl < S; ++sl) {
        const double u = (sl == 0) ? __dadd_rd(tt, magic) : __fma_rd(tt, 256.0, magic);      // floor: the remainder stays in [0, 1)
        const double qd = u - magic;
        tt = (sl == 0) ? (tt - qd) : fma(tt, 256.0, -qd);
        dg[sl] = __double2loint(u);             // floor(t) in [-64, 63], then digits in [0, 255]
      }
      int carry = 0;                            // balance: [0, 255] -> [-128, 127] with a carry into the next higher digit
#pragma unroll
      for (int sl = S - 1; sl >= 1; --sl) {
        const int vv = dg[sl] + carry;
        carry = vv >= 128 ? 1 : 0;
        dg[sl] = vv - (carry << 8);
      }
      dg[0] += carry;
#pragma unroll
      for (int sl = 0; sl < S; ++sl) pk[sl][k >> 2] |= ((uint32_t)dg[sl] & 0xffu) << ((k & 3) * 8);
    }
  }
}

template <int S, bool TRANS>
__global__ void __launch_bounds__(128) oz_slice_kernel(int8_t* __restrict__ out, const double* __restrict__ scale, int rows_pad,
                                                       const double* __restrict__ X, long ld, long sq, int rows, int K, int RT, int nkb,
                                                       int group, int stacked, long k_valid, const OzRowPack pack) {
  const int c2 = blockIdx.x, q = blockIdx.z;
  const int row = blockIdx.y * 128 + threadIdx.x;
  const int rt = row / RT, r = row - rt * RT, nrt = rows_pad / RT;
  const int k0 = c2 * 16;
  double x[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) x[k] = 0.0;
  double sc = 0.0;
  const long off = TRANS ? (row < rows ? 0L : -1L) : oz_src_row(pack, q, row, rows, ld);
  if (off >= 0) {
    sc = scale[(long)(q / group) * rows_pad + row];
    const int kmax = (int)min((long)K, k_valid - (long)q * K);      // valid k of this q-slice
    if (TRANS) {
      const double* src = X + (long)q * sq + (long)k0 * ld + row;    // lanes = consecutive rows: coalesced for every k
#pragma unroll
      for (int k = 0; k < 16; ++k)
        if (k0 + k < kmax) x[k] = src[(long)k * ld];
    } else {
      const double* src = X + (long)q * sq + off + k0;
      if (k0 + 16 <= kmax) {
#pragma unroll
        for (int k = 0; k < 16; k += 2) {
          const double2 v = *reinterpret_cast<const double2*>(src + k);
          x[k] = v.x;
          x[k + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 16; ++k)
          if (k0 + k < kmax) x[k] = src[k];
      }
    }
  }
  // 1 / scale for a power of two: flip the exponent
  const double inv = sc > 0.0 ? __hiloint2double(0x7fe00000 - __double2hiint(sc), 0) : 0.0;
  uint32_t pk[S][4];
#pragma unroll
  for (int k = 0; k < 16; ++k) x[k] *= inv;   // |t| < 64
  oz_digits16<S>(x, pk);
  // plane-major image (A): [plane][chunk][row]; stacked image (B): [chunk][plane][row]
  int8_t* dst = out + ((((long)q * nrt + rt) * nkb + (c2 >> 1)) * S) * ((long)RT * OZ_KB) + (long)r * 16 +
                (stacked ? (long)(c2 & 1) * S * RT * 16 : (long)(c2 & 1) * RT * 16);
  const long plane = stacked ? (long)RT * 16 : (long)RT * OZ_KB;
#pragma unroll
  for (int sl = 0; sl < S; ++sl) *reinterpret_cast<uint4*>(dst + sl * plane) = make_uint4(pk[sl][0], pk[sl][1], pk[sl][2], pk[sl][3]);
}

// The fp64 values a stacked (B operand, 64-row tile) image stands for: out[p][row][k] = scale[(q0 + p) / group][row] *
// sum_l d_l 2^(-8 l) of q-slice q0 + p -- exactly what the INT8 contraction multiplies.  One thread per element.
__global__ void oz_unslice_b_kernel(double* __restrict__ out, long ld, long sp, const int8_t* __restrict__ img, const double* __restrict__ scale,
                                    int S, int rows, int rows_pad, int K, int nkb, int group, long q0, int np) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long p = blockIdx.y;
  if (e >= (long)rows * K || p >= np) return;
  const int row = (int)(e / K), k = (int)(e - (long)row * K);
  const long q = q0 + p;
  const int nrt = rows_pad / OZ_BN, rt = row / OZ_BN, r = row - rt * OZ_BN;
  const int8_t* src = img + (((q * nrt + rt) * nkb + k / OZ_KB) * S) * ((long)OZ_BN * OZ_KB) + (long)((k % OZ_KB) / 16) * S * OZ_BN * 16 +
                      (long)r * 16 + (k % 16);
  double acc = 0.0;
  for (int l = S - 1; l >= 0; --l) acc = acc * (1.0 / 256.0) + (double)src[(long)l * OZ_BN * 16];
  out[p * sp + (long)row * ld + k] = scale[(q / group) * rows_pad + row] * acc;
}

// ---- the INT8 tensor-core kernel ------------------------------------------------------------------------------------------
struct OzGemmParams {
  const int8_t* A;      // [nq][nmt][nkb][S][128 x 32]
  const int8_t* B;      // [..][nnt][nkb][2][S][64 x 16] (planes stacked along N), first slice used: b_q0
  const double* sa;     // [ngroups][Mpad]           (group index relative to this launch)
  const double* sb;     // [..][Npad], first group used: b_q0 / group
  int nmt, nnt, nkb, nq, group, b_q0;
  int Mpad, Npad, splits;
  double* W;            // partial tiles [splits][Mpad][Npad]
  double alpha;
  // independent problems in one launch (blockIdx.y): per-batch offsets of the operands (bytes), scales and output (doubles)
  int batches = 1;
  long a_bstride = 0, b_bstride = 0, sa_bstride = 0, sb_bstride = 0, w_bstride = 0;
};

__device__ __forceinline__ void oz_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(oz_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void oz_mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = oz_smem_u32(bar);
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void oz_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(oz_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void oz_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(oz_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void oz_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(oz_smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(oz_smem_u32(bar))
               : "memory");
}
// the same copy delivered to the same shared-memory offset (and signalled on the same barrier offset) of every CTA in `mask`
__device__ __forceinline__ void oz_bulk_load_mc(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
                   oz_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(oz_smem_u32(bar)), "h"(mask)
               : "memory");
}
__device__ __forceinline__ void oz_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(oz_smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ uint32_t oz_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void oz_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle: start address, leading (K-direction) and stride (row-group) byte offsets
__device__ __forceinline__ uint64_t oz_smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void oz_mma_i8(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void oz_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(oz_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void oz_tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

// CN = CTAs per cluster along N: they share the A tile (same output row tile, consecutive column tiles); each loads 1 / CN of
// every A stage and multicasts it to the whole cluster, so the L2 -> SM traffic per MMA drops from A + B to A / CN + B.
template <int S, int CN>
__global__ void __launch_bounds__(OZ_THREADS, 1) oz_gemm_kernel(const OzGemmParams p) {
  constexpr int A_SLICE = OZ_BM * OZ_KB, B_SLICE = OZ_BN * OZ_KB;
  constexpr int A_BYTES = S * A_SLICE, B_BYTES = S * B_SLICE, STAGE = A_BYTES + B_BYTES;
  extern __shared__ __align__(128) uint8_t oz_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(oz_smem + OZ_STAGES * STAGE);
  uint64_t* empty = full + OZ_STAGES;
  uint64_t* tmem_full = empty + OZ_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x;
  const long zb = blockIdx.y;
  const int nt = item % p.nnt, mt = (item / p.nnt) % p.nmt, sp = item / (p.nnt * p.nmt);
  const int ngroups = (p.nq + p.group - 1) / p.group;
  const int g0 = (int)((long)ngroups * sp / p.splits), g1 = (int)((long)ngroups * (sp + 1) / p.splits);

  const uint32_t crank = CN > 1 ? oz_cluster_rank() : 0u;
  constexpr uint16_t cmask = (uint16_t)((1u << CN) - 1u);
  if (threadIdx.x == 0) {
    for (int s = 0; s < OZ_STAGES; ++s) {
      oz_mbar_init(&full[s], 1);
      oz_mbar_init(&empty[s], CN);          // a stage is rewritten by every CTA of the cluster: all of them must have drained it
    }
    oz_mbar_init(tmem_full, 1);
    oz_mbar_init(tmem_empty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz_smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (CN > 1) oz_cluster_sync();            // every CTA's barriers exist before the first multicast copy / arrive
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== producer: two bulk copies per k-step =====================
    if (lane == 0) {
      long it = 0;
      for (int g = g0; g < g1; ++g) {
        const int q1 = min(p.nq, (g + 1) * p.group);
        for (int q = g * p.group; q < q1; ++q) {
          const int8_t* a = p.A + zb * p.a_bstride + (((long)q * p.nmt + mt) * p.nkb) * A_BYTES;
          const int8_t* b = p.B + zb * p.b_bstride + (((long)(q + p.b_q0) * p.nnt + nt) * p.nkb) * B_BYTES;
          for (int kb = 0; kb < p.nkb; ++kb, ++it) {
            const int s = (int)(it % OZ_STAGES);
            const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
            oz_mbar_wait(&empty[s], ph ^ 1u);
            oz_mbar_expect_tx(&full[s], STAGE);
            uint8_t* sa = oz_smem + s * STAGE;
            if (CN == 1) {
              oz_bulk_load(sa, a + (long)kb * A_BYTES, A_BYTES, &full[s]);
            } else {
              constexpr int PART = A_BYTES / CN;
              oz_bulk_load_mc(sa + crank * PART, a + (long)kb * A_BYTES + crank * PART, PART, &full[s], cmask);
            }
            oz_bulk_load(sa + A_BYTES, b + (long)kb * B_BYTES, B_BYTES, &full[s]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: S(S+1)/2 int8 MMAs per k-step, one accumulator per level i + j =====================
    if (lane == 0) {
      // instruction descriptor: D = s32, A = B = signed int8, both K-major, M = 128; N = 64 x (planes of B in the instruction)
      constexpr uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BM >> 4) << 24);
      const uint32_t smem_base = oz_smem_u32(oz_smem);
      long it = 0;
      for (int g = g0; g < g1; ++g) {
        if (g > g0) oz_mbar_wait(tmem_empty, (uint32_t)((g - g0 - 1) & 1));   // epilogue has drained the previous group
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q1 = min(p.nq, (g + 1) * p.group);
        const long nsteps = (long)(q1 - g * p.group) * p.nkb;
        for (long st = 0; st < nsteps; ++st, ++it) {
          const int s = (int)(it % OZ_STAGES);
          const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
          oz_mbar_wait(&full[s], ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_base = smem_base + s * STAGE, b_base = a_base + A_BYTES;
          const uint32_t later = st > 0 ? 1u : 0u;
#pragma unroll
          for (int i = 0; i < S; ++i) {
            const uint64_t da = oz_smem_desc(a_base + i * A_SLICE, OZ_BM * 16, 128);
            // planes B_0 .. B_{S-1-i} at once, in pieces of at most 256 columns: levels i .. S-1
#pragma unroll
            for (int j0 = 0; j0 < S - i; j0 += 4) {
              const int nj = (S - i - j0) < 4 ? (S - i - j0) : 4;
              const uint64_t db = oz_smem_desc(b_base + j0 * (OZ_BN * 16), S * OZ_BN * 16, 128);
              const uint32_t idesc = idesc0 | ((uint32_t)((nj * OZ_BN) >> 3) << 17);
              oz_mma_i8(tmem_base + (uint32_t)((i + j0) * OZ_BN), da, db, idesc, (i > 0) ? 1u : later);
            }
          }
          if (CN == 1) oz_commit(&empty[s]);      // frees the stage when these MMAs have read it
          else oz_commit_mc(&empty[s], cmask);    // ... in every CTA of the cluster (each of them writes a part of it)
        }
        oz_commit(tmem_full);        // all levels of this group are complete
      }
    }
  } else {
    // ===================== epilogue: levels -> fp64, scale, accumulate =====================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
    double acc[OZ_BN];
#pragma unroll
    for (int c = 0; c < OZ_BN; ++c) acc[c] = 0.0;
    for (int g = g0; g < g1; ++g) {
      oz_mbar_wait(tmem_full, (uint32_t)((g - g0) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const double sa = p.sa[zb * p.sa_bstride + (long)g * p.Mpad + mt * OZ_BM + row];
      const double* sb = p.sb + zb * p.sb_bstride + (long)(g + p.b_q0 / p.group) * p.Npad + nt * OZ_BN;
#pragma unroll
      for (int c0 = 0; c0 < OZ_BN; c0 += 16) {
        double v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = 0.0;
#pragma unroll
        for (int l = S - 1; l >= 0; --l) {
          uint32_t r[16];
          oz_tmem_ld16(taddr + (uint32_t)(l * OZ_BN + c0), r);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] = fma(v[k], 0.00390625, (double)(int)r[k]);
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[c0 + k] = fma(v[k], sa * sb[c0 + k], acc[c0 + k]);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      oz_mbar_arrive(tmem_empty);
    }
    double* w = p.W + zb * p.w_bstride + ((long)sp * p.Mpad + mt * OZ_BM + row) * p.Npad + nt * OZ_BN;
#pragma unroll
    for (int c = 0; c < OZ_BN; c += 2) *reinterpret_cast<double2*>(w + c) = make_double2(p.alpha * acc[c], p.alpha * acc[c + 1]);
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (CN > 1) oz_cluster_sync();            // no CTA leaves while a peer may still multicast into it or arrive on its barriers
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---- the same contraction as a PERSISTENT kernel ------------------------------------------------------------------------------
// One CTA per SM walks the (split, row tile, column tile, batch) items in launch order, so the barriers, the TMEM allocation and the
// pipeline fill are paid once per SM instead of once per 128 x 64 tile, and the MMAs of the next group / tile run under the fp64
// part of the epilogue: eight epilogue warps (two per TMEM lane quadrant, 32 columns each) first DRAIN the level accumulators into
// fp64 registers, hand the accumulators back, and only then scale / accumulate / store.  This is what short contractions need
// (the grid GEMMs: one accumulation group per tile; the non-persistent kernel showed the tensor pipe 63 % active there against 85 %
// for the long exchange contraction).  No cluster multicast (measured: no gain at 2 CTAs).
template <int S>
__global__ void __launch_bounds__(OZ_K1_THREADS, 1) oz_gemm_p_kernel(const OzGemmParams p) {
  constexpr int A_SLICE = OZ_BM * OZ_KB, B_SLICE = OZ_BN * OZ_KB;
  constexpr int A_BYTES = S * A_SLICE, B_BYTES = S * B_SLICE, STAGE = A_BYTES + B_BYTES;
  extern __shared__ __align__(128) uint8_t oz_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(oz_smem + OZ_STAGES * STAGE);
  uint64_t* empty = full + OZ_STAGES;
  uint64_t* tmem_full = empty + OZ_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngroups = (p.nq + p.group - 1) / p.group;
  const long per_batch = (long)p.nnt * p.nmt * p.splits;
  const long nitems = per_batch * p.batches;

  if (threadIdx.x == 0) {
    for (int s = 0; s < OZ_STAGES; ++s) {
      oz_mbar_init(&full[s], 1);
      oz_mbar_init(&empty[s], 1);
    }
    oz_mbar_init(tmem_full, 1);
    oz_mbar_init(tmem_empty, OZ_K1_THREADS - 64);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz_smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      long it = 0;
      for (long item = blockIdx.x; item < nitems; item += gridDim.x) {
        const long zb = item / per_batch;
        const int r = (int)(item - zb * per_batch);
        const int nt = r % p.nnt, mt = (r / p.nnt) % p.nmt, sp = r / (p.nnt * p.nmt);
        const int g0 = (int)((long)ngroups * sp / p.splits), g1 = (int)((long)ngroups * (sp + 1) / p.splits);
        for (int g = g0; g < g1; ++g) {
          const int q1 = min(p.nq, (g + 1) * p.group);
          for (int q = g * p.group; q < q1; ++q) {
            const int8_t* a = p.A + zb * p.a_bstride + (((long)q * p.nmt + mt) * p.nkb) * A_BYTES;
            const int8_t* b = p.B + zb * p.b_bstride + (((long)(q + p.b_q0) * p.nnt + nt) * p.nkb) * B_BYTES;
            for (int kb = 0; kb < p.nkb; ++kb, ++it) {
              const int s = (int)(it % OZ_STAGES);
              const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
              oz_mbar_wait(&empty[s], ph ^ 1u);
              oz_mbar_expect_tx(&full[s], STAGE);
              uint8_t* sa = oz_smem + s * STAGE;
              oz_bulk_load(sa, a + (long)kb * A_BYTES, A_BYTES, &full[s]);
              oz_bulk_load(sa + A_BYTES, b + (long)kb * B_BYTES, B_BYTES, &full[s]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BM >> 4) << 24);
      const uint32_t smem_base = oz_smem_u32(oz_smem);
      long it = 0, n = 0;
      for (long item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int r = (int)(item % per_batch);
        const int sp = r / (p.nnt * p.nmt);
        const int g0 = (int)((long)ngroups * sp / p.splits), g1 = (int)((long)ngroups * (sp + 1) / p.splits);
        for (int g = g0; g < g1; ++g, ++n) {
          if (n > 0) oz_mbar_wait(tmem_empty, (uint32_t)((n - 1) & 1));      // the epilogue has drained the previous group / tile
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const int q1 = min(p.nq, (g + 1) * p.group);
          const long nsteps = (long)(q1 - g * p.group) * p.nkb;
          for (long st = 0; st < nsteps; ++st, ++it) {
            const int s = (int)(it % OZ_STAGES);
            const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
            oz_mbar_wait(&full[s], ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_base = smem_base + s * STAGE, b_base = a_base + A_BYTES;
            const uint32_t later = st > 0 ? 1u : 0u;
#pragma unroll
            for (int i = 0; i < S; ++i) {
              const uint64_t da = oz_smem_desc(a_base + i * A_SLICE, OZ_BM * 16, 128);
#pragma unroll
              for (int j0 = 0; j0 < S - i; j0 += 4) {
                const int nj = (S - i - j0) < 4 ? (S - i - j0) : 4;
                const uint64_t db = oz_smem_desc(b_base + j0 * (OZ_BN * 16), S * OZ_BN * 16, 128);
                const uint32_t idesc = idesc0 | ((uint32_t)((nj * OZ_BN) >> 3) << 17);
                oz_mma_i8(tmem_base + (uint32_t)((i + j0) * OZ_BN), da, db, idesc, (i > 0) ? 1u : later);
              }
            }
            oz_commit(&empty[s]);
          }
          oz_commit(tmem_full);
        }
      }
    }
  } else {
    const int quad = warp & 3, half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
    constexpr int HC = OZ_BN / 2;
    long n = 0;
    for (long item = blockIdx.x; item < nitems; item += gridDim.x) {
      const long zb = item / per_batch;
      const int r = (int)(item - zb * per_batch);
      const int nt = r % p.nnt, mt = (r / p.nnt) % p.nmt, sp = r / (p.nnt * p.nmt);
      const int g0 = (int)((long)ngroups * sp / p.splits), g1 = (int)((long)ngroups * (sp + 1) / p.splits);
      double acc[HC];
#pragma unroll
      for (int c = 0; c < HC; ++c) acc[c] = 0.0;
      for (int g = g0; g < g1; ++g, ++n) {
        const double sa = p.sa[zb * p.sa_bstride + (long)g * p.Mpad + mt * OZ_BM + row];
        const double* sb = p.sb + zb * p.sb_bstride + (long)(g + p.b_q0 / p.group) * p.Npad + nt * OZ_BN + half * HC;
        oz_mbar_wait(tmem_full, (uint32_t)(n & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        double v[HC];
#pragma unroll
        for (int k = 0; k < HC; ++k) v[k] = 0.0;
#pragma unroll
        for (int l = S - 1; l >= 0; --l) {
          uint32_t rr[HC];
#pragma unroll
          for (int cc = 0; cc < HC; cc += 16) oz_tmem_ld16(taddr + (uint32_t)(l * OZ_BN + half * HC + cc), rr + cc);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int k = 0; k < HC; ++k)     // int32 -> fp64 through the 2^52 + 2^31 offset (no conversion instruction)
            v[k] = fma(v[k], 0.00390625, __hiloint2double(0x43300000, (int)(rr[k] ^ 0x80000000u)) - 4503601774854144.0);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        oz_mbar_arrive(tmem_empty);                  // accumulators handed back: the next group's MMAs run under the lines below
#pragma unroll
        for (int k = 0; k < HC; ++k) acc[k] = fma(v[k], sa * sb[k], acc[k]);
      }
      double* w = p.W + zb * p.w_bstride + ((long)sp * p.Mpad + mt * OZ_BM + row) * p.Npad + nt * OZ_BN + half * HC;
#pragma unroll
      for (int c = 0; c < HC; c += 2) *reinterpret_cast<double2*>(w + c) = make_double2(p.alpha * acc[c], p.alpha * acc[c + 1]);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---- fused half-transform: U = Loo . z on the INT8 tensor cores, written directly as the A planes of the contraction above ----
//
//   U[P][(x,i)][b] = sum_j Loo[P][i][j] zt[x][b][j]            (K = occupied count: a few k-steps per tile)
//
// A = int8 planes of Loo (static; one q-slice per group of `group` aux functions, whose rows (P, i) are packed as oz_unpack_row
// describes and padded to 128 per group), B = planes of zt (per call, one q-slice per trial vector).  A persistent CTA walks tiles
// (group, 128 packed rows, x, 64 columns b); its epilogue recombines the levels in fp64, and instead of storing fp64 U it cuts the
// value into the digit planes of row m = x no + i of the NEXT GEMM's A operand, under an a-priori power-of-two scale per (row, group)
// -- the Cauchy-Schwarz bound |U| <= |Loo[P,i,:]| |z[x,:,b]| -- so the 190 GB fp64 intermediate of a config-5 step (written once, read
// twice by the slicing pass) never exists.
// The CTAs run in clusters of 2 that take the same row tile and two consecutive (x, b tile) items: each loads half of every A stage
// and multicasts it to both, so the L2 -> SM traffic per tile drops from A + B to A / 2 + B (the kernel needs about as many bytes per
// clock from L2 as the L2 delivers to all SMs when every CTA loads its own A).
struct OzK1Params {
  const int8_t* A;    // [groups][ntg][nkb1][S][128 x 32]
  const int8_t* B;    // [nvec][nbt][nkb1][2][S][64 x 16]
  const double* sa;   // [groups][ntg * 128]  row scales of the Loo planes (packed rows)
  const double* sb;   // [nvec][nbt * 64]     row scales of the zt planes
  const double* so;   // [groups][Mpad2]      output row scales (2^(e-6), |U| < 2^e guaranteed by the bound)
  int8_t* out;        // [np][nmt2][nkb2][S][128 x 32]
  int np, ntg, nbt, nkb1, nvec, no, o2, group, nmt2, nkb2, Mpad2;
  int t0, nt_run;     // row tiles [t0, t0 + nt_run) of every group are computed ...
  int i_lo, i_hi;     // ... and only rows with i in [i_lo, i_hi) are written (a row block of a block-weighted term)
  long npairs;        // groups * nt_run * cdiv(nvec * nbt, 2): items of a CTA pair
};

// The item of CTA `crank` in pair item u: group gl, row tile, vector x, column tile bt.  When nvec * nbt is odd the second CTA of the
// last pair of a row tile repeats its partner's item (it still loads B and its half of A for the partner) and stores nothing.
struct OzK1Item {
  int gl, tile, x, bt;
  bool live;
};
__device__ __forceinline__ OzK1Item oz_k1_item(const OzK1Params& p, long u, uint32_t crank) {
  const long nxb = (long)p.nvec * p.nbt, nxb2 = (nxb + 1) >> 1, per_g = (long)p.nt_run * nxb2;
  OzK1Item t;
  t.gl = (int)(u / per_g);
  const long r0 = u - (long)t.gl * per_g;
  const int itile = (int)(r0 / nxb2);
  t.tile = p.t0 + itile;
  long xb = 2 * (r0 - (long)itile * nxb2) + crank;
  t.live = xb < nxb;
  if (!t.live) xb = nxb - 1;
  t.x = (int)(xb / p.nbt);
  t.bt = (int)(xb - (long)t.x * p.nbt);
  return t;
}

template <int S>
__global__ void __launch_bounds__(OZ_K1_THREADS, 1) oz_k1_kernel(const OzK1Params p) {
  constexpr int A_SLICE = OZ_BM * OZ_KB, B_SLICE = OZ_BN * OZ_KB;
  constexpr int A_BYTES = S * A_SLICE, B_BYTES = S * B_SLICE, STAGE = A_BYTES + B_BYTES;
  constexpr int A_HALF = A_BYTES / 2;
  constexpr uint16_t cmask = 3;
  extern __shared__ __align__(128) uint8_t oz_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(oz_smem + OZ_STAGES * STAGE);
  uint64_t* empty = full + OZ_STAGES;
  uint64_t* tmem_full = empty + OZ_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = oz_cluster_rank();
  const long pair0 = blockIdx.x >> 1, npair_ctas = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < OZ_STAGES; ++s) {
      oz_mbar_init(&full[s], 1);
      oz_mbar_init(&empty[s], 2);           // a stage is rewritten by both CTAs of the pair: both must have drained it
    }
    oz_mbar_init(tmem_full, 1);
    oz_mbar_init(tmem_empty, OZ_K1_THREADS - 64);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz_smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  oz_cluster_sync();                        // both CTAs' barriers exist before the first multicast copy / arrive
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      long it = 0;
      for (long u = pair0; u < p.npairs; u += npair_ctas) {
        const OzK1Item t = oz_k1_item(p, u, crank);
        const int8_t* a = p.A + (((long)t.gl * p.ntg + t.tile) * p.nkb1) * A_BYTES + crank * A_HALF;
        const int8_t* b = p.B + (((long)t.x * p.nbt + t.bt) * p.nkb1) * B_BYTES;
        for (int kb = 0; kb < p.nkb1; ++kb, ++it) {
          const int s = (int)(it % OZ_STAGES);
          const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
          oz_mbar_wait(&empty[s], ph ^ 1u);
          oz_mbar_expect_tx(&full[s], STAGE);
          uint8_t* sa = oz_smem + s * STAGE;
          oz_bulk_load_mc(sa + crank * A_HALF, a + (long)kb * A_BYTES, A_HALF, &full[s], cmask);
          oz_bulk_load(sa + A_BYTES, b + (long)kb * B_BYTES, B_BYTES, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BM >> 4) << 24);
      const uint32_t smem_base = oz_smem_u32(oz_smem);
      long it = 0, n = 0;
      for (long u = pair0; u < p.npairs; u += npair_ctas, ++n) {
        if (n > 0) oz_mbar_wait(tmem_empty, (uint32_t)((n - 1) & 1));      // the epilogue has drained the previous tile
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int kb = 0; kb < p.nkb1; ++kb, ++it) {
          const int s = (int)(it % OZ_STAGES);
          const uint32_t ph = (uint32_t)((it / OZ_STAGES) & 1);
          oz_mbar_wait(&full[s], ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_base = smem_base + s * STAGE, b_base = a_base + A_BYTES;
          const uint32_t later = kb > 0 ? 1u : 0u;
#pragma unroll
          for (int i = 0; i < S; ++i) {
            const uint64_t da = oz_smem_desc(a_base + i * A_SLICE, OZ_BM * 16, 128);
#pragma unroll
            for (int j0 = 0; j0 < S - i; j0 += 4) {
              const int nj = (S - i - j0) < 4 ? (S - i - j0) : 4;
              const uint64_t db = oz_smem_desc(b_base + j0 * (OZ_BN * 16), S * OZ_BN * 16, 128);
              const uint32_t idesc = idesc0 | ((uint32_t)((nj * OZ_BN) >> 3) << 17);
              oz_mma_i8(tmem_base + (uint32_t)((i + j0) * OZ_BN), da, db, idesc, (i > 0) ? 1u : later);
            }
          }
          oz_commit_mc(&empty[s], cmask);       // frees the stage in both CTAs (each of them writes half of its A part)
        }
        oz_commit(tmem_full);
      }
    }
  } else {
    // eight epilogue warps: two per TMEM lane quadrant, each takes half of the 64 columns (latency hiding for the fp64 chains)
    const int quad = warp & 3, half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const int rowsA = p.ntg * OZ_BM, rowsB = p.nbt * OZ_BN;
    long n = 0;
    for (long u = pair0; u < p.npairs; u += npair_ctas, ++n) {
      const OzK1Item t = oz_k1_item(p, u, crank);
      const int x = t.x, bt = t.bt;
      const int pr = t.tile * OZ_BM + row;             // packed row of the group
      int Pl = 0, i = 0;
      const bool valid = t.live && oz_unpack_row(pr, p.group, p.o2, p.no, Pl, i) && i >= p.i_lo && i < p.i_hi && t.gl * p.group + Pl < p.np;
      const int P = t.gl * p.group + Pl;               // aux function of the chunk
      const int m = x * p.no + i;
      const double sa = valid ? p.sa[(long)t.gl * rowsA + pr] : 0.0;
      const double so = valid ? p.so[(long)t.gl * p.Mpad2 + m] : 0.0;
      const double inv = so > 0.0 ? __hiloint2double(0x7fe00000 - __double2hiint(so), 0) : 0.0;
      const double f = sa * inv;                       // both powers of two: exact
      const double* sb = p.sb + (long)x * rowsB + bt * OZ_BN;
      int8_t* dst = p.out + ((((long)P * p.nmt2 + (m >> 7)) * p.nkb2 + bt * 2) * S) * (long)A_SLICE + (long)(m & 127) * 16;
      oz_mbar_wait(tmem_full, (uint32_t)(n & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // Drain first, cut later: all levels of this thread's 32 columns are recombined into fp64 registers and the accumulators
      // are handed back to the MMA warp BEFORE the digit extraction (two thirds of the epilogue's arithmetic), so the next
      // tile's MMAs run under it.  (With the hand-back at the end of the epilogue the tensor pipe was active 43 % of the time.)
      constexpr int HC = OZ_BN / 2;
      double v[HC];
#pragma unroll
      for (int k = 0; k < HC; ++k) v[k] = 0.0;
#pragma unroll
      for (int l = S - 1; l >= 0; --l) {
        uint32_t r[HC];
#pragma unroll
        for (int cc = 0; cc < HC; cc += 16) oz_tmem_ld16(taddr + (uint32_t)(l * OZ_BN + half * HC + cc), r + cc);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int k = 0; k < HC; ++k)     // int32 -> fp64 through the 2^52 + 2^31 offset (no conversion instruction)
          v[k] = fma(v[k], 0.00390625, __hiloint2double(0x43300000, (int)(r[k] ^ 0x80000000u)) - 4503601774854144.0);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      oz_mbar_arrive(tmem_empty);
      if (!__any_sync(0xffffffffu, valid)) continue;   // no row of this warp is stored (chunk or row-block edge, masked partner)
#pragma unroll
      for (int cc = 0; cc < HC; cc += 16) {
        const int c0 = half * HC + cc;
        uint32_t pk[S][4];
        double tt[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) tt[k] = v[cc + k] * (f * sb[c0 + k]);       // U / output scale, |tt| < 64 by the a-priori bound
        oz_digits16<S>(tt, pk);
        if (valid && bt * 2 + (c0 >> 5) < p.nkb2) {     // (a column tile may reach past the last k block of the output operand)
          // columns c0 .. c0+15 of this tile = k block (bt * 2 + c0 / 32) of the output operand, 16-byte chunk (c0 / 16) & 1
          int8_t* d = dst + (long)(c0 >> 5) * S * A_SLICE + ((c0 >> 4) & 1) * (OZ_BM * 16);
#pragma unroll
          for (int sl = 0; sl < S; ++sl) *reinterpret_cast<uint4*>(d + (long)sl * A_SLICE) = make_uint4(pk[sl][0], pk[sl][1], pk[sl][2], pk[sl][3]);
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  oz_cluster_sync();                        // no CTA leaves while its partner may still multicast into it or arrive on its barriers
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// 2-norms of the rows of a [nq][rows][K] operand (K-contiguous): out[q * rows_pad + row]
__global__ void oz_rownorm_kernel(double* __restrict__ out, int rows_pad, const double* __restrict__ X, long ld, long sq, int rows, int K) {
  const int row = blockIdx.x, q = blockIdx.y;
  double a = 0.0;
  if (row < rows) {
    const double* x = X + (long)q * sq + (long)row * ld;
    for (int k = threadIdx.x; k < K; k += blockDim.x) a = fma(x[k], x[k], a);
  }
  __shared__ double red[8];
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) a += red[w];
    out[(long)q * rows_pad + row] = sqrt(a);
  }
}
// zmax[x] = max_b |z[x][b][:]|  from the row norms [nvec][rows_pad]
__global__ void oz_colmax_kernel(double* __restrict__ zmax, const double* __restrict__ norms, int rows_pad, int rows) {
  const int x = blockIdx.x;
  double m = 0.0;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) m = fmax(m, norms[(long)x * rows_pad + r]);
  __shared__ double red[8];
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, red[w]);
    zmax[x] = m;
  }
}
// so[g][m = x no + i] = scale of the bound  zmax[x] * max_{P in group g} |Loo[P][i][:]|   (1 + 1e-9 covers rounding of the norms and
// the emulation error of U itself)
// Only rows with i in [i_lo, i_hi) are written (plus the padding rows m >= nvec no when i_lo == 0).
__global__ void oz_bound_scale_kernel(double* __restrict__ so, int Mpad2, const double* __restrict__ loo_norm, int rowsA, const double* __restrict__ zmax,
                                      int np, int group, int nvec, int no, int i_lo, int i_hi) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x, g = blockIdx.y;
  if (m >= Mpad2) return;
  double s = 0.0;
  if (m < nvec * no) {
    const int x = m / no, i = m - x * no;
    if (i < i_lo || i >= i_hi) return;
    double nl = 0.0;
    const int p1 = min(np, (g + 1) * group);
    for (int P = g * group; P < p1; ++P) nl = fmax(nl, loo_norm[(long)P * rowsA + i]);
    s = oz_scale_of(nl * zmax[x] * (1.0 + 1e-9));
  } else if (i_lo != 0) {
    return;
  }
  so[(long)g * Mpad2 + m] = s;
}

inline size_t oz_gemm_smem(int S) { return (size_t)OZ_STAGES * S * (OZ_BM + OZ_BN) * OZ_KB + 256; }

// one cluster of 2 CTAs per pair of SMs that can hold them, as many as there are pair items
template <int S>
inline int oz_k1_launch(const OzK1Params& p, cudaStream_t st) {
  static bool attr_set[64] = {false};
  static int max_clusters[64] = {0};
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(OZ_K1_THREADS);
  cfg.dynamicSmemBytes = oz_gemm_smem(S);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (!attr_set[dev & 63]) {
    XTD_CUDA(cudaFuncSetAttribute(oz_k1_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz_gemm_smem(S)));
    cfg.gridDim = dim3(2);
    XTD_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters[dev & 63], oz_k1_kernel<S>, &cfg));
    XTD_REQUIRE(max_clusters[dev & 63] >= 1, XTD_ERR_CUDA, "oz_k1: no 2-CTA cluster of the fused half-transform fits this device");
    attr_set[dev & 63] = true;
  }
  cfg.gridDim = dim3((unsigned)(2 * std::min<long>(p.npairs, max_clusters[dev & 63])));
  XTD_CUDA(cudaLaunchKernelEx(&cfg, oz_k1_kernel<S>, p));
  XTD_COUNT_LAUNCH();
  XTD_CUDA(cudaGetLastError());
  return XTD_OK;
}

inline int oz_k1(int S, const OzK1Params& p, cudaStream_t st) {
  switch (S) {
    case 3: return oz_k1_launch<3>(p, st);
    case 4: return oz_k1_launch<4>(p, st);
    case 5: return oz_k1_launch<5>(p, st);
    case 6: return oz_k1_launch<6>(p, st);
    case 7: return oz_k1_launch<7>(p, st);
    case 8: return oz_k1_launch<8>(p, st);
  }
  XTD_SET_ERR("oz_k1: %d slices (3..8)", S);
  return XTD_ERR_ARG;
}

// ---- host side --------------------------------------------------------------------------------------------------------------
struct OzShape {
  int rows = 0, RT = 0, rows_pad = 0, nrt = 0, K = 0, nkb = 0;
  void set(int rows_, int RT_, int K_) {
    rows = rows_; RT = RT_; K = K_;
    rows_pad = (int)round_up(rows_, 128);       // 128 rows per slicing block; a multiple of both tile heights
    nrt = rows_pad / RT_;
    nkb = (int)cdiv(K_, OZ_KB);
  }
  size_t slice_bytes(long nq, int S) const { return (size_t)nq * nrt * nkb * S * RT * OZ_KB; }
  size_t scale_doubles(long nq, int group) const { return (size_t)cdiv(nq, group) * rows_pad; }
};

// the largest group (q-slices sharing one scale and one int32 accumulation) that cannot overflow: per k a level holds at most
// S products of magnitude <= 2^14
inline int oz_max_group(int K, int S) {
  const long kpad = round_up(K, OZ_KB);
  const long g = ((1L << 31) - 1) / ((long)S * 16384 * kpad);
  return (int)std::max<long>(g, 0);
}

template <int S>
inline int oz_slice_launch(int8_t* out, double* scale, const OzShape& sh, const double* X, long ld, long sq, int nq, int group,
                           bool trans, long k_valid, const OzRowPack& pk, cudaStream_t st) {
  const int ng = (int)cdiv(nq, group);
  const int stacked = sh.RT == OZ_BN ? 1 : 0;
  const dim3 sgrid(2 * sh.nkb, sh.rows_pad / 128, nq);
  if (trans) {
    oz_rowmax_t_kernel<<<dim3(sh.rows_pad / 32, ng), dim3(32, 32), 0, st>>>(scale, sh.rows_pad, X, ld, sq, sh.rows, sh.K, nq, group, k_valid);
    XTD_COUNT_LAUNCH();
    XTD_CUDA(cudaGetLastError());
    oz_slice_kernel<S, true><<<sgrid, 128, 0, st>>>(out, scale, sh.rows_pad, X, ld, sq, sh.rows, sh.K, sh.RT, sh.nkb, group, stacked, k_valid, pk);
  } else {
    oz_rowmax_kernel<<<dim3(sh.rows_pad, ng), 256, 0, st>>>(scale, sh.rows_pad, X, ld, sq, sh.rows, sh.K, nq, group, k_valid, pk);
    XTD_COUNT_LAUNCH();
    XTD_CUDA(cudaGetLastError());
    oz_slice_kernel<S, false><<<sgrid, 128, 0, st>>>(out, scale, sh.rows_pad, X, ld, sq, sh.rows, sh.K, sh.RT, sh.nkb, group, stacked, k_valid, pk);
  }
  XTD_COUNT_LAUNCH();
  XTD_CUDA(cudaGetLastError());
  return XTD_OK;
}

// trans: the contraction index is the ROW index of the source array (element (row, k) at X[q sq + k ld + row]).
// k_valid: number of valid contraction indices over all q-slices together (q K + k < k_valid), <= 0 = all.
// pk: packed rows (K-contiguous sources only); the default reads plain rows.
inline int oz_slice(int S, int8_t* out, double* scale, const OzShape& sh, const double* X, long ld, long sq, int nq, int group,
                    cudaStream_t st, bool trans = false, long k_valid = 0, const OzRowPack& pk = OzRowPack()) {
  XTD_REQUIRE(nq >= 1 && nq <= 65535, XTD_ERR_ARG, "oz_slice: %d q-slices per launch (1..65535)", nq);
  XTD_REQUIRE(trans || (ld % 2 == 0 && sq % 2 == 0 && pk.sp % 2 == 0 && ((uintptr_t)X & 15) == 0), XTD_ERR_ALIGN,
              "oz_slice: operand must be 16-byte aligned with even strides");
  XTD_REQUIRE(pk.G == 0 || (!trans && pk.o2 >= 1 && pk.o2 <= pk.no && pk.G * pk.no <= sh.rows_pad), XTD_ERR_ARG, "oz_slice: bad row packing");
  if (k_valid <= 0) k_valid = (long)nq * sh.K;
  switch (S) {
    case 3: return oz_slice_launch<3>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
    case 4: return oz_slice_launch<4>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
    case 5: return oz_slice_launch<5>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
    case 6: return oz_slice_launch<6>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
    case 7: return oz_slice_launch<7>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
    case 8: return oz_slice_launch<8>(out, scale, sh, X, ld, sq, nq, group, trans, k_valid, pk, st);
  }
  XTD_SET_ERR("oz_slice: %d slices (3..8)", S);
  return XTD_ERR_ARG;
}

template <int S, int CN>
inline int oz_gemm_launch_cn(const OzGemmParams& p, cudaStream_t st) {
  static bool attr_set[64] = {false};
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    XTD_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<S, CN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz_gemm_smem(S)));
    attr_set[dev & 63] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(p.nmt * p.nnt * p.splits), (unsigned)p.batches);
  cfg.blockDim = dim3(OZ_THREADS);
  cfg.dynamicSmemBytes = oz_gemm_smem(S);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CN;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  XTD_CUDA(cudaLaunchKernelEx(&cfg, oz_gemm_kernel<S, CN>, p));
  XTD_COUNT_LAUNCH();
  XTD_CUDA(cudaGetLastError());
  return XTD_OK;
}

template <int S>
inline int oz_gemm_p_launch(const OzGemmParams& p, cudaStream_t st) {
  static bool attr_set[64] = {false};
  static int sms[64] = {0};
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    XTD_CUDA(cudaFuncSetAttribute(oz_gemm_p_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz_gemm_smem(S)));
    XTD_CUDA(cudaDeviceGetAttribute(&sms[dev & 63], cudaDevAttrMultiProcessorCount, dev));
    attr_set[dev & 63] = true;
  }
  const long items = (long)p.nmt * p.nnt * p.splits * p.batches;
  const unsigned grid = (unsigned)std::min<long>(items, sms[dev & 63]);
  oz_gemm_p_kernel<S><<<grid, OZ_K1_THREADS, oz_gemm_smem(S), st>>>(p);
  XTD_COUNT_LAUNCH();
  XTD_CUDA(cudaGetLastError());
  return XTD_OK;
}

// Which kernel runs a contraction: the persistent one pays off when a tile holds one or two accumulation groups (grid GEMMs, short
// contractions: config 5 grid GEMMs 163 -> 148 ms at a LOWER clock), the one-tile-per-CTA kernel with its cluster multicast of the A
// tile for long contractions (exchange: 587 vs 646 ms -- the step is power-capped and the multicast halves the A traffic per SM).
inline bool oz_persistent(const OzGemmParams& p) {
  const int ngroups = (p.nq + p.group - 1) / p.group;
  return ngroups <= 2 * p.splits;
}

// The one-tile-per-CTA kernel multicasts the A tile to a cluster of 2 CTAs along N when the column-tile count is even
// (4 CTAs measured slower: 16 SMs strand).
template <int S>
inline int oz_gemm_launch(const OzGemmParams& p, cudaStream_t st) {
  if (oz_persistent(p)) return oz_gemm_p_launch<S>(p, st);
  if (p.nnt % 2 == 0) return oz_gemm_launch_cn<S, 2>(p, st);
  return oz_gemm_launch_cn<S, 1>(p, st);
}

inline int oz_gemm(int S, const OzGemmParams& p, cudaStream_t st) {
  XTD_REQUIRE(p.group >= 1 && p.group <= oz_max_group(p.nkb * OZ_KB, S), XTD_ERR_ARG, "oz_gemm: group %d would overflow int32 (max %d)", p.group,
              oz_max_group(p.nkb * OZ_KB, S));
  XTD_REQUIRE(p.b_q0 % p.group == 0, XTD_ERR_ARG, "oz_gemm: first B slice %d must sit on a group boundary (%d)", p.b_q0, p.group);
  switch (S) {
    case 3: return oz_gemm_launch<3>(p, st);
    case 4: return oz_gemm_launch<4>(p, st);
    case 5: return oz_gemm_launch<5>(p, st);
    case 6: return oz_gemm_launch<6>(p, st);
    case 7: return oz_gemm_launch<7>(p, st);
    case 8: return oz_gemm_launch<8>(p, st);
  }
  XTD_SET_ERR("oz_gemm: %d slices (3..8)", S);
  return XTD_ERR_ARG;
}

// split of the group range that fills the SMs with whole waves
inline int oz_choose_splits(int tiles, int ngroups, int num_sms) {
  int best = 1;
  double best_cost = 1e300;
  const int max_s = std::min(ngroups, 64);
  for (int s = 1; s <= max_s; ++s) {
    const long waves = cdiv((long)tiles * s, num_sms);
    const double cost = (double)waves * ((double)cdiv(ngroups, s) + 0.05);
    if (cost < best_cost * 0.995) { best_cost = cost; best = s; }
  }
  return best;
}

}  // namespace xtd
