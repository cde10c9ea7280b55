// libxtdsigma.so: engine + C-ABI (include/xtd_sigma.h).  sm_100a only.
//
// Data layout in HBM (all fp64, leading dimensions padded to 16 doubles):
//   per channel   Co/Cv [nao][ld], CoT/CvT [n][ldN]        AO <-> internal MO positions (zero pad orbitals)
//   per (tensor, channel) with an exchange term
//                 Loo [naux_loc][no][ld_oo], Lvv [naux_loc][nv][ld_vv]   MO-resident 3-centre blocks
//   per Coulomb block  Ljb [naux_loc][nr][ld]
//   grid          phi [ch][nvar][ng][ld_o] = ao . Co and phiv [ch][nvar][ng][ld_v] = ao . Cv (the caller's ao buffer is
//                 only read by xtd_grid_commit), per-point kernel table wf
//   per call (workspace arena)  Z, ZT, ZTs, SIG, Y/U chunk, split-K partials
#include "../../include/xtd_sigma.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include "ozaki.cuh"
#include "davidson.cuh"

#include <cuda_profiler_api.h>

#include <algorithm>
#include <cstring>
#include <vector>

namespace xtd {
thread_local char g_last_error[512] = {0};
unsigned long long g_launch_count = 0;

// Owned device buffer, zero-filled on the stream whose kernels will fill it (a cudaMemset on the legacy stream is not
// ordered against work on a non-blocking side stream and could land after the producer's output).
struct DevBuf {
  double* p = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  int alloc(size_t n_doubles, cudaStream_t s) {
    release();
    bytes = std::max<size_t>(n_doubles, 2) * 8;
    XTD_CUDA(cudaMalloc(&p, bytes));
    XTD_CUDA(cudaMemsetAsync(p, 0, bytes, s));
    return XTD_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
};

struct Channel {
  int spin_o, spin_v, no, nv;
  std::vector<int> occ_idx, vir_idx;
  std::vector<std::pair<int, int>> o_blocks, v_blocks;
  long ldz, ldzt, ldco, ldcv, ldN;
  DevBuf Co, Cv, CoT, CvT;          // [nao][ldco], [nao][ldcv], [no][ldN], [nv][ldN]
  DevBuf Loo[2], Lvv[2];            // per DF tensor
  DevBuf Loob[2][2];                // per DF tensor and occupied row block: [naux_loc][rows of the block][ldoo], so that
  bool need_split[2] = {false, false};   // (aux, row) flattens into one uniformly strided row index for block weights
  DevBuf Lvo[2];                    // [naux_loc][v2off][ldvv]: rows of Lvv in the narrow first virtual block (open shells),
  bool need_narrow[2] = {false, false};   // gathered so (aux, row) flattens: narrow-output exchange pass (run_k)
  DevBuf Lvt[2];                    // [naux_loc][tail_w][ldvv]: the last rows of Lvv past a multiple of 128 in the second block
  DevBuf Lov[2];                    // [naux_loc][no][ldz]: occupied-virtual block, exchange of the transposed trial density
  bool need_kt[2] = {false, false}; // (xtd_add_kterm_t: the B-matrix-type term of the Z-vector operator)
  int tail_start = 0, tail_w = 0;   // (a short column tail of the block-weighted output takes the same pass)
  long ldoo, ldvv;
  bool need_k[2] = {false, false};
  // INT8-emulated exchange contraction (ozaki.cuh): Lvv kept only as int8 slices + row scales, no fp64 copy
  bool use_oz[2] = {false, false};
  int8_t* LvvS[2] = {nullptr, nullptr};     // [naux_loc][nnt][nkb][S][64 x 32]
  double* LvvScale[2] = {nullptr, nullptr}; // [groups][rows_pad]
  OzShape ozB;
  int oz_group = 0;
  int oz_col0[2] = {0, 0};                  // first output column of the emulated block: 0, or the start of the second virtual
                                            // block for block-weighted terms (the narrow first block keeps its DMMA pass)
  // ... and the occupied-occupied block as the A operand of the fused half-transform (oz_k1_kernel): planes and row scales with the
  // rows (P, i) of oz_group aux functions packed into one q-slice (oz_unpack_row, split at oz_row_split()), row 2-norms [naux_loc][no]
  int8_t* LooS[2] = {nullptr, nullptr};
  double *LooScale[2] = {nullptr, nullptr}, *LooNorm[2] = {nullptr, nullptr};
  OzShape ozL;
  int oz_row_split() const { return o_blocks.size() > 1 ? o_blocks[1].first : no; }
  // grid path on the emulated GEMMs (one AO component): MO values of the virtual orbitals kept as int8 planes in both operand
  // roles -- rows = grid points, K = virtual index (forward Y = phiv . z^T) and rows = virtual index, K = blocks of OZ_XC_KQ grid
  // points (backward sigma += A^T . phiv) -- instead of the fp64 array
  bool xc_oz = false;
  int8_t *phivF = nullptr, *phivB = nullptr;
  double *phivFs = nullptr, *phivBs = nullptr;
  OzShape ozPF, ozPB;
  // value + gradient kernels in the split-gradient form: the four value GEMMs are emulated (planes of the value component of phiv
  // as above, and of the value component of phi: rows = grid points, K = occupied index / rows = occupied index, K = grid blocks);
  // the fp64 arrays stay (the streaming kernel reads the gradient components)
  bool xc_oz_split = false;
  int8_t *phiF = nullptr, *phiB = nullptr;
  double *phiFs = nullptr, *phiBs = nullptr;
  OzShape ozOF, ozOB;
  DevBuf phi;                       // occupied values on the grid  [nvar_eff][ng][ldphi]
  long ldphi = 0;
  DevBuf phiv;                      // virtual values on the grid   [nvar_eff][ng][ldphiv]
  long ldphiv = 0;
  // gather CSR
  long *g_indptr = nullptr, *g_cols = nullptr;
  double* g_vals = nullptr;
  long g_nnz = 0;
};

constexpr long XC_SPLIT_SMEM_MAX = 200 * 1024;   // shared memory of the split-gradient streaming kernel (MO values of one point)
constexpr int XC_OP_MAX_NVEC = 8;   // batches up to this size take the orbital-range streaming kernel (xc_weight_split_op_kernel)
constexpr int OZ_XC_KQ = 8192;   // grid points per int32 accumulation group of the backward grid GEMM (8192 * S * 2^14 < 2^31)
constexpr int NARROW_MAX = 16;   // widest first virtual block that takes the narrow-output exchange pass

struct KTermRec {
  int tensor, ch, nob, nvb;
  double w[2][2][2][2];
  bool uniform;
};
struct KTermTRec {
  int tensor, ch;
  double w;
};
struct JBlockRec {
  int ch, r0, nr, c0, nc;
  long ld;
  DevBuf L;   // [naux_loc][nr][ld]
};
struct LocalGemmRec {
  int side, dch, r0, nr, c0, nc, sch, sr0, sc0, mrows, mcols;
  long ldm;
  double alpha;
  DevBuf M;
};
struct Rank1Rec {
  int dch, sch;
  DevBuf U, V;
};
struct DiagRec {
  int ch;
  DevBuf D;
};

// Environment switches that force a path the engine also takes by itself on some inputs (tests use them to reach those paths at
// small sizes) or that place a profiler range.  Read once, in xtd_create, so every decision of an engine sees the same values.
struct EnvSwitches {
  // XTD_CHUNK_AUX / XTD_CHUNK_GRID: upper bounds on the aux / grid chunk of a call (tests force the multi-chunk loops that
  // BASELINE-size runs take at oracle-sized inputs); the chunk counts of the last call are reported by xtd_last_chunks
  long max_pc = 0, max_gb = 0;
  // XTD_OZ_SHORT_K: contraction lengths below this stay on the FP64 DMMA GEMM where a kernel offers the choice (tests use 0)
  int oz_short_k = 100;
  int xc_split = -1;          // XTD_XC_SPLIT: 1 / 0 forces the split-gradient / four-component grid form, -1 chooses by cost
  bool no_narrow = false;     // XTD_NO_NARROW set: block-weighted exchange without the narrow-output pass
  bool j_stream = false;      // XTD_J_STREAM set: Coulomb blocks on the streaming kernels only
  // XTD_PROFILE_PHASE=<XTD_T_* id>: cudaProfilerStart/Stop around that phase (ncu --profile-from-start off)
  int prof_phase = -1;
};

struct Arena {
  char* base = nullptr;
  size_t cap = 0, used = 0;
  double* take(size_t n_doubles) {
    size_t b = (n_doubles * 8 + 255) & ~(size_t)255;
    if (used + b > cap) return nullptr;
    double* p = (double*)(base + used);
    used += b;
    return p;
  }
  size_t left() const { return cap - used; }
};

}  // namespace xtd

using namespace xtd;

struct xtd_engine {
  int nao = 0;
  long ldN = 0;
  cudaStream_t stream = 0;
  GemmContext gemm;
  Arena arena;
  EnvSwitches env;
  // orbitals
  const double* C[2] = {nullptr, nullptr};
  long ldC[2] = {0, 0};
  int nmo[2] = {0, 0};
  std::vector<Channel*> ch;
  std::vector<KTermRec> kterms;
  std::vector<KTermTRec> ktterms;
  std::vector<JBlockRec*> jblocks;
  std::vector<double> jmix;
  DevBuf jmix_dev;
  // ROHF-form Fock difference K[D_open] (xtd_set_open_orbitals): accumulated from the streamed tensor
  int kopen_spin = -1, n_open = 0;
  DevBuf CuT, CallT, kopen;    // [n_open][ldN], [nmo][ldN], [nmo][ld_mo]
  long ld_mo = 0;
  long naux[2] = {0, 0};       // local aux count per tensor
  long naux_filled[2] = {0, 0};
  // grid
  const double* ao = nullptr;
  const double* wgrid = nullptr;
  int nvar = 0, nvar_eff = 0;
  long ng = 0, ao_ld = 0, ao_comp = 0;
  int fxc_kind = XTD_FXC_NONE;
  bool tau = false;            // meta-GGA: kernel tables with a fifth (tau) component
  const double* fxc = nullptr;
  DevBuf wf;
  bool grid_committed = false;
  // local terms
  bool small_local = false;            // all local GEMM / diagonal terms in one launch (launch-bound molecules)
  LocalTermDev *lt_dev = nullptr, *ld_dev = nullptr;
  std::vector<LocalGemmRec*> lgemms;
  std::vector<Rank1Rec*> rank1s;
  std::vector<DiagRec*> diags;
  // scatter
  long ext_dim = 0;
  long *s_indptr = nullptr, *s_offs = nullptr;
  signed char* s_chans = nullptr;
  double* s_vals = nullptr;
  // state
  bool finalized = false;
  int max_nvec = 0;
  int cur_nvec = 0;
  // per-call buffers (arena)
  double *Z[2] = {nullptr, nullptr}, *ZT[2] = {nullptr, nullptr}, *ZTs[2] = {nullptr, nullptr};
  double* SIG = nullptr;
  long sig_base[2] = {0, 0};
  double* scratch = nullptr;      // Y / U chunk region
  size_t scratch_doubles = 0;
  double *jR = nullptr, *jRm = nullptr, *r1d = nullptr;
  // pinned staging for the host entry
  double *pin_in = nullptr, *pin_out = nullptr, *dev_in = nullptr, *dev_out = nullptr;
  size_t pin_doubles = 0;
  // timers: a pool of event pairs, one per phase occurrence of the last call, summed per phase on query
  struct EvRec { cudaEvent_t a, b; int id; };
  std::vector<EvRec> evpool;
  size_t ev_used = 0;
  cudaEvent_t ev_total[2];
  bool ev_ok = false;
  unsigned long long launches0 = 0;
  double flops0 = 0;
  double phase_flops[12] = {0};   // GEMM flops per phase of the last call
  int oz_slices = 0;              // 0: FP64 DMMA exchange contraction; 3..8: INT8 tensor-core emulation with that many slices
  long last_aux_chunks = 0, last_grid_chunks = 0;
  long last_dens_batches = 0;     // passes over the densities of the last xtd_block_response_batch (workspace-bound sub-batches)
  // Launch-bound calls (small molecules: ~50-100 launches of a few microseconds each) are replayed as CUDA graphs: the
  // first call with a given (nvec, z, hz) runs eagerly, the second is captured, later ones are one cudaGraphLaunch.
  struct GraphRec {
    int nvec; const double* z; double* hz;
    cudaGraphExec_t exec;
    unsigned long long launches; double flops; double phase_flops[12];
  };
  std::vector<GraphRec> graphs;
  bool graphs_off = false;        // set when a capture failed: later calls run eagerly
  // xtd_enable_block_response: Loo / Lvv of tensor 0 stay resident for every channel (Coulomb of occupied-occupied and
  // virtual-virtual densities) and the fp64 virtual MO values stay on the grid next to their int8 planes
  bool block_resp = false;
  bool capturing = false;
  cudaStream_t cap_stream = nullptr;   // calls are recorded on this stream (the caller's may be the legacy default stream,
                                       // which cannot be captured) and replayed on the caller's
  int last_eager_nvec = 0; const double* last_eager_z = nullptr; double* last_eager_hz = nullptr; double last_eager_flops = 0;
};

namespace {

struct PhaseTimer {
  xtd_engine* h;
  size_t slot = (size_t)-1;
  int phase;
  double f0;
  PhaseTimer(xtd_engine* h_, int id) : h(h_), phase(id), f0(h_->gemm.flops) {
    if (!h->ev_ok || h->capturing) return;
    if (h->ev_used == h->evpool.size()) {
      if (h->evpool.size() >= 4096) return;
      xtd_engine::EvRec r;
      cudaEventCreate(&r.a);
      cudaEventCreate(&r.b);
      r.id = id;
      h->evpool.push_back(r);
    }
    slot = h->ev_used++;
    h->evpool[slot].id = id;
    if (id == h->env.prof_phase) cudaProfilerStart();
    cudaEventRecord(h->evpool[slot].a, h->stream);
  }
  ~PhaseTimer() {
    h->phase_flops[phase] += h->gemm.flops - f0;
    if (slot == (size_t)-1) return;
    cudaEventRecord(h->evpool[slot].b, h->stream);
    if (h->evpool[slot].id == h->env.prof_phase) cudaProfilerStop();
  }
};

inline dim3 grid1d(long n, int threads, int y = 1, int z = 1) { return dim3((unsigned)cdiv(n, threads), y, z); }

#define LAUNCH_CHECK()              \
  do {                              \
    XTD_COUNT_LAUNCH();             \
    XTD_CUDA(cudaGetLastError());   \
  } while (0)

int upload_padded(DevBuf& dst, long& ld, const double* host, int rows, int cols, cudaStream_t s) {
  ld = pad_ld(cols);
  XTD_TRY(dst.alloc((size_t)std::max(rows, 1) * ld, s));
  if (rows > 0 && cols > 0) {      // after the zero fill, on the same stream
    XTD_CUDA(cudaMemcpy2DAsync(dst.p, ld * 8, host, (size_t)cols * 8, (size_t)cols * 8, rows, cudaMemcpyHostToDevice, s));
    XTD_CUDA(cudaStreamSynchronize(s));
  }
  return XTD_OK;
}

template <typename T>
int upload_array(T** dst, const T* host, size_t n, cudaStream_t s) {
  if (*dst) cudaFree(*dst);
  *dst = nullptr;
  XTD_CUDA(cudaMalloc((void**)dst, std::max<size_t>(n, 1) * sizeof(T)));
  if (n) {
    XTD_CUDA(cudaMemcpyAsync(*dst, host, n * sizeof(T), cudaMemcpyHostToDevice, s));
    XTD_CUDA(cudaStreamSynchronize(s));
  }
  return XTD_OK;
}

// ---- layout of the internal sigma / Z buffers for nvec vectors: channel-major, each [nvec*no][ldz] -----
void sig_layout(const xtd_engine* h, int nvec, long* base, long* total) {
  long off = 0;
  for (size_t c = 0; c < h->ch.size(); ++c) {
    base[c] = off;
    off += (long)nvec * h->ch[c]->no * h->ch[c]->ldz;
  }
  *total = off;
}

int build_channel_matrices(xtd_engine* h, Channel* c) {
  XTD_REQUIRE(h->C[c->spin_o] && h->C[c->spin_v], XTD_ERR_STATE, "xtd_set_mo must precede xtd_add_channel");
  const int N = h->nao;
  c->ldco = pad_ld(c->no);
  c->ldcv = pad_ld(c->nv);
  c->ldN = h->ldN;
  XTD_TRY(c->Co.alloc((size_t)N * c->ldco, h->stream));
  XTD_TRY(c->Cv.alloc((size_t)N * c->ldcv, h->stream));
  XTD_TRY(c->CoT.alloc((size_t)c->no * c->ldN, h->stream));
  XTD_TRY(c->CvT.alloc((size_t)c->nv * c->ldN, h->stream));
  int *d_oi = nullptr, *d_vi = nullptr;
  XTD_TRY(upload_array(&d_oi, c->occ_idx.data(), c->occ_idx.size(), h->stream));
  XTD_TRY(upload_array(&d_vi, c->vir_idx.data(), c->vir_idx.size(), h->stream));
  gather_cols_kernel<<<dim3((unsigned)cdiv(c->no, 128), N), 128, 0, h->stream>>>(c->Co.p, c->ldco, h->C[c->spin_o], h->ldC[c->spin_o], N,
                                                                               d_oi, c->no);
  LAUNCH_CHECK();
  gather_cols_kernel<<<dim3((unsigned)cdiv(c->nv, 128), N), 128, 0, h->stream>>>(c->Cv.p, c->ldcv, h->C[c->spin_v], h->ldC[c->spin_v], N,
                                                                               d_vi, c->nv);
  LAUNCH_CHECK();
  dim3 tb(32, 8);
  transpose_kernel<<<dim3((unsigned)cdiv(c->no, 32), (unsigned)cdiv(N, 32), 1), tb, 0, h->stream>>>(c->CoT.p, c->ldN, 0, c->Co.p, c->ldco,
                                                                                                    0, N, c->no);
  LAUNCH_CHECK();
  transpose_kernel<<<dim3((unsigned)cdiv(c->nv, 32), (unsigned)cdiv(N, 32), 1), tb, 0, h->stream>>>(c->CvT.p, c->ldN, 0, c->Cv.p, c->ldcv,
                                                                                                    0, N, c->nv);
  LAUNCH_CHECK();
  XTD_CUDA(cudaStreamSynchronize(h->stream));
  cudaFree(d_oi);
  cudaFree(d_vi);
  return XTD_OK;
}

// Loo / Lvv of `tensor` are built for channel c: an exchange term needs them, or the block response keeps the Coulomb ones
bool oovv_resident(const xtd_engine* h, const Channel* c, int tensor) { return c->need_k[tensor] || (tensor == 0 && h->block_resp); }

MatView view2d(const double* base, long ld, int rows, int cols, int row0 = 0, int col0 = 0) {
  MatView v;
  v.base = base; v.ld = ld; v.sq = 0; v.row0 = row0; v.col0 = col0; v.rows = rows; v.cols = cols; v.q0 = 0; v.nq = 1;
  return v;
}
MatView view3d(const double* base, long ld, long sq, int nq, int rows, int cols, int row0 = 0, int col0 = 0, int q0 = 0) {
  MatView v = view2d(base, ld, rows, cols, row0, col0);
  v.sq = sq; v.nq = nq; v.q0 = q0;
  return v;
}

// AO values -> MO values on the grid, once per solve (the MO<->AO transforms of the reference's vind applied to the
// grid basis instead of to every trial vector):
//   phi [c][g][o] = sum_mu ao[c][g][mu] Co[mu][o]      phiv[c][g][v] = sum_mu ao[c][g][mu] Cv[mu][v]
// plus the per-point kernel tables.  Afterwards the caller's ao / weights buffers are no longer referenced.
int grid_commit(xtd_engine* h) {
  XTD_REQUIRE(h->ao && h->fxc_kind != XTD_FXC_NONE, XTD_ERR_STATE, "grid commit: xtd_set_grid and xtd_set_fxc come first");
  XTD_REQUIRE(!h->ch.empty(), XTD_ERR_STATE, "grid commit: channels must be declared first");
  if (h->fxc_kind == XTD_FXC_UKS) XTD_REQUIRE(h->ch.size() == 2, XTD_ERR_ARG, "UKS kernel needs two channels");
  else XTD_REQUIRE(h->ch.size() == 1, XTD_ERR_ARG, "spin-flip kernels need one channel");
  cudaStream_t s = h->stream;
  h->nvar_eff = (h->fxc_kind == XTD_FXC_ALDA0) ? 1 : h->nvar;
  if (h->ng > 0) {
    h->arena.used = 0;
    size_t split_bytes = std::min<size_t>(h->arena.cap / 4, (size_t)1 << 30);
    h->gemm.split_ws = h->arena.take(split_bytes / 8);
    h->gemm.split_ws_bytes = split_bytes;
    for (auto* c : h->ch) {
      c->ldphi = pad_ld(c->no);
      c->ldphiv = pad_ld(c->nv);
      XTD_TRY(c->phi.alloc((size_t)h->nvar_eff * h->ng * c->ldphi, h->stream));
      XTD_TRY(c->phiv.alloc((size_t)h->nvar_eff * h->ng * c->ldphiv, h->stream));
      GemmDesc d;
      d.A = view3d(h->ao, h->ao_ld, h->ao_comp, h->nvar_eff, (int)h->ng, h->nao);
      d.B = view2d(c->CoT.p, h->ldN, c->no, h->nao);
      d.M = (int)h->ng; d.N = c->no; d.K = h->nao; d.batches = h->nvar_eff; d.a_hi = 1; d.b_hi = 0;
      d.C = c->phi.p; d.ldc = c->ldphi; d.c_batch_stride = h->ng * c->ldphi;
      XTD_TRY(gemm(h->gemm, d, s));
      GemmDesc e = d;
      e.B = view2d(c->CvT.p, h->ldN, c->nv, h->nao);
      e.N = c->nv;
      e.C = c->phiv.p; e.ldc = c->ldphiv; e.c_batch_stride = h->ng * c->ldphiv;
      XTD_TRY(gemm(h->gemm, e, s));
      bool split_oz = false;
      if (h->oz_slices > 0 && h->nvar_eff == 4 && !h->tau && h->env.xc_split != 0) {
        int no2[2] = {0, 0}, nv2[2] = {0, 0};
        for (size_t k = 0; k < h->ch.size(); ++k) { no2[k] = h->ch[k]->no; nv2[k] = h->ch[k]->nv; }
        split_oz = xc_split_smem_doubles((int)h->ch.size(), no2, nv2) * 8 <= XC_SPLIT_SMEM_MAX;
      }
      if (h->oz_slices > 0 && (h->nvar_eff == 1 || split_oz)) {
        // both operand roles of (the value component of) phiv as int8 planes
        const int S = h->oz_slices;
        c->ozPF.set((int)h->ng, OZ_BM, c->nv);
        c->ozPB.set(c->nv, OZ_BN, OZ_XC_KQ);
        const long nqg = cdiv(h->ng, OZ_XC_KQ);
        XTD_REQUIRE(nqg <= 65535, XTD_ERR_UNSUPPORTED, "grid too long for the emulated grid path");
        XTD_CUDA(cudaMalloc((void**)&c->phivF, c->ozPF.slice_bytes(1, S)));
        XTD_CUDA(cudaMalloc((void**)&c->phivFs, c->ozPF.scale_doubles(1, 1) * 8));
        XTD_CUDA(cudaMalloc((void**)&c->phivB, c->ozPB.slice_bytes(nqg, S)));
        XTD_CUDA(cudaMalloc((void**)&c->phivBs, c->ozPB.scale_doubles(nqg, 1) * 8));
        XTD_TRY(oz_slice(S, c->phivF, c->phivFs, c->ozPF, c->phiv.p, c->ldphiv, 0, 1, 1, s));
        XTD_TRY(oz_slice(S, c->phivB, c->phivBs, c->ozPB, c->phiv.p, c->ldphiv, (long)OZ_XC_KQ * c->ldphiv, (int)nqg, 1, s, true, h->ng));
        if (split_oz) {
          // ... and of the value component of phi (occupied side of the split-gradient form)
          c->ozOF.set((int)h->ng, OZ_BM, c->no);
          c->ozOB.set(c->no, OZ_BM, OZ_XC_KQ);
          if (c->no >= h->env.oz_short_k) {
            XTD_CUDA(cudaMalloc((void**)&c->phiF, c->ozOF.slice_bytes(1, S)));
            XTD_CUDA(cudaMalloc((void**)&c->phiFs, c->ozOF.scale_doubles(1, 1) * 8));
          }
          XTD_CUDA(cudaMalloc((void**)&c->phiB, c->ozOB.slice_bytes(nqg, S)));
          XTD_CUDA(cudaMalloc((void**)&c->phiBs, c->ozOB.scale_doubles(nqg, 1) * 8));
          if (c->no >= h->env.oz_short_k) XTD_TRY(oz_slice(S, c->phiF, c->phiFs, c->ozOF, c->phi.p, c->ldphi, 0, 1, 1, s));
          XTD_TRY(oz_slice(S, c->phiB, c->phiBs, c->ozOB, c->phi.p, c->ldphi, (long)OZ_XC_KQ * c->ldphi, (int)nqg, 1, s, true, h->ng));
        }
        XTD_CUDA(cudaStreamSynchronize(s));
        if (split_oz) {
          c->xc_oz_split = true;
        } else {
          if (!h->block_resp) c->phiv.release();   // one component: the sigma path does not read the fp64 array again
          c->xc_oz = true;
        }
      }
    }
    if (h->tau) XTD_REQUIRE(h->nvar == 4, XTD_ERR_ARG, "meta-GGA kernels need value + gradient AO components (nvar = 4)");
    const int nk = h->tau ? 5 : h->nvar;        // kernel components
    if (h->fxc_kind == XTD_FXC_UKS) {
      const int nr = 2 * nk;
      XTD_TRY(h->wf.alloc((size_t)h->ng * nr * nr, h->stream));
      build_wf_uks_kernel<<<grid1d(h->ng, 128), 128, 0, s>>>(h->wf.p, h->fxc, h->wgrid, h->ng, nk);
      LAUNCH_CHECK();
    } else if (h->fxc_kind == XTD_FXC_MCOL) {
      XTD_TRY(h->wf.alloc((size_t)h->ng * nk * nk, h->stream));
      build_wf_mcol_kernel<<<grid1d(h->ng, 128), 128, 0, s>>>(h->wf.p, h->fxc, h->wgrid, h->ng, nk);
      LAUNCH_CHECK();
    }
    XTD_CUDA(cudaStreamSynchronize(s));
  }
  h->grid_committed = true;
  h->ao = nullptr;
  h->wgrid = nullptr;
  if (h->fxc_kind != XTD_FXC_ALDA0) h->fxc = nullptr;   // ALDA0 reads the caller's weighted kernel f[ng] on every call
  return XTD_OK;
}

}  // namespace

// =========================================================================================================
// C-ABI
// =========================================================================================================
extern "C" {

const char* xtd_last_error(void) { return g_last_error; }
int xtd_version(void) { return 100; }
unsigned long long xtd_launch_count(void) { return g_launch_count; }

int xtd_create(xtd_handle* out, int nao, long workspace_bytes) {
  XTD_REQUIRE(out && nao > 0 && workspace_bytes >= (64L << 20), XTD_ERR_ARG, "xtd_create: bad arguments (workspace >= 64 MiB)");
  int dev = 0, major = 0, minor = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  XTD_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  XTD_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  // the library carries sm_100a SASS only (no PTX): any other device would fail at the first launch
  XTD_REQUIRE(major == 10 && minor == 0, XTD_ERR_UNSUPPORTED, "xtd_create: needs an sm_100a device (found compute capability %d.%d)", major,
              minor);
  xtd_engine* h = new xtd_engine();
  h->nao = nao;
  h->ldN = pad_ld(nao);
  int r = gemm_context_init(h->gemm);
  if (r != XTD_OK) { delete h; return r; }
  cudaError_t e = cudaMalloc((void**)&h->arena.base, (size_t)workspace_bytes);
  if (e != cudaSuccess) {
    XTD_SET_ERR("xtd_create: cannot allocate %ld workspace bytes: %s", workspace_bytes, cudaGetErrorString(e));
    delete h;
    return XTD_ERR_NOMEM;
  }
  h->arena.cap = (size_t)workspace_bytes;
  cudaEventCreate(&h->ev_total[0]);
  cudaEventCreate(&h->ev_total[1]);
  h->ev_ok = true;
  EnvSwitches& env = h->env;
  if (const char* e = getenv("XTD_CHUNK_AUX")) env.max_pc = atol(e);
  if (const char* e = getenv("XTD_CHUNK_GRID")) env.max_gb = atol(e);
  if (const char* e = getenv("XTD_OZ_SHORT_K")) env.oz_short_k = atoi(e);
  if (const char* e = getenv("XTD_XC_SPLIT")) env.xc_split = atoi(e) != 0;
  env.no_narrow = getenv("XTD_NO_NARROW") != nullptr;
  env.j_stream = getenv("XTD_J_STREAM") != nullptr;
  if (const char* e = getenv("XTD_PROFILE_PHASE")) env.prof_phase = atoi(e);
  *out = h;
  return XTD_OK;
}

int xtd_destroy(xtd_handle h) {
  if (!h) return XTD_OK;
  cudaDeviceSynchronize();
  for (auto* c : h->ch) {
    c->Co.release(); c->Cv.release(); c->CoT.release(); c->CvT.release(); c->phi.release(); c->phiv.release();
    for (int t = 0; t < 2; ++t) { c->Loo[t].release(); c->Lvv[t].release(); c->Lvo[t].release(); c->Lvt[t].release(); c->Loob[t][0].release(); c->Loob[t][1].release(); }
    for (int t = 0; t < 2; ++t) {
      if (c->LvvS[t]) cudaFree(c->LvvS[t]);
      if (c->LvvScale[t]) cudaFree(c->LvvScale[t]);
      if (c->LooS[t]) cudaFree(c->LooS[t]);
      if (c->LooScale[t]) cudaFree(c->LooScale[t]);
      if (c->LooNorm[t]) cudaFree(c->LooNorm[t]);
    }
    if (c->phiF) cudaFree(c->phiF);
    if (c->phiB) cudaFree(c->phiB);
    if (c->phiFs) cudaFree(c->phiFs);
    if (c->phiBs) cudaFree(c->phiBs);
    if (c->phivF) cudaFree(c->phivF);
    if (c->phivB) cudaFree(c->phivB);
    if (c->phivFs) cudaFree(c->phivFs);
    if (c->phivBs) cudaFree(c->phivBs);
    if (c->g_indptr) cudaFree(c->g_indptr);
    if (c->g_cols) cudaFree(c->g_cols);
    if (c->g_vals) cudaFree(c->g_vals);
    delete c;
  }
  for (auto* j : h->jblocks) { j->L.release(); delete j; }
  for (auto* l : h->lgemms) { l->M.release(); delete l; }
  for (auto* r : h->rank1s) { r->U.release(); r->V.release(); delete r; }
  for (auto* d : h->diags) { d->D.release(); delete d; }
  h->jmix_dev.release(); h->wf.release(); h->CuT.release(); h->CallT.release(); h->kopen.release();
  if (h->lt_dev) cudaFree(h->lt_dev);
  if (h->ld_dev) cudaFree(h->ld_dev);
  if (h->s_indptr) cudaFree(h->s_indptr);
  if (h->s_offs) cudaFree(h->s_offs);
  if (h->s_chans) cudaFree(h->s_chans);
  if (h->s_vals) cudaFree(h->s_vals);
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->arena.base) cudaFree(h->arena.base);
  if (h->pin_in) cudaFreeHost(h->pin_in);
  if (h->pin_out) cudaFreeHost(h->pin_out);
  if (h->dev_in) cudaFree(h->dev_in);
  if (h->dev_out) cudaFree(h->dev_out);
  if (h->ev_ok) {
    cudaEventDestroy(h->ev_total[0]);
    cudaEventDestroy(h->ev_total[1]);
    for (auto& r : h->evpool) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  }
  delete h;
  return XTD_OK;
}

int xtd_set_stream(xtd_handle h, void* s) {
  XTD_REQUIRE(h, XTD_ERR_ARG, "null handle");
  h->stream = (cudaStream_t)s;
  return XTD_OK;
}

int xtd_set_mo(xtd_handle h, int spin, const double* c_dev, long ld, int nmo) {
  XTD_REQUIRE(h && (spin == 0 || spin == 1) && c_dev && ld >= nmo && nmo > 0, XTD_ERR_ARG, "xtd_set_mo: bad arguments");
  h->C[spin] = c_dev; h->ldC[spin] = ld; h->nmo[spin] = nmo;
  return XTD_OK;
}

int xtd_add_channel(xtd_handle h, int spin_o, const int* occ_idx, int no, int spin_v, const int* vir_idx, int nv, const int* o_blocks,
                    int nob, const int* v_blocks, int nvb) {
  XTD_REQUIRE(h && !h->finalized, XTD_ERR_STATE, "xtd_add_channel after finalize");
  XTD_REQUIRE(h->ch.size() < 2, XTD_ERR_UNSUPPORTED, "at most two channels");
  XTD_REQUIRE(no > 0 && nv > 0 && nob >= 1 && nob <= 2 && nvb >= 1 && nvb <= 2, XTD_ERR_ARG, "xtd_add_channel: bad sizes");
  Channel* c = new Channel();
  c->spin_o = spin_o; c->spin_v = spin_v; c->no = no; c->nv = nv;
  c->occ_idx.assign(occ_idx, occ_idx + no);
  c->vir_idx.assign(vir_idx, vir_idx + nv);
  for (int i = 0; i < nob; ++i) c->o_blocks.push_back({o_blocks[2 * i], o_blocks[2 * i + 1]});
  for (int i = 0; i < nvb; ++i) c->v_blocks.push_back({v_blocks[2 * i], v_blocks[2 * i + 1]});
  for (int i = 1; i < nob; ++i)
    if (c->o_blocks[i].first % 2) { delete c; XTD_SET_ERR("occ block start must be even"); return XTD_ERR_ALIGN; }
  for (int i = 1; i < nvb; ++i)
    if (c->v_blocks[i].first % 2) { delete c; XTD_SET_ERR("vir block start must be even"); return XTD_ERR_ALIGN; }
  for (int i = 0; i < no; ++i)
    if (occ_idx[i] >= h->nmo[spin_o]) { delete c; XTD_SET_ERR("occ index out of range"); return XTD_ERR_ARG; }
  for (int i = 0; i < nv; ++i)
    if (vir_idx[i] >= h->nmo[spin_v]) { delete c; XTD_SET_ERR("vir index out of range"); return XTD_ERR_ARG; }
  c->ldz = pad_ld(nv);
  c->ldzt = pad_ld(no);
  c->ldoo = pad_ld(no);
  c->ldvv = pad_ld(nv);
  int r = build_channel_matrices(h, c);
  if (r != XTD_OK) { delete c; return r; }
  h->ch.push_back(c);
  return (int)h->ch.size() - 1;
}

int xtd_channel_layout(xtd_handle h, int chn, int nvec, long* base, long* vec_stride, long* ld) {
  XTD_REQUIRE(h && chn >= 0 && chn < (int)h->ch.size(), XTD_ERR_ARG, "bad channel");
  long b[2], tot;
  sig_layout(h, nvec, b, &tot);
  if (base) *base = b[chn];
  if (vec_stride) *vec_stride = (long)h->ch[chn]->no * h->ch[chn]->ldz;
  if (ld) *ld = h->ch[chn]->ldz;
  return XTD_OK;
}

int xtd_add_kterm(xtd_handle h, int tensor, int chn, const double* w, int nob, int nvb) {
  XTD_REQUIRE(h && !h->finalized && (tensor == 0 || tensor == 1), XTD_ERR_ARG, "xtd_add_kterm: bad arguments");
  XTD_REQUIRE(chn >= 0 && chn < (int)h->ch.size(), XTD_ERR_ARG, "bad channel");
  Channel* c = h->ch[chn];
  XTD_REQUIRE(nob == (int)c->o_blocks.size() && nvb == (int)c->v_blocks.size(), XTD_ERR_ARG, "weight table shape != channel blocks");
  XTD_REQUIRE(h->naux_filled[tensor] == 0, XTD_ERR_STATE, "exchange terms must be declared before xtd_df_add");
  KTermRec k;
  k.tensor = tensor; k.ch = chn; k.nob = nob; k.nvb = nvb;
  memset(k.w, 0, sizeof(k.w));
  k.uniform = true;
  for (int i = 0; i < nob; ++i)
    for (int a = 0; a < nvb; ++a)
      for (int j = 0; j < nob; ++j)
        for (int b = 0; b < nvb; ++b) {
          k.w[i][a][j][b] = w[((i * nvb + a) * nob + j) * nvb + b];
          if (k.w[i][a][j][b] != w[0]) k.uniform = false;
        }
  h->kterms.push_back(k);
  c->need_k[tensor] = true;
  if (!k.uniform && c->o_blocks.size() > 1) c->need_split[tensor] = true;
  if (!k.uniform && c->v_blocks.size() > 1 && c->v_blocks[1].first <= NARROW_MAX) {
    c->need_narrow[tensor] = true;
    const int v2 = c->v_blocks[1].first, wide = c->nv - v2, q = wide / 128, w = wide - 128 * q;
    if (q >= 1 && w > 0 && w <= NARROW_MAX) { c->tail_start = v2 + 128 * q; c->tail_w = w; }
  }
  return XTD_OK;
}

int xtd_add_kterm_t(xtd_handle h, int tensor, int chn, double weight) {
  XTD_REQUIRE(h && !h->finalized && (tensor == 0 || tensor == 1), XTD_ERR_ARG, "xtd_add_kterm_t: bad arguments");
  XTD_REQUIRE(chn >= 0 && chn < (int)h->ch.size(), XTD_ERR_ARG, "bad channel");
  XTD_REQUIRE(h->naux_filled[tensor] == 0 && h->naux[tensor] == 0, XTD_ERR_STATE, "exchange terms must be declared before xtd_df_begin");
  KTermTRec k;
  k.tensor = tensor; k.ch = chn; k.w = weight;
  h->ktterms.push_back(k);
  h->ch[chn]->need_kt[tensor] = true;
  return XTD_OK;
}

int xtd_add_jblock(xtd_handle h, int chn, int r0, int nr, int c0, int nc) {
  XTD_REQUIRE(h && !h->finalized && chn >= 0 && chn < (int)h->ch.size(), XTD_ERR_ARG, "xtd_add_jblock: bad arguments");
  Channel* c = h->ch[chn];
  XTD_REQUIRE(r0 >= 0 && nr > 0 && r0 + nr <= c->no && c0 >= 0 && nc > 0 && c0 + nc <= c->nv, XTD_ERR_ARG, "J block out of range");
  XTD_REQUIRE(h->naux_filled[0] == 0, XTD_ERR_STATE, "Coulomb blocks must be declared before xtd_df_add");
  JBlockRec* j = new JBlockRec();
  j->ch = chn; j->r0 = r0; j->nr = nr; j->c0 = c0; j->nc = nc; j->ld = pad_ld(nc);
  h->jblocks.push_back(j);
  return (int)h->jblocks.size() - 1;
}

int xtd_set_jmix(xtd_handle h, const double* mix, int n) {
  XTD_REQUIRE(h && n == (int)h->jblocks.size(), XTD_ERR_ARG, "xtd_set_jmix: size != number of J blocks");
  XTD_REQUIRE(!h->finalized, XTD_ERR_STATE, "xtd_set_jmix after finalize (recorded graphs hold the old buffer)");
  h->jmix.assign(mix, mix + (size_t)n * n);
  XTD_TRY(h->jmix_dev.alloc((size_t)n * n, h->stream));
  XTD_CUDA(cudaMemcpyAsync(h->jmix_dev.p, mix, (size_t)n * n * 8, cudaMemcpyHostToDevice, h->stream));
  XTD_CUDA(cudaStreamSynchronize(h->stream));
  return XTD_OK;
}

int xtd_set_exchange_emulation(xtd_handle h, int slices) {
  XTD_REQUIRE(h && !h->finalized, XTD_ERR_STATE, "xtd_set_exchange_emulation after finalize");
  XTD_REQUIRE(slices == 0 || (slices >= OZ_MIN_S && slices <= OZ_MAX_S), XTD_ERR_ARG, "xtd_set_exchange_emulation: slices %d (0 or %d..%d)", slices,
              OZ_MIN_S, OZ_MAX_S);
  XTD_REQUIRE(h->naux_filled[0] == 0 && h->naux_filled[1] == 0, XTD_ERR_STATE, "xtd_set_exchange_emulation must precede xtd_df_add");
  h->oz_slices = slices;
  return XTD_OK;
}

int xtd_set_open_orbitals(xtd_handle h, int spin, const int* open_idx_host, int n_open) {
  XTD_REQUIRE(h && !h->finalized && (spin == 0 || spin == 1) && open_idx_host && n_open >= 1 && n_open <= 64, XTD_ERR_ARG,
              "xtd_set_open_orbitals: bad arguments");
  XTD_REQUIRE(h->C[spin], XTD_ERR_STATE, "xtd_set_mo must precede xtd_set_open_orbitals");
  XTD_REQUIRE(h->naux_filled[0] == 0, XTD_ERR_STATE, "xtd_set_open_orbitals must precede xtd_df_add");
  const int N = h->nao, nmo = h->nmo[spin];
  for (int i = 0; i < n_open; ++i) XTD_REQUIRE(open_idx_host[i] >= 0 && open_idx_host[i] < nmo, XTD_ERR_ARG, "open orbital index out of range");
  cudaStream_t s = h->stream;
  h->kopen_spin = spin; h->n_open = n_open; h->ld_mo = pad_ld(nmo);
  DevBuf cu, call;
  XTD_TRY(cu.alloc((size_t)N * pad_ld(n_open), s));
  XTD_TRY(call.alloc((size_t)N * h->ld_mo, s));
  XTD_TRY(h->CuT.alloc((size_t)n_open * h->ldN, s));
  XTD_TRY(h->CallT.alloc((size_t)nmo * h->ldN, s));
  XTD_TRY(h->kopen.alloc((size_t)nmo * h->ld_mo, s));
  std::vector<int> all(nmo);
  for (int i = 0; i < nmo; ++i) all[i] = i;
  int *d_u = nullptr, *d_all = nullptr;
  XTD_TRY(upload_array(&d_u, open_idx_host, (size_t)n_open, s));
  XTD_TRY(upload_array(&d_all, all.data(), (size_t)nmo, s));
  gather_cols_kernel<<<dim3((unsigned)cdiv(n_open, 128), N), 128, 0, s>>>(cu.p, pad_ld(n_open), h->C[spin], h->ldC[spin], N, d_u, n_open);
  LAUNCH_CHECK();
  gather_cols_kernel<<<dim3((unsigned)cdiv(nmo, 128), N), 128, 0, s>>>(call.p, h->ld_mo, h->C[spin], h->ldC[spin], N, d_all, nmo);
  LAUNCH_CHECK();
  dim3 tb(32, 8);
  transpose_kernel<<<dim3((unsigned)cdiv(n_open, 32), (unsigned)cdiv(N, 32), 1), tb, 0, s>>>(h->CuT.p, h->ldN, 0, cu.p, pad_ld(n_open), 0, N, n_open);
  LAUNCH_CHECK();
  transpose_kernel<<<dim3((unsigned)cdiv(nmo, 32), (unsigned)cdiv(N, 32), 1), tb, 0, s>>>(h->CallT.p, h->ldN, 0, call.p, h->ld_mo, 0, N, nmo);
  LAUNCH_CHECK();
  XTD_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_u);
  cudaFree(d_all);
  return XTD_OK;
}

int xtd_get_kopen(xtd_handle h, double* out_dev, long ld) {
  XTD_REQUIRE(h && out_dev && h->n_open > 0, XTD_ERR_STATE, "xtd_get_kopen: xtd_set_open_orbitals and the tensor come first");
  const int nmo = h->nmo[h->kopen_spin];
  XTD_REQUIRE(ld >= nmo, XTD_ERR_ARG, "xtd_get_kopen: ld < nmo");
  XTD_CUDA(cudaMemcpy2DAsync(out_dev, (size_t)ld * 8, h->kopen.p, (size_t)h->ld_mo * 8, (size_t)nmo * 8, nmo, cudaMemcpyDeviceToDevice, h->stream));
  return XTD_OK;
}

int xtd_df_begin(xtd_handle h, int tensor, long naux_local) {
  XTD_REQUIRE(h && (tensor == 0 || tensor == 1) && naux_local >= 0, XTD_ERR_ARG, "xtd_df_begin: bad arguments");
  h->naux[tensor] = naux_local;
  h->naux_filled[tensor] = 0;
  for (auto* c : h->ch)
    if (c->need_kt[tensor]) XTD_TRY(c->Lov[tensor].alloc((size_t)naux_local * c->no * c->ldz, h->stream));
  for (auto* c : h->ch) {
    if (!oovv_resident(h, c, tensor)) continue;
    XTD_TRY(c->Loo[tensor].alloc((size_t)naux_local * c->no * c->ldoo, h->stream));
    // emulated path: uniform-weight terms, or block-weighted terms whose first virtual block is narrow (it keeps its DMMA pass;
    // the wide second block is emulated with one half-transform per occupied row block).  Mixed term lists stay on DMMA.
    c->use_oz[tensor] = false;
    c->oz_col0[tensor] = 0;
    if (h->oz_slices > 0 && oz_max_group(c->nv, h->oz_slices) >= 1) {
      int n_uni = 0, n_blk = 0;
      for (const KTermRec& k : h->kterms)
        if (k.tensor == tensor && h->ch[k.ch] == c) (k.uniform ? n_uni : n_blk)++;
      if (n_blk == 0) c->use_oz[tensor] = n_uni > 0;
      else if (n_uni == 0) {
        if (c->v_blocks.size() == 1) c->use_oz[tensor] = true;
        else if (c->need_narrow[tensor]) { c->use_oz[tensor] = true; c->oz_col0[tensor] = c->v_blocks[1].first; }
      }
      if (c->use_oz[tensor]) c->tail_w = 0;           // no short-tail pass: the emulated block pads to 64-column tiles anyway
    }
    if (c->use_oz[tensor]) {
      c->ozB.set(c->nv - c->oz_col0[tensor], OZ_BN, c->nv);
      c->oz_group = std::min(4, oz_max_group(c->nv, h->oz_slices));
      if (c->LvvS[tensor]) cudaFree(c->LvvS[tensor]);
      if (c->LvvScale[tensor]) cudaFree(c->LvvScale[tensor]);
      c->LvvS[tensor] = nullptr; c->LvvScale[tensor] = nullptr;
      XTD_CUDA(cudaMalloc((void**)&c->LvvS[tensor], std::max<size_t>(c->ozB.slice_bytes(naux_local, h->oz_slices), 16)));
      XTD_CUDA(cudaMalloc((void**)&c->LvvScale[tensor], std::max<size_t>(c->ozB.scale_doubles(naux_local, c->oz_group), 2) * 8));
      c->Lvv[tensor].release();
      // Packing G aux functions per row tile, padded per group rather than per aux function: the chunks of xtd_df_add and of
      // run_k_emulated start on group boundaries, so no row tile straddles a chunk (config 5: 4 x 277 rows in 9 tiles, against 12)
      c->ozL.set(c->oz_group * c->no, OZ_BM, c->no);
      const long loo_groups = cdiv(naux_local, c->oz_group);
      if (c->LooS[tensor]) cudaFree(c->LooS[tensor]);
      if (c->LooScale[tensor]) cudaFree(c->LooScale[tensor]);
      if (c->LooNorm[tensor]) cudaFree(c->LooNorm[tensor]);
      c->LooS[tensor] = nullptr; c->LooScale[tensor] = c->LooNorm[tensor] = nullptr;
      XTD_CUDA(cudaMalloc((void**)&c->LooS[tensor], std::max<size_t>(c->ozL.slice_bytes(loo_groups, h->oz_slices), 16)));
      XTD_CUDA(cudaMalloc((void**)&c->LooScale[tensor], std::max<size_t>(c->ozL.scale_doubles(loo_groups, 1), 2) * 8));
      XTD_CUDA(cudaMalloc((void**)&c->LooNorm[tensor], std::max<size_t>((size_t)naux_local * c->no, 2) * 8));
    } else {
      XTD_TRY(c->Lvv[tensor].alloc((size_t)naux_local * c->nv * c->ldvv, h->stream));
    }
    if (c->need_narrow[tensor]) XTD_TRY(c->Lvo[tensor].alloc((size_t)naux_local * c->v_blocks[1].first * c->ldvv, h->stream));
    if (c->need_narrow[tensor] && c->tail_w > 0) XTD_TRY(c->Lvt[tensor].alloc((size_t)naux_local * c->tail_w * c->ldvv, h->stream));
    if (c->need_split[tensor]) {
      const int o2 = c->o_blocks[1].first;
      XTD_TRY(c->Loob[tensor][0].alloc((size_t)naux_local * o2 * c->ldoo, h->stream));
      XTD_TRY(c->Loob[tensor][1].alloc((size_t)naux_local * (c->no - o2) * c->ldoo, h->stream));
    }
  }
  if (tensor == 0)
    for (auto* j : h->jblocks) XTD_TRY(j->L.alloc((size_t)naux_local * j->nr * j->ld, h->stream));
  return XTD_OK;
}

int xtd_df_add(xtd_handle h, int tensor, const double* l_dev, long np, long ld_row, long stride_p, int packed) {
  XTD_REQUIRE(h && (tensor == 0 || tensor == 1) && l_dev && np > 0, XTD_ERR_ARG, "xtd_df_add: bad arguments");
  XTD_REQUIRE(h->naux_filled[tensor] + np <= h->naux[tensor], XTD_ERR_ARG, "xtd_df_add: more aux rows than declared (%ld + %ld > %ld)",
              h->naux_filled[tensor], np, h->naux[tensor]);
  const int N = h->nao;
  const long ldN = h->ldN;
  cudaStream_t s = h->stream;
  const bool direct = !packed && (ld_row % 2 == 0) && (stride_p % 2 == 0) && (((uintptr_t)l_dev & 15) == 0);
  // per-aux workspace: staging copy (if needed) + the largest half-transformed block
  int max_n = 0;
  for (auto* c : h->ch) {
    bool need_o = oovv_resident(h, c, tensor) || c->need_kt[tensor];
    if (tensor == 0)
      for (auto* j : h->jblocks) need_o = need_o || (h->ch[j->ch] == c);
    if (need_o) max_n = std::max(max_n, c->no);
    if (oovv_resident(h, c, tensor)) max_n = std::max(max_n, c->nv);
  }
  if (tensor == 0 && h->n_open > 0) max_n = std::max(max_n, 1);
  if (max_n == 0) { h->naux_filled[tensor] += np; return XTD_OK; }
  h->arena.used = 0;
  size_t split_bytes = std::min<size_t>(h->arena.cap / 4, (size_t)1 << 30);
  h->gemm.split_ws = h->arena.take(split_bytes / 8);
  h->gemm.split_ws_bytes = split_bytes;
  size_t oz_tmp = 0;       // emulated path: the fp64 Lvv chunk is a temporary that is cut into int8 slices
  long oz_align = 1;
  for (auto* c : h->ch)
    if (c->use_oz[tensor]) {
      oz_tmp = std::max(oz_tmp, (size_t)c->nv * c->ldvv);
      oz_align = std::max<long>(oz_align, c->oz_group);
    }
  if (oz_tmp) {
    const bool last = h->naux_filled[tensor] + np == h->naux[tensor];
    XTD_REQUIRE(h->naux_filled[tensor] % oz_align == 0 && (np % oz_align == 0 || last), XTD_ERR_ARG,
                "xtd_df_add: with the INT8-emulated exchange contraction every chunk but the last must hold a multiple of %ld aux functions",
                oz_align);
  }
  const size_t ko_tmp = (tensor == 0 && h->n_open > 0) ? (size_t)h->n_open * (ldN + h->ld_mo) : 0;   // Hu + Lu of K[D_open]
  const size_t per_p = ((size_t)(direct ? 0 : N) + (size_t)max_n) * ldN + oz_tmp + ko_tmp;
  long pc = (long)(h->arena.left() / 8 / per_p);
  XTD_REQUIRE(pc >= oz_align, XTD_ERR_NOMEM, "xtd_df_add: workspace too small for %ld aux functions (%zu doubles each)", oz_align, per_p);
  pc = std::min<long>(pc, np);
  if (pc < np) pc = pc / oz_align * oz_align;
  double* stage = direct ? nullptr : h->arena.take((size_t)pc * N * ldN);
  double* half = h->arena.take((size_t)pc * max_n * ldN);
  double* lvv_tmp = oz_tmp ? h->arena.take((size_t)pc * oz_tmp) : nullptr;
  double* ko_buf = ko_tmp ? h->arena.take((size_t)pc * ko_tmp) : nullptr;
  XTD_REQUIRE(half && (direct || stage) && (!oz_tmp || lvv_tmp) && (!ko_tmp || ko_buf), XTD_ERR_NOMEM, "xtd_df_add: workspace exhausted");

  for (long p0 = 0; p0 < np; p0 += pc) {
    const int pn = (int)std::min<long>(pc, np - p0);
    const long P0 = h->naux_filled[tensor] + p0;
    MatView Lv;
    if (direct) {
      Lv = view3d(l_dev + p0 * stride_p, ld_row, stride_p, pn, N, N);
    } else {
      if (packed) {
        unpack_tril_kernel<<<dim3((unsigned)cdiv(N, 128), N, pn), 128, 0, s>>>(stage, ldN, (long)N * ldN, l_dev + p0 * stride_p, stride_p, N);
      } else {
        pad_copy_kernel<<<dim3((unsigned)cdiv(N, 128), N, pn), 128, 0, s>>>(stage, ldN, (long)N * ldN, l_dev + p0 * stride_p, ld_row,
                                                                            stride_p, N, N);
      }
      LAUNCH_CHECK();
      Lv = view3d(stage, ldN, (long)N * ldN, pn, N, N);
    }
    if (ko_buf) {
      // K[D_open][p][q] += sum_P sum_u L^P_pu L^P_qu:  Hu[P][u][mu] = sum_nu CuT[u][nu] L[P][mu][nu],  Lu[P][u][q] = sum_mu Hu C[mu][q]
      const int nu_ = h->n_open, nmo = h->nmo[h->kopen_spin];
      double* Hu = ko_buf;
      double* Lu = ko_buf + (size_t)pc * nu_ * ldN;
      GemmDesc d;
      d.A = view2d(h->CuT.p, ldN, nu_, N); d.B = Lv; d.M = nu_; d.N = N; d.K = N;
      d.batches = pn; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
      d.C = Hu; d.ldc = ldN; d.c_batch_stride = (long)nu_ * ldN;
      XTD_TRY(gemm(h->gemm, d, s));
      GemmDesc e;
      e.A = view3d(Hu, ldN, (long)nu_ * ldN, pn, nu_, N); e.B = view2d(h->CallT.p, ldN, nmo, N);
      e.M = nu_; e.N = nmo; e.K = N; e.batches = pn; e.a_hi = 1; e.b_hi = 0;
      e.C = Lu; e.ldc = h->ld_mo; e.c_batch_stride = (long)nu_ * h->ld_mo;
      XTD_TRY(gemm(h->gemm, e, s));
      GemmDesc f;
      f.a_kc = false; f.b_kc = false;
      f.A = view2d(Lu, h->ld_mo, pn * nu_, nmo); f.B = view2d(Lu, h->ld_mo, pn * nu_, nmo);
      f.M = nmo; f.N = nmo; f.K = pn * nu_;
      f.C = h->kopen.p; f.ldc = h->ld_mo; f.accumulate = true;
      XTD_TRY(gemm(h->gemm, f, s));
    }
    for (size_t ci = 0; ci < h->ch.size(); ++ci) {
      Channel* c = h->ch[ci];
      bool need_o = oovv_resident(h, c, tensor) || c->need_kt[tensor];
      if (tensor == 0)
        for (auto* j : h->jblocks) need_o = need_o || (j->ch == (int)ci);
      if (need_o) {
        // HoT[P][i][mu] = sum_nu CoT[i][nu] L[P][mu][nu]
        GemmDesc d;
        d.A = view2d(c->CoT.p, ldN, c->no, N); d.B = Lv; d.M = c->no; d.N = N; d.K = N;
        d.batches = pn; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
        d.C = half; d.ldc = ldN; d.c_batch_stride = (long)c->no * ldN;
        XTD_TRY(gemm(h->gemm, d, s));
        MatView Hv = view3d(half, ldN, (long)c->no * ldN, pn, c->no, N);
        if (oovv_resident(h, c, tensor)) {
          // Loo[P][i][j] = sum_mu HoT[P][i][mu] CoT[j][mu]
          GemmDesc e;
          e.A = Hv; e.B = view2d(c->CoT.p, ldN, c->no, N); e.M = c->no; e.N = c->no; e.K = N;
          e.batches = pn; e.a_hi = 1; e.b_hi = 0;
          e.C = c->Loo[tensor].p + P0 * c->no * c->ldoo; e.ldc = c->ldoo; e.c_batch_stride = (long)c->no * c->ldoo;
          XTD_TRY(gemm(h->gemm, e, s));
          if (c->use_oz[tensor]) {
            // A operand of the fused half-transform: one q-slice per group of oz_group aux functions (P0 is a group boundary), rows
            // (P, i) packed, one scale per (aux function, row)
            const int G = c->oz_group;
            XTD_REQUIRE(P0 % G == 0, XTD_ERR_ARG, "xtd_df_add: aux chunk at %ld does not start a group of %d", P0, G);
            const double* lc = c->Loo[tensor].p + P0 * c->no * c->ldoo;
            OzRowPack pk;
            pk.G = G; pk.o2 = c->oz_row_split(); pk.no = c->no; pk.np = pn; pk.sp = (long)c->no * c->ldoo;
            XTD_TRY(oz_slice(h->oz_slices, c->LooS[tensor] + c->ozL.slice_bytes(P0 / G, h->oz_slices), c->LooScale[tensor] + (size_t)(P0 / G) * c->ozL.rows_pad,
                             c->ozL, lc, c->ldoo, (long)G * c->no * c->ldoo, (int)cdiv(pn, G), 1, s, false, 0, pk));
            oz_rownorm_kernel<<<dim3(c->no, pn), 128, 0, s>>>(c->LooNorm[tensor] + (size_t)P0 * c->no, c->no, lc, c->ldoo, (long)c->no * c->ldoo, c->no,
                                                              c->no);
            LAUNCH_CHECK();
          }
          if (c->need_split[tensor]) {
            const int o2 = c->o_blocks[1].first;
            const int r0s[2] = {0, o2}, nrs[2] = {o2, c->no - o2};
            for (int ib = 0; ib < 2; ++ib) {
              GemmDesc f = e;
              f.A = view3d(half, ldN, (long)c->no * ldN, pn, nrs[ib], N, r0s[ib], 0);
              f.M = nrs[ib];
              f.C = c->Loob[tensor][ib].p + P0 * nrs[ib] * c->ldoo; f.c_batch_stride = (long)nrs[ib] * c->ldoo;
              XTD_TRY(gemm(h->gemm, f, s));
            }
          }
        }
        if (c->need_kt[tensor]) {
          // Lov[P][i][a] = sum_mu HoT[P][i][mu] CvT[a][mu]
          GemmDesc e;
          e.A = Hv; e.B = view2d(c->CvT.p, ldN, c->nv, N);
          e.M = c->no; e.N = c->nv; e.K = N; e.batches = pn; e.a_hi = 1; e.b_hi = 0;
          e.C = c->Lov[tensor].p + P0 * c->no * c->ldz; e.ldc = c->ldz; e.c_batch_stride = (long)c->no * c->ldz;
          XTD_TRY(gemm(h->gemm, e, s));
        }
        if (tensor == 0)
          for (auto* j : h->jblocks) {
            if (j->ch != (int)ci) continue;
            // Ljb[P][i][a] = sum_mu HoT[P][r0+i][mu] CvT[c0+a][mu]
            GemmDesc e;
            e.A = view3d(half, ldN, (long)c->no * ldN, pn, j->nr, N, j->r0, 0);
            e.B = view2d(c->CvT.p, ldN, j->nc, N, j->c0, 0);
            e.M = j->nr; e.N = j->nc; e.K = N; e.batches = pn; e.a_hi = 1; e.b_hi = 0;
            e.C = j->L.p + P0 * j->nr * j->ld; e.ldc = j->ld; e.c_batch_stride = (long)j->nr * j->ld;
            XTD_TRY(gemm(h->gemm, e, s));
          }
      }
      if (oovv_resident(h, c, tensor)) {
        // HvT[P][a][mu] = sum_nu CvT[a][nu] L[P][mu][nu] ;  Lvv[P][a][b] = sum_mu HvT[P][a][mu] CvT[b][mu]
        GemmDesc d;
        d.A = view2d(c->CvT.p, ldN, c->nv, N); d.B = Lv; d.M = c->nv; d.N = N; d.K = N;
        d.batches = pn; d.a_hi = 0; d.b_hi = 1;
        d.C = half; d.ldc = ldN; d.c_batch_stride = (long)c->nv * ldN;
        XTD_TRY(gemm(h->gemm, d, s));
        GemmDesc e;
        e.A = view3d(half, ldN, (long)c->nv * ldN, pn, c->nv, N); e.B = view2d(c->CvT.p, ldN, c->nv, N);
        e.M = c->nv; e.N = c->nv; e.K = N; e.batches = pn; e.a_hi = 1; e.b_hi = 0;
        e.C = c->use_oz[tensor] ? lvv_tmp : c->Lvv[tensor].p + P0 * c->nv * c->ldvv;
        e.ldc = c->ldvv; e.c_batch_stride = (long)c->nv * c->ldvv;
        XTD_TRY(gemm(h->gemm, e, s));
        if (c->use_oz[tensor])
          XTD_TRY(oz_slice(h->oz_slices, c->LvvS[tensor] + c->ozB.slice_bytes(P0, h->oz_slices),
                           c->LvvScale[tensor] + (size_t)(P0 / c->oz_group) * c->ozB.rows_pad, c->ozB,
                           lvv_tmp + (long)c->oz_col0[tensor] * c->ldvv, c->ldvv, (long)c->nv * c->ldvv, pn, c->oz_group, s));
        if (c->need_narrow[tensor]) {
          const size_t v2 = (size_t)c->v_blocks[1].first;
          const double* lsrc = c->use_oz[tensor] ? lvv_tmp : c->Lvv[tensor].p + P0 * c->nv * c->ldvv;     // this chunk's [pn][nv][ldvv]
          XTD_CUDA(cudaMemcpy2DAsync(c->Lvo[tensor].p + P0 * v2 * c->ldvv, v2 * c->ldvv * 8, lsrc, (size_t)c->nv * c->ldvv * 8,
                                     v2 * c->ldvv * 8, pn, cudaMemcpyDeviceToDevice, s));
          if (c->tail_w > 0) {
            const size_t tw = (size_t)c->tail_w;
            XTD_CUDA(cudaMemcpy2DAsync(c->Lvt[tensor].p + P0 * tw * c->ldvv, tw * c->ldvv * 8, lsrc + (size_t)c->tail_start * c->ldvv,
                                       (size_t)c->nv * c->ldvv * 8, tw * c->ldvv * 8, pn, cudaMemcpyDeviceToDevice, s));
          }
        }
      }
    }
  }
  h->naux_filled[tensor] += np;
  XTD_CUDA(cudaStreamSynchronize(s));   // the caller may free / overwrite its chunk
  return XTD_OK;
}

int xtd_jblock_diag(xtd_handle h, int jb, double* out_dev) {
  XTD_REQUIRE(h && jb >= 0 && jb < (int)h->jblocks.size() && out_dev, XTD_ERR_ARG, "xtd_jblock_diag: bad arguments");
  JBlockRec* j = h->jblocks[jb];
  jblock_diag_kernel<<<grid1d((long)j->nr * j->nc, 256), 256, 0, h->stream>>>(out_dev, j->L.p, j->ld, (long)j->nr * j->ld, h->naux[0], j->nr,
                                                                             j->nc, 0);
  LAUNCH_CHECK();
  return XTD_OK;
}

int xtd_set_grid(xtd_handle h, const double* ao_dev, int nvar, long ng, long ld_row, long stride_comp, const double* w_dev) {
  XTD_REQUIRE(h && !h->finalized && !h->grid_committed, XTD_ERR_STATE, "xtd_set_grid after commit / finalize");
  XTD_REQUIRE(ao_dev && w_dev && (nvar == 1 || nvar == 4) && ng >= 0 && ld_row >= h->nao, XTD_ERR_ARG, "xtd_set_grid: bad arguments");
  XTD_REQUIRE(ld_row % 2 == 0 && stride_comp % 2 == 0 && ((uintptr_t)ao_dev & 15) == 0, XTD_ERR_ALIGN,
              "xtd_set_grid: ao needs even ld_row / stride_comp and a 16-byte aligned base (pad with xtd helpers)");
  h->ao = ao_dev; h->nvar = nvar; h->ng = ng; h->ao_ld = ld_row; h->ao_comp = stride_comp; h->wgrid = w_dev;
  return XTD_OK;
}

int xtd_set_fxc(xtd_handle h, int kind, const double* fxc_dev) {
  XTD_REQUIRE(h && !h->finalized && !h->grid_committed, XTD_ERR_STATE, "xtd_set_fxc after commit / finalize");
  XTD_REQUIRE(kind >= XTD_FXC_NONE && kind <= XTD_FXC_MCOL_TAU && (kind == XTD_FXC_NONE || fxc_dev), XTD_ERR_ARG, "xtd_set_fxc: bad arguments");
  h->tau = (kind == XTD_FXC_UKS_TAU || kind == XTD_FXC_MCOL_TAU);
  if (h->tau) XTD_REQUIRE(h->ao == nullptr || h->nvar == 4, XTD_ERR_ARG, "meta-GGA kernels need value + gradient AO components (nvar = 4)");
  h->fxc_kind = kind == XTD_FXC_UKS_TAU ? XTD_FXC_UKS : (kind == XTD_FXC_MCOL_TAU ? XTD_FXC_MCOL : kind);
  h->fxc = fxc_dev;
  return XTD_OK;
}

int xtd_grid_commit(xtd_handle h) {
  XTD_REQUIRE(h && !h->finalized, XTD_ERR_STATE, "xtd_grid_commit after finalize");
  if (h->fxc_kind == XTD_FXC_NONE || h->grid_committed) return XTD_OK;
  return grid_commit(h);
}

int xtd_add_local_gemm(xtd_handle h, int side, int dch, int r0, int nr, int c0, int nc, int sch, int sr0, int sc0, const double* mat,
                       int mrows, int mcols, double alpha) {
  XTD_REQUIRE(h && !h->finalized && mat, XTD_ERR_ARG, "xtd_add_local_gemm: bad arguments");
  XTD_REQUIRE(dch >= 0 && dch < (int)h->ch.size() && sch >= 0 && sch < (int)h->ch.size(), XTD_ERR_ARG, "bad channel");
  Channel *dc = h->ch[dch], *sc = h->ch[sch];
  XTD_REQUIRE(r0 >= 0 && r0 + nr <= dc->no && c0 >= 0 && c0 + nc <= dc->nv, XTD_ERR_ARG, "local gemm: destination out of range");
  XTD_REQUIRE(c0 % 2 == 0 && sc0 % 2 == 0, XTD_ERR_ALIGN, "local gemm: column offsets must be even");
  if (side == XTD_SIDE_RIGHT) {
    XTD_REQUIRE(mcols == nc && sr0 + nr <= sc->no && sc0 + mrows <= sc->nv, XTD_ERR_ARG, "right gemm: shapes inconsistent");
  } else if (side == XTD_SIDE_LEFT) {
    XTD_REQUIRE(mrows == nr && sr0 + mcols <= sc->no && sc0 + nc <= sc->nv, XTD_ERR_ARG, "left gemm: shapes inconsistent");
  } else if (side == XTD_SIDE_LEFT_T) {      // dst[r][c] += alpha sum_k M[r][k] src[sr0 + c][sc0 + k]
    XTD_REQUIRE(mrows == nr && sr0 + nc <= sc->no && sc0 + mcols <= sc->nv, XTD_ERR_ARG, "transposed left gemm: shapes inconsistent");
  } else {                                   // dst[r][c] += alpha sum_j src[sr0 + j][sc0 + r] M[j][c]
    XTD_REQUIRE(side == XTD_SIDE_RIGHT_T && mcols == nc && sr0 + mrows <= sc->no && sc0 + nr <= sc->nv, XTD_ERR_ARG,
                "transposed right gemm: shapes inconsistent");
  }
  LocalGemmRec* l = new LocalGemmRec();
  l->side = side; l->dch = dch; l->r0 = r0; l->nr = nr; l->c0 = c0; l->nc = nc; l->sch = sch; l->sr0 = sr0; l->sc0 = sc0;
  l->mrows = mrows; l->mcols = mcols; l->alpha = alpha;
  int r = upload_padded(l->M, l->ldm, mat, mrows, mcols, h->stream);
  if (r != XTD_OK) { delete l; return r; }
  h->lgemms.push_back(l);
  return XTD_OK;
}

int xtd_add_rank1(xtd_handle h, int dch, const double* u, int sch, const double* v) {
  XTD_REQUIRE(h && !h->finalized && u && v && dch >= 0 && dch < (int)h->ch.size() && sch >= 0 && sch < (int)h->ch.size(), XTD_ERR_ARG,
              "xtd_add_rank1: bad arguments");
  Rank1Rec* r = new Rank1Rec();
  r->dch = dch; r->sch = sch;
  long ld;
  XTD_TRY(upload_padded(r->U, ld, u, h->ch[dch]->no, h->ch[dch]->nv, h->stream));
  XTD_TRY(upload_padded(r->V, ld, v, h->ch[sch]->no, h->ch[sch]->nv, h->stream));
  h->rank1s.push_back(r);
  return XTD_OK;
}

int xtd_add_diag(xtd_handle h, int chn, const double* d_host) {
  XTD_REQUIRE(h && !h->finalized && d_host && chn >= 0 && chn < (int)h->ch.size(), XTD_ERR_ARG, "xtd_add_diag: bad arguments");
  DiagRec* d = new DiagRec();
  d->ch = chn;
  long ld;
  XTD_TRY(upload_padded(d->D, ld, d_host, h->ch[chn]->no, h->ch[chn]->nv, h->stream));
  h->diags.push_back(d);
  return XTD_OK;
}

int xtd_set_gather(xtd_handle h, int chn, const long* indptr, const long* cols, const double* vals, long nnz) {
  XTD_REQUIRE(h && chn >= 0 && chn < (int)h->ch.size() && indptr && nnz >= 0, XTD_ERR_ARG, "xtd_set_gather: bad arguments");
  XTD_REQUIRE(!h->finalized, XTD_ERR_STATE, "xtd_set_gather after finalize (recorded graphs hold the old map)");
  Channel* c = h->ch[chn];
  XTD_TRY(upload_array(&c->g_indptr, indptr, (size_t)c->no * c->nv + 1, h->stream));
  XTD_TRY(upload_array(&c->g_cols, cols, (size_t)nnz, h->stream));
  XTD_TRY(upload_array(&c->g_vals, vals, (size_t)nnz, h->stream));
  c->g_nnz = nnz;
  return XTD_OK;
}

int xtd_set_scatter(xtd_handle h, long ext_dim, const long* indptr, const long* offs, const signed char* chans, const double* vals,
                    long nnz) {
  XTD_REQUIRE(h && ext_dim > 0 && indptr && nnz >= 0, XTD_ERR_ARG, "xtd_set_scatter: bad arguments");
  XTD_REQUIRE(!h->finalized, XTD_ERR_STATE, "xtd_set_scatter after finalize (recorded graphs hold the old map)");
  h->ext_dim = ext_dim;
  XTD_TRY(upload_array(&h->s_indptr, indptr, (size_t)ext_dim + 1, h->stream));
  XTD_TRY(upload_array(&h->s_offs, offs, (size_t)nnz, h->stream));
  XTD_TRY(upload_array(&h->s_chans, chans, (size_t)nnz, h->stream));
  XTD_TRY(upload_array(&h->s_vals, vals, (size_t)nnz, h->stream));
  return XTD_OK;
}

int xtd_finalize(xtd_handle h, int max_nvec) {
  XTD_REQUIRE(h && max_nvec >= 1, XTD_ERR_ARG, "xtd_finalize: bad arguments");
  XTD_REQUIRE(!h->ch.empty() && h->ext_dim > 0, XTD_ERR_STATE, "xtd_finalize: channels and layout maps are required");
  for (auto* c : h->ch) XTD_REQUIRE(c->g_indptr, XTD_ERR_STATE, "xtd_finalize: gather map missing");
  for (int t = 0; t < 2; ++t)
    XTD_REQUIRE(h->naux_filled[t] == h->naux[t], XTD_ERR_STATE, "xtd_finalize: DF tensor %d incomplete (%ld of %ld)", t,
                h->naux_filled[t], h->naux[t]);
  if (!h->jblocks.empty()) XTD_REQUIRE(h->jmix.size() == h->jblocks.size() * h->jblocks.size(), XTD_ERR_STATE, "xtd_finalize: J mix missing");
  cudaStream_t s = h->stream;
  h->max_nvec = max_nvec;
  const bool xc = (h->fxc_kind != XTD_FXC_NONE) && h->ng > 0;
  if (h->fxc_kind != XTD_FXC_NONE) XTD_REQUIRE(h->ao || h->grid_committed, XTD_ERR_STATE, "xtd_finalize: kernel set but no grid");
  if (xc && !h->grid_committed) XTD_TRY(grid_commit(h));
  XTD_CUDA(cudaStreamSynchronize(s));
  // check that the fixed per-call buffers for max_nvec fit in the arena with room for a work chunk
  size_t fixed = 0;
  for (auto* c : h->ch) {
    fixed += (size_t)max_nvec * c->no * c->ldz * 2;              // Z, SIG
    fixed += (size_t)max_nvec * c->nv * c->ldzt * 2;             // ZT, ZTs
  }
  XTD_REQUIRE(fixed * 8 + (32u << 20) < h->arena.cap, XTD_ERR_NOMEM, "xtd_finalize: workspace of %zu bytes too small for %d vectors (%zu fixed)",
              h->arena.cap, max_nvec, fixed * 8);
  // small problems: the local GEMM and diagonal terms become one launch
  long max_elems = 0;
  for (auto* c : h->ch) max_elems = std::max<long>(max_elems, (long)c->no * c->nv);
  h->small_local = max_elems <= 16384;
  if (h->small_local && (!h->lgemms.empty() || !h->diags.empty())) {
    std::vector<LocalTermDev> lt, ld;
    for (auto* l : h->lgemms) {
      LocalTermDev t;
      t.side = l->side; t.dch = l->dch; t.r0 = l->r0; t.nr = l->nr; t.c0 = l->c0; t.nc = l->nc;
      t.sch = l->sch; t.sr0 = l->sr0; t.sc0 = l->sc0;
      t.k = (l->side == XTD_SIDE_RIGHT || l->side == XTD_SIDE_RIGHT_T) ? l->mrows : l->mcols;
      t.ldm = l->ldm; t.alpha = l->alpha; t.M = l->M.p;
      lt.push_back(t);
    }
    for (auto* d : h->diags) {
      LocalTermDev t = {};
      t.dch = d->ch; t.M = d->D.p;
      ld.push_back(t);
    }
    XTD_TRY(upload_array(&h->lt_dev, lt.data(), lt.size(), s));
    XTD_TRY(upload_array(&h->ld_dev, ld.data(), ld.size(), s));
  }
  h->finalized = true;
  return XTD_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// sigma
// ---------------------------------------------------------------------------------------------------------
static int setup_call_buffers(xtd_engine* h, int nvec) {
  h->arena.used = 0;
  long base[2], total;
  sig_layout(h, nvec, base, &total);
  h->SIG = h->arena.take((size_t)total);
  double* zall = h->arena.take((size_t)total);
  XTD_REQUIRE(h->SIG && zall, XTD_ERR_NOMEM, "workspace exhausted (sigma buffers)");
  for (size_t c = 0; c < h->ch.size(); ++c) {
    Channel* ch = h->ch[c];
    h->sig_base[c] = base[c];
    h->Z[c] = zall + base[c];
    h->ZT[c] = h->arena.take((size_t)nvec * ch->nv * ch->ldzt);
    h->ZTs[c] = h->arena.take((size_t)nvec * ch->nv * ch->ldzt);
    XTD_REQUIRE(h->ZT[c] && h->ZTs[c], XTD_ERR_NOMEM, "workspace exhausted (transposed trial vectors)");
  }
  const size_t njb = h->jblocks.size();
  if (njb) {
    h->jR = h->arena.take((size_t)nvec * njb * (std::max<long>(h->naux[0], 1) + 1));
    h->jRm = h->arena.take((size_t)nvec * njb * (std::max<long>(h->naux[0], 1) + 1));
    XTD_REQUIRE(h->jR && h->jRm, XTD_ERR_NOMEM, "workspace exhausted (Coulomb vectors)");
  }
  h->r1d = h->arena.take((size_t)nvec + 8);
  size_t split_bytes = std::min<size_t>(h->arena.left() / 4, (size_t)1 << 30);
  h->gemm.split_ws = h->arena.take(split_bytes / 8);
  h->gemm.split_ws_bytes = split_bytes;
  h->scratch_doubles = h->arena.left() / 8 - 64;
  h->scratch = h->arena.take(h->scratch_doubles);
  XTD_REQUIRE(h->scratch && h->scratch_doubles > (1u << 20), XTD_ERR_NOMEM, "workspace exhausted (chunk scratch)");
  h->cur_nvec = nvec;
  return XTD_OK;
}

template <int NVAR, int KIND, bool TAU = false>
static void launch_xc(const XcArgs& a, cudaStream_t s) {
  // vectors per pass: 4 for one AO component, 2 for value + gradient (register budget); 16-byte accesses when every
  // (vector, component) row segment is 16-byte aligned, i.e. all occupied counts are even
  constexpr int XU = NVAR == 1 ? 4 : 2;
  const bool even = (a.no[0] % 2 == 0) && (a.nch == 1 || a.no[1] % 2 == 0);
  const unsigned grid = (unsigned)cdiv(a.gb, 8);
  if (even) xc_weight_kernel<NVAR, KIND, XU, 2, TAU><<<grid, 256, 0, s>>>(a);
  else xc_weight_kernel<NVAR, KIND, XU, 1, TAU><<<grid, 256, 0, s>>>(a);
}


template <int KIND>
static int launch_xc_split(const XcArgs2& a, cudaStream_t s) {
  const bool even = (a.no[0] % 2 == 0) && (a.nch == 1 || a.no[1] % 2 == 0);
  const size_t smem = (size_t)xc_split_smem_doubles(a.nch, a.no, a.nv) * 8;
  // warps = trial vectors, in as few equal rounds as 16 warps allow
  const int rounds = (int)cdiv(a.nvec, 16);
  const int nwarps = (int)cdiv(a.nvec, rounds);
  static bool attr_set_dev[64] = {false};      // the shared-memory opt-in is per device
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  bool& attr_set = attr_set_dev[dev & 63];
  if (!attr_set) {
    XTD_CUDA(cudaFuncSetAttribute(xc_weight_split_kernel<XC_KIND_UKS, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SPLIT_SMEM_MAX));
    XTD_CUDA(cudaFuncSetAttribute(xc_weight_split_kernel<XC_KIND_UKS, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SPLIT_SMEM_MAX));
    XTD_CUDA(cudaFuncSetAttribute(xc_weight_split_kernel<XC_KIND_MCOL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SPLIT_SMEM_MAX));
    XTD_CUDA(cudaFuncSetAttribute(xc_weight_split_kernel<XC_KIND_MCOL, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SPLIT_SMEM_MAX));
    attr_set = true;
  }
  // few trial vectors: the warps of a CTA share the point by orbital range (xc_weight_split_op_kernel)
  if (a.nvec <= XC_OP_MAX_NVEC) {
    constexpr int NRK = (KIND == XC_KIND_UKS ? 2 : 1) * 4;
    static bool op_attr_dev[64] = {false};
    bool& op_set = op_attr_dev[dev & 63];
    if (!op_set) {
#define XTD_OP_ATTR(K, W_, XB_) \
  XTD_CUDA(cudaFuncSetAttribute(xc_weight_split_op_kernel<K, W_, XB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SPLIT_SMEM_MAX + 2 * 8 * 4 * 8 * 8))
      XTD_OP_ATTR(XC_KIND_UKS, 1, 1); XTD_OP_ATTR(XC_KIND_UKS, 2, 1); XTD_OP_ATTR(XC_KIND_UKS, 1, 2); XTD_OP_ATTR(XC_KIND_UKS, 2, 2);
      XTD_OP_ATTR(XC_KIND_UKS, 1, 4); XTD_OP_ATTR(XC_KIND_UKS, 2, 4);
      XTD_OP_ATTR(XC_KIND_MCOL, 1, 1); XTD_OP_ATTR(XC_KIND_MCOL, 2, 1); XTD_OP_ATTR(XC_KIND_MCOL, 1, 2); XTD_OP_ATTR(XC_KIND_MCOL, 2, 2);
      XTD_OP_ATTR(XC_KIND_MCOL, 1, 4); XTD_OP_ATTR(XC_KIND_MCOL, 2, 4);
#undef XTD_OP_ATTR
      op_set = true;
    }
    const int xb = a.nvec == 1 ? 1 : (a.nvec == 2 ? 2 : 4);
    const size_t smem_op = smem + (size_t)2 * 8 * xb * NRK * 8;
#define XTD_OP_LAUNCH(W_, XB_) xc_weight_split_op_kernel<KIND, W_, XB_><<<(unsigned)a.gb, 256, smem_op, s>>>(a)
    if (even) { if (xb == 1) XTD_OP_LAUNCH(2, 1); else if (xb == 2) XTD_OP_LAUNCH(2, 2); else XTD_OP_LAUNCH(2, 4); }
    else { if (xb == 1) XTD_OP_LAUNCH(1, 1); else if (xb == 2) XTD_OP_LAUNCH(1, 2); else XTD_OP_LAUNCH(1, 4); }
#undef XTD_OP_LAUNCH
    return XTD_OK;
  }
  if (even) xc_weight_split_kernel<KIND, 2><<<(unsigned)a.gb, 32 * nwarps, smem, s>>>(a);
  else xc_weight_split_kernel<KIND, 1><<<(unsigned)a.gb, 32 * nwarps, smem, s>>>(a);
  return XTD_OK;
}

// Value + gradient kernels: GEMM work (in padded 128-row tiles x contraction length, per grid point) of the
// four-component form against the split-gradient form; the latter halves it unless an orbital block barely exceeds
// a tile or the problem is tiny.
static bool xc_use_split(const xtd_engine* h, int nvec) {
  if (h->nvar_eff != 4 || h->tau) return false;      // tau needs the gradient of both orbitals: four-component form
  if (!h->ch.empty() && h->ch[0]->xc_oz_split) return true;     // the emulated grid path always takes the split-gradient form
  {
    int no[2] = {0, 0}, nv[2] = {0, 0};
    for (size_t c = 0; c < h->ch.size(); ++c) { no[c] = h->ch[c]->no; nv[c] = h->ch[c]->nv; }
    if (xc_split_smem_doubles((int)h->ch.size(), no, nv) * 8 > XC_SPLIT_SMEM_MAX) return false;   // MO values of a point must fit shared memory
  }
  if (h->env.xc_split >= 0) return h->env.xc_split != 0;
  auto tile = [](long n) { return (double)(cdiv(n, 128) * 128); };
  double four = 0.0, split = 0.0;
  for (auto* c : h->ch) {
    four += 8.0 * tile((long)nvec * c->no) * c->nv;
    split += 2.0 * tile((long)nvec * c->no) * c->nv + (double)nvec * (tile(c->nv) * pad_ld(c->no) + tile(c->no) * c->nv);
  }
  return split < 0.9 * four;
}

// Grid path with both GEMMs emulated on the INT8 tensor cores (one AO component: ALDA0 and LDA kernels):
//   forward   Y[g][(x,o)] = sum_v phiv[g][v] Z[(x,o)][v]          A = int8 planes of phiv (static), B = planes of Z (per call)
//   weighting xc_weight_kernel in place (unchanged)
//   backward  SIG[(x,o)][v] += sum_g A[g][(x,o)] phiv[g][v]        contraction over grid points: both operands sliced from
//             their transposed sources, q-slices = blocks of OZ_XC_KQ points, one power-of-two scale per (row, block)
static int run_xc_emulated(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  const int nch = (int)h->ch.size();
  const int S = h->oz_slices;
  OzShape shZ[2], shA[2];
  size_t per_g = 0, fixed = 0, w_doubles = 0;
  int splits_max = 8;
  for (int c = 0; c < nch; ++c) {
    Channel* ch = h->ch[c];
    shZ[c].set(nvec * ch->no, OZ_BN, ch->nv);
    shA[c].set(nvec * ch->no, OZ_BM, OZ_XC_KQ);
    per_g += (size_t)shZ[c].rows_pad + (size_t)shA[c].rows_pad * S / 8 + 1;
    fixed += shZ[c].slice_bytes(1, S) / 8 + shZ[c].rows_pad + 64;
    fixed += (size_t)(65536 / OZ_XC_KQ) * shA[c].rows_pad + 64;
    w_doubles = std::max(w_doubles, (size_t)splits_max * shA[c].rows_pad * ch->ozPB.rows_pad);
  }
  fixed += w_doubles + 4096;
  XTD_REQUIRE(h->scratch_doubles > fixed + per_g * OZ_XC_KQ, XTD_ERR_NOMEM, "workspace too small for one block of the emulated grid path");
  long GB = (long)((h->scratch_doubles - fixed) / per_g);
  GB = std::min<long>(GB, 1 << 16);
  if (h->env.max_gb > 0) GB = std::min<long>(GB, std::max<long>(h->env.max_gb, OZ_XC_KQ));
  GB = GB / OZ_XC_KQ * OZ_XC_KQ;
  h->last_grid_chunks = cdiv(h->ng, GB);
  // carve the scratch region
  double* cur = h->scratch;
  auto take = [&](size_t n) { double* p = cur; cur += (n + 31) & ~(size_t)31; return p; };
  double* W = take(w_doubles);
  int8_t* zS[2]; double* zsc[2]; double* Y[2]; int8_t* aS[2]; double* asc[2];
  const long gbmax = std::min<long>(GB, round_up(h->ng, 128));
  for (int c = 0; c < nch; ++c) {
    zS[c] = reinterpret_cast<int8_t*>(take(shZ[c].slice_bytes(1, S) / 8));
    zsc[c] = take(shZ[c].rows_pad);
    Y[c] = take((size_t)gbmax * shZ[c].rows_pad);
    aS[c] = reinterpret_cast<int8_t*>(take((size_t)cdiv(gbmax, OZ_XC_KQ) * shA[c].slice_bytes(1, S) / 8));
    asc[c] = take((size_t)cdiv(gbmax, OZ_XC_KQ) * shA[c].rows_pad);
  }
  {
    PhaseTimer t(h, XTD_T_XC_SLICE);
    for (int c = 0; c < nch; ++c)
      XTD_TRY(oz_slice(S, zS[c], zsc[c], shZ[c], h->Z[c], h->ch[c]->ldz, 0, 1, 1, s));
  }
  for (long g0 = 0; g0 < h->ng; g0 += GB) {
    const int gb = (int)std::min<long>(GB, h->ng - g0);
    const int nmt_g = (int)cdiv(gb, OZ_BM);
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        OzGemmParams p;
        p.A = ch->phivF + (size_t)(g0 / OZ_BM) * ch->ozPF.nkb * S * (OZ_BM * OZ_KB);
        p.B = zS[c]; p.sa = ch->phivFs + g0; p.sb = zsc[c];
        p.nmt = nmt_g; p.nnt = shZ[c].nrt; p.nkb = ch->ozPF.nkb; p.nq = 1; p.group = 1; p.b_q0 = 0;
        p.Mpad = nmt_g * OZ_BM; p.Npad = shZ[c].rows_pad; p.splits = 1; p.W = Y[c]; p.alpha = 1.0;
        XTD_TRY(oz_gemm(S, p, s));
        h->gemm.flops += 2.0 * gb * (double)(nvec * ch->no) * ch->nv;
      }
    }
    {
      PhaseTimer t(h, XTD_T_XC_STREAM);
      XcArgs a;
      a.nch = nch; a.nvec = nvec; a.gb = gb; a.g0 = g0;
      for (int c = 0; c < 2; ++c) {
        const bool on = c < nch;
        a.Y[c] = on ? Y[c] : nullptr; a.ldY[c] = on ? shZ[c].rows_pad : 0; a.y_comp[c] = 0;
        a.phi[c] = on ? h->ch[c]->phi.p : nullptr; a.ldphi[c] = on ? h->ch[c]->ldphi : 0; a.phi_comp[c] = on ? h->ng * h->ch[c]->ldphi : 0;
        a.no[c] = on ? h->ch[c]->no : 0;
      }
      a.wf = (h->fxc_kind == XTD_FXC_ALDA0) ? h->fxc : h->wf.p;
      if (h->fxc_kind == XTD_FXC_UKS) launch_xc<1, XC_KIND_UKS, false>(a, s);
      else if (h->fxc_kind == XTD_FXC_ALDA0) launch_xc<1, XC_KIND_ALDA0, false>(a, s);
      else launch_xc<1, XC_KIND_MCOL, false>(a, s);
      LAUNCH_CHECK();
    }
    const int nqc = (int)cdiv(gb, OZ_XC_KQ);
    {
      PhaseTimer t(h, XTD_T_XC_SLICE);
      for (int c = 0; c < nch; ++c)
        XTD_TRY(oz_slice(S, aS[c], asc[c], shA[c], Y[c], shZ[c].rows_pad, (long)OZ_XC_KQ * shZ[c].rows_pad, nqc, 1, s, true, gb));
    }
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        OzGemmParams p;
        p.A = aS[c]; p.B = ch->phivB; p.sa = asc[c]; p.sb = ch->phivBs;
        p.nmt = shA[c].nrt; p.nnt = ch->ozPB.nrt; p.nkb = shA[c].nkb; p.nq = nqc; p.group = 1; p.b_q0 = (int)(g0 / OZ_XC_KQ);
        p.Mpad = shA[c].rows_pad; p.Npad = ch->ozPB.rows_pad;
        p.splits = std::min(splits_max, oz_choose_splits(p.nmt * p.nnt, nqc, h->gemm.num_sms));
        p.W = W; p.alpha = 1.0;
        XTD_TRY(oz_gemm(S, p, s));
        const int M = nvec * ch->no, N = ch->nv;
        const long nblk = cdiv((long)M * N, 256);
        reduce_splits_kernel<<<dim3((unsigned)(nblk > 4096 ? 4096 : nblk), 1), 256, 0, s>>>(
            h->SIG + h->sig_base[c], ch->ldz, 0, W, ch->ozPB.rows_pad, 0, (long)shA[c].rows_pad * ch->ozPB.rows_pad, p.splits, M, N, 1, 0, 0, 0);
        LAUNCH_CHECK();
        h->gemm.flops += 2.0 * gb * (double)M * N;
      }
    }
  }
  return XTD_OK;
}

// Value + gradient kernels (UKS GGA of X-TDA, multicollinear GGA) in the split-gradient form with its four value GEMMs emulated:
//   F1  Y0[g][(x,o)] = sum_v phiv0[g][v] Z[(x,o)][v]            F2  T[x][g][v] = sum_o phi0[g][o] Z[x][o][v]      (batched over x)
//   streaming kernel (unchanged): rho from Y0, T and the gradient components; A -> Y0, B -> T in place
//   B1  SIG[(x,o)][v] += sum_g A[g][(x,o)] phiv0[g][v]           B2  SIG[x][o][v] += sum_g phi0[g][o] B[x][g][v]   (batched over x)
static int run_xc_split_emulated(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  const int nch = (int)h->ch.size();
  const int S = h->oz_slices;
  OzShape shZ[2], shA[2], shZt[2], shBt[2];
  size_t per_g = 0, fixed = 0, w_doubles = 0;
  const int splits_max = 8;
  for (int c = 0; c < nch; ++c) {
    Channel* ch = h->ch[c];
    shZ[c].set(nvec * ch->no, OZ_BN, ch->nv);        // F1 B operand: rows (x,o), K = v
    shA[c].set(nvec * ch->no, OZ_BM, OZ_XC_KQ);      // B1 A operand: rows (x,o), K = grid block
    shZt[c].set(ch->nv, OZ_BN, ch->no);              // F2 B operand: rows v, K = o, one q-slice (batch) per x
    shBt[c].set(ch->nv, OZ_BN, OZ_XC_KQ);            // B2 B operand: rows v, K = grid block, one batch per x
    per_g += (size_t)shZ[c].rows_pad + (size_t)nvec * shZt[c].rows_pad + (size_t)shA[c].rows_pad * S / 8 + (size_t)nvec * shBt[c].rows_pad * S / 8 + 2;
    fixed += shZ[c].slice_bytes(1, S) / 8 + shZ[c].rows_pad + shZt[c].slice_bytes(nvec, S) / 8 + (size_t)nvec * shZt[c].rows_pad + 256;
    fixed += (size_t)(65536 / OZ_XC_KQ) * ((size_t)shA[c].rows_pad + (size_t)nvec * shBt[c].rows_pad) + 256;
    w_doubles = std::max(w_doubles, (size_t)splits_max * shA[c].rows_pad * ch->ozPB.rows_pad);
    w_doubles = std::max(w_doubles, (size_t)splits_max * nvec * ch->ozOB.rows_pad * shBt[c].rows_pad);
  }
  fixed += w_doubles + 8192;
  XTD_REQUIRE(h->scratch_doubles > fixed + per_g * (OZ_XC_KQ + 128), XTD_ERR_NOMEM, "workspace too small for one block of the emulated grid path");
  long GB = (long)((h->scratch_doubles - fixed) / per_g) - 128;
  GB = std::min<long>(GB, 1 << 16);
  if (h->env.max_gb > 0) GB = std::min<long>(GB, std::max<long>(h->env.max_gb, OZ_XC_KQ));
  GB = GB / OZ_XC_KQ * OZ_XC_KQ;
  h->last_grid_chunks = cdiv(h->ng, GB);
  double* cur = h->scratch;
  auto take = [&](size_t n) { double* p = cur; cur += (n + 31) & ~(size_t)31; return p; };
  double* W = take(w_doubles);
  const long gbmax = round_up(std::min<long>(GB, h->ng), 128);
  const long nqmax = cdiv(gbmax, OZ_XC_KQ);
  int8_t *zS[2], *ztS[2], *aS[2], *bS[2];
  double *zsc[2], *ztsc[2], *Y[2], *T[2], *asc[2], *bsc[2];
  for (int c = 0; c < nch; ++c) {
    zS[c] = reinterpret_cast<int8_t*>(take(shZ[c].slice_bytes(1, S) / 8));
    zsc[c] = take(shZ[c].rows_pad);
    ztS[c] = reinterpret_cast<int8_t*>(take(shZt[c].slice_bytes(nvec, S) / 8));
    ztsc[c] = take((size_t)nvec * shZt[c].rows_pad);
    Y[c] = take((size_t)gbmax * shZ[c].rows_pad);
    T[c] = take((size_t)nvec * gbmax * shZt[c].rows_pad);
    aS[c] = reinterpret_cast<int8_t*>(take((size_t)nqmax * shA[c].slice_bytes(1, S) / 8));
    asc[c] = take((size_t)nqmax * shA[c].rows_pad);
    bS[c] = reinterpret_cast<int8_t*>(take((size_t)nvec * nqmax * shBt[c].slice_bytes(1, S) / 8));
    bsc[c] = take((size_t)nvec * nqmax * shBt[c].rows_pad);
  }
  {
    PhaseTimer t(h, XTD_T_XC_SLICE);
    for (int c = 0; c < nch; ++c) {
      Channel* ch = h->ch[c];
      XTD_TRY(oz_slice(S, zS[c], zsc[c], shZ[c], h->Z[c], ch->ldz, 0, 1, 1, s));
      if (ch->no >= h->env.oz_short_k) XTD_TRY(oz_slice(S, ztS[c], ztsc[c], shZt[c], h->ZT[c], ch->ldzt, (long)ch->nv * ch->ldzt, nvec, 1, s));
    }
  }
  for (long g0 = 0; g0 < h->ng; g0 += GB) {
    const int gb = (int)std::min<long>(GB, h->ng - g0);
    const int nmt_g = (int)cdiv(gb, OZ_BM);
    const long mpad_g = (long)nmt_g * OZ_BM;
    const int nqc = (int)cdiv(gb, OZ_XC_KQ);
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        OzGemmParams p;                       // F1
        p.A = ch->phivF + (size_t)(g0 / OZ_BM) * ch->ozPF.nkb * S * (OZ_BM * OZ_KB);
        p.B = zS[c]; p.sa = ch->phivFs + g0; p.sb = zsc[c];
        p.nmt = nmt_g; p.nnt = shZ[c].nrt; p.nkb = ch->ozPF.nkb; p.nq = 1; p.group = 1; p.b_q0 = 0;
        p.Mpad = (int)mpad_g; p.Npad = shZ[c].rows_pad; p.splits = 1; p.W = Y[c]; p.alpha = 1.0;
        XTD_TRY(oz_gemm(S, p, s));
        h->gemm.flops += 2.0 * gb * (double)(nvec * ch->no) * ch->nv;
        if (ch->no < h->env.oz_short_k) {
          // F2 has the occupied count as its contraction length: a few k-steps per tile, where the INT8 kernel is all epilogue
          // (measured at no = 137: 7.4 ms per 40 960-point chunk against 5.4 ms on the DMMA GEMM) -- keep it on FP64 DMMA
          GemmDesc e;
          e.b_kc = false;
          e.A = view2d(ch->phi.p, ch->ldphi, gb, ch->no, (int)g0, 0);
          e.B = view3d(h->Z[c], ch->ldz, (long)ch->no * ch->ldz, nvec, ch->no, ch->nv);
          e.M = gb; e.N = ch->nv; e.K = ch->no; e.batches = nvec; e.z_div = 1; e.a_hi = 0; e.b_hi = 1;
          e.C = T[c]; e.ldc = shZt[c].rows_pad; e.c_batch_stride = mpad_g * shZt[c].rows_pad;
          XTD_TRY(gemm(h->gemm, e, s));
          h->gemm.flops += 2.0 * gb * (double)(nvec * ch->no) * ch->nv;
          continue;
        }
        OzGemmParams q;                       // F2, one batch per trial vector
        q.A = ch->phiF + (size_t)(g0 / OZ_BM) * ch->ozOF.nkb * S * (OZ_BM * OZ_KB);
        q.B = ztS[c]; q.sa = ch->phiFs + g0; q.sb = ztsc[c];
        q.nmt = nmt_g; q.nnt = shZt[c].nrt; q.nkb = ch->ozOF.nkb; q.nq = 1; q.group = 1; q.b_q0 = 0;
        q.Mpad = (int)mpad_g; q.Npad = shZt[c].rows_pad; q.splits = 1; q.W = T[c]; q.alpha = 1.0;
        q.batches = nvec; q.b_bstride = (long)shZt[c].slice_bytes(1, S); q.sb_bstride = shZt[c].rows_pad;
        q.w_bstride = mpad_g * shZt[c].rows_pad;
        XTD_TRY(oz_gemm(S, q, s));
        h->gemm.flops += 2.0 * gb * (double)(nvec * ch->no) * ch->nv;
      }
    }
    {
      PhaseTimer t(h, XTD_T_XC_STREAM);
      XcArgs2 a;
      a.nch = nch; a.nvec = nvec; a.gb = gb; a.g0 = g0; a.t_rows = mpad_g;
      for (int c = 0; c < 2; ++c) {
        const bool on = c < nch;
        Channel* ch = on ? h->ch[c] : nullptr;
        a.Y[c] = on ? Y[c] : nullptr; a.ldY[c] = on ? shZ[c].rows_pad : 0;
        a.T[c] = on ? T[c] : nullptr; a.ldT[c] = on ? shZt[c].rows_pad : 0;
        a.phi[c] = on ? ch->phi.p : nullptr; a.ldphi[c] = on ? ch->ldphi : 0; a.phi_comp[c] = on ? h->ng * ch->ldphi : 0;
        a.phiv[c] = on ? ch->phiv.p : nullptr; a.ldphiv[c] = on ? ch->ldphiv : 0; a.phiv_comp[c] = on ? h->ng * ch->ldphiv : 0;
        a.no[c] = on ? ch->no : 0; a.nv[c] = on ? ch->nv : 0;
      }
      a.wf = h->wf.p;
      if (h->fxc_kind == XTD_FXC_UKS) XTD_TRY(launch_xc_split<XC_KIND_UKS>(a, s));
      else XTD_TRY(launch_xc_split<XC_KIND_MCOL>(a, s));
      LAUNCH_CHECK();
    }
    {
      PhaseTimer t(h, XTD_T_XC_SLICE);
      for (int c = 0; c < nch; ++c) {
        // A planes of B1 from Y (now holding A[g][(x,o)]); B planes of B2 from T (now holding B[x][g][v]), one batch per x
        XTD_TRY(oz_slice(S, aS[c], asc[c], shA[c], Y[c], shZ[c].rows_pad, (long)OZ_XC_KQ * shZ[c].rows_pad, nqc, 1, s, true, gb));
        for (int x = 0; x < nvec; ++x)
          XTD_TRY(oz_slice(S, bS[c] + (size_t)x * nqmax * shBt[c].slice_bytes(1, S), bsc[c] + (size_t)x * nqmax * shBt[c].rows_pad, shBt[c],
                           T[c] + (size_t)x * mpad_g * shZt[c].rows_pad, shZt[c].rows_pad, (long)OZ_XC_KQ * shZt[c].rows_pad, nqc, 1, s, true, gb));
      }
    }
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        const int M = nvec * ch->no, N = ch->nv;
        OzGemmParams p;                       // B1
        p.A = aS[c]; p.B = ch->phivB; p.sa = asc[c]; p.sb = ch->phivBs;
        p.nmt = shA[c].nrt; p.nnt = ch->ozPB.nrt; p.nkb = shA[c].nkb; p.nq = nqc; p.group = 1; p.b_q0 = (int)(g0 / OZ_XC_KQ);
        p.Mpad = shA[c].rows_pad; p.Npad = ch->ozPB.rows_pad;
        p.splits = std::min(splits_max, oz_choose_splits(p.nmt * p.nnt, nqc, h->gemm.num_sms));
        p.W = W; p.alpha = 1.0;
        XTD_TRY(oz_gemm(S, p, s));
        long nblk = cdiv((long)M * N, 256);
        reduce_splits_kernel<<<dim3((unsigned)(nblk > 4096 ? 4096 : nblk), 1), 256, 0, s>>>(
            h->SIG + h->sig_base[c], ch->ldz, 0, W, ch->ozPB.rows_pad, 0, (long)shA[c].rows_pad * ch->ozPB.rows_pad, p.splits, M, N, 1, 0, 0, 0);
        LAUNCH_CHECK();
        OzGemmParams q;                       // B2, one batch per trial vector: A = planes of phi0^T (shared), B = planes of B[x]^T
        q.A = ch->phiB; q.B = bS[c]; q.sa = ch->phiBs; q.sb = bsc[c];
        q.nmt = ch->ozOB.nrt; q.nnt = shBt[c].nrt; q.nkb = shBt[c].nkb; q.nq = nqc; q.group = 1; q.b_q0 = 0;
        q.Mpad = ch->ozOB.rows_pad; q.Npad = shBt[c].rows_pad;
        q.splits = std::min(splits_max, oz_choose_splits(q.nmt * q.nnt * nvec, nqc, h->gemm.num_sms));
        q.W = W; q.alpha = 1.0;
        q.batches = nvec;
        q.b_bstride = (long)nqmax * shBt[c].slice_bytes(1, S); q.sb_bstride = (long)nqmax * shBt[c].rows_pad;
        q.w_bstride = (long)q.splits * q.Mpad * q.Npad;
        // the A operand / its scales start at this chunk's first grid block for every batch
        q.A = ch->phiB + (size_t)(g0 / OZ_XC_KQ) * ch->ozOB.slice_bytes(1, S);
        q.sa = ch->phiBs + (size_t)(g0 / OZ_XC_KQ) * ch->ozOB.rows_pad;
        XTD_TRY(oz_gemm(S, q, s));
        nblk = cdiv((long)ch->no * N, 256);
        reduce_splits_kernel<<<dim3((unsigned)(nblk > 4096 ? 4096 : nblk), nvec), 256, 0, s>>>(
            h->SIG + h->sig_base[c], ch->ldz, (long)ch->no * ch->ldz, W, shBt[c].rows_pad, q.w_bstride, (long)q.Mpad * q.Npad, q.splits, ch->no, N,
            1, 0, 0, 0);
        LAUNCH_CHECK();
        h->gemm.flops += 4.0 * gb * (double)M * N;
      }
    }
  }
  return XTD_OK;
}

static int run_xc(xtd_engine* h, int nvec) {
  if (h->ch[0]->xc_oz) return run_xc_emulated(h, nvec);
  if (h->ch[0]->xc_oz_split) return run_xc_split_emulated(h, nvec);
  cudaStream_t s = h->stream;
  const int nch = (int)h->ch.size();
  const int nve = h->nvar_eff;
  const bool split = xc_use_split(h, nvec);
  // grid chunk: the per-point buffers of all channels must fit the scratch region
  size_t per_g = 0;
  long ldY[2] = {0, 0};
  for (int c = 0; c < nch; ++c) {
    ldY[c] = pad_ld((long)nvec * h->ch[c]->no);
    per_g += split ? (size_t)ldY[c] + (size_t)nvec * h->ch[c]->ldphiv : (size_t)nve * ldY[c];
  }
  long GB = (long)(h->scratch_doubles / per_g);
  GB = std::min<long>(GB, 1 << 16);
  if (h->env.max_gb > 0) GB = std::min<long>(GB, std::max<long>(h->env.max_gb, 128));
  GB = (GB / 128) * 128;
  XTD_REQUIRE(GB >= 128, XTD_ERR_NOMEM, "workspace too small for a 128-point grid chunk");
  h->last_grid_chunks = cdiv(h->ng, GB);
  for (long g0 = 0; g0 < h->ng; g0 += GB) {
    const int gb = (int)std::min<long>(GB, h->ng - g0);
    double *Y[2] = {nullptr, nullptr}, *T[2] = {nullptr, nullptr};
    double* cur = h->scratch;
    for (int c = 0; c < nch; ++c) {
      Y[c] = cur;
      cur += (size_t)(split ? 1 : nve) * gb * ldY[c];
      if (split) {
        T[c] = cur;
        cur += (size_t)nvec * gb * h->ch[c]->ldphiv;
      }
    }
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        // Y[cmp][g][(x,o)] = sum_v phiv[cmp][g0+g][v] Z[(x,o)][v]     (trial vectors evaluated on the grid, virtual side;
        // only the value component in the split-gradient form)
        GemmDesc d;
        d.A = view3d(ch->phiv.p, ch->ldphiv, h->ng * ch->ldphiv, nve, gb, ch->nv, (int)g0, 0);
        d.B = view2d(h->Z[c], ch->ldz, nvec * ch->no, ch->nv);
        d.M = gb; d.N = nvec * ch->no; d.K = ch->nv; d.batches = split ? 1 : nve; d.a_hi = 1; d.b_hi = 0;
        d.C = Y[c]; d.ldc = ldY[c]; d.c_batch_stride = (long)gb * ldY[c];
        XTD_TRY(gemm(h->gemm, d, s));
        if (split) {
          // T[x][g][v] = sum_o phi_0[g0+g][o] Z[x][o][v]              (occupied side)
          GemmDesc e;
          e.b_kc = false;
          e.A = view2d(ch->phi.p, ch->ldphi, gb, ch->no, (int)g0, 0);
          e.B = view3d(h->Z[c], ch->ldz, (long)ch->no * ch->ldz, nvec, ch->no, ch->nv);
          e.M = gb; e.N = ch->nv; e.K = ch->no; e.batches = nvec; e.z_div = 1; e.a_hi = 0; e.b_hi = 1;
          e.C = T[c]; e.ldc = ch->ldphiv; e.c_batch_stride = (long)gb * ch->ldphiv;
          XTD_TRY(gemm(h->gemm, e, s));
        }
      }
    }
    {
      PhaseTimer t(h, XTD_T_XC_STREAM);
      if (split) {
        XcArgs2 a;
        a.nch = nch; a.nvec = nvec; a.gb = gb; a.g0 = g0;
        for (int c = 0; c < 2; ++c) {
          const bool on = c < nch;
          Channel* ch = on ? h->ch[c] : nullptr;
          a.Y[c] = on ? Y[c] : nullptr; a.ldY[c] = on ? ldY[c] : 0;
          a.T[c] = on ? T[c] : nullptr; a.ldT[c] = on ? ch->ldphiv : 0;
          a.phi[c] = on ? ch->phi.p : nullptr; a.ldphi[c] = on ? ch->ldphi : 0; a.phi_comp[c] = on ? h->ng * ch->ldphi : 0;
          a.phiv[c] = on ? ch->phiv.p : nullptr; a.ldphiv[c] = on ? ch->ldphiv : 0; a.phiv_comp[c] = on ? h->ng * ch->ldphiv : 0;
          a.no[c] = on ? ch->no : 0; a.nv[c] = on ? ch->nv : 0;
        }
        a.wf = h->wf.p;
        if (h->fxc_kind == XTD_FXC_UKS) XTD_TRY(launch_xc_split<XC_KIND_UKS>(a, s));
        else XTD_TRY(launch_xc_split<XC_KIND_MCOL>(a, s));
      } else {
        XcArgs a;
        a.nch = nch; a.nvec = nvec; a.gb = gb; a.g0 = g0;
        for (int c = 0; c < nch; ++c) {
          a.Y[c] = Y[c]; a.ldY[c] = ldY[c]; a.y_comp[c] = (long)gb * ldY[c];
          a.phi[c] = h->ch[c]->phi.p; a.ldphi[c] = h->ch[c]->ldphi; a.phi_comp[c] = h->ng * h->ch[c]->ldphi;
          a.no[c] = h->ch[c]->no;
        }
        if (nch == 1) { a.Y[1] = nullptr; a.phi[1] = nullptr; a.no[1] = 0; a.ldY[1] = a.y_comp[1] = a.ldphi[1] = a.phi_comp[1] = 0; }
        a.wf = (h->fxc_kind == XTD_FXC_ALDA0) ? h->fxc : h->wf.p;
        if (h->fxc_kind == XTD_FXC_UKS) {
          if (nve == 1) launch_xc<1, XC_KIND_UKS>(a, s);
          else if (h->tau) launch_xc<4, XC_KIND_UKS, true>(a, s);
          else launch_xc<4, XC_KIND_UKS>(a, s);
        } else if (h->fxc_kind == XTD_FXC_ALDA0) {
          launch_xc<1, XC_KIND_ALDA0>(a, s);
        } else {
          if (nve == 1) launch_xc<1, XC_KIND_MCOL>(a, s);
          else if (h->tau) launch_xc<4, XC_KIND_MCOL, true>(a, s);
          else launch_xc<4, XC_KIND_MCOL>(a, s);
        }
      }
      LAUNCH_CHECK();
    }
    {
      PhaseTimer t(h, XTD_T_XC_GEMM);
      for (int c = 0; c < nch; ++c) {
        Channel* ch = h->ch[c];
        // SIG[(x,o)][v] += sum_cmp sum_g A[cmp][g][(x,o)] phiv[cmp][g0+g][v]      (integration straight into the MO block)
        GemmDesc d;
        d.a_kc = false; d.b_kc = false;
        d.A = view3d(Y[c], ldY[c], (long)gb * ldY[c], split ? 1 : nve, gb, nvec * ch->no);
        d.B = view3d(ch->phiv.p, ch->ldphiv, h->ng * ch->ldphiv, nve, gb, ch->nv, (int)g0, 0);
        d.M = nvec * ch->no; d.N = ch->nv; d.K = gb; d.nouter = split ? 1 : nve;
        d.C = h->SIG + h->sig_base[c]; d.ldc = ch->ldz; d.accumulate = true;
        XTD_TRY(gemm(h->gemm, d, s));
        if (split) {
          // SIG[x][o][v] += sum_g phi_0[g0+g][o] B[x][g][v]
          GemmDesc e;
          e.a_kc = false; e.b_kc = false;
          e.A = view2d(ch->phi.p, ch->ldphi, gb, ch->no, (int)g0, 0);
          e.B = view3d(T[c], ch->ldphiv, (long)gb * ch->ldphiv, nvec, gb, ch->nv);
          e.M = ch->no; e.N = ch->nv; e.K = gb; e.batches = nvec; e.z_div = 1; e.a_hi = 0; e.b_hi = 1;
          e.C = h->SIG + h->sig_base[c]; e.ldc = ch->ldz; e.c_batch_stride = (long)ch->no * ch->ldz; e.accumulate = true;
          XTD_TRY(gemm(h->gemm, e, s));
        }
      }
    }
  }
  return XTD_OK;
}

// Uniform-weight exchange term with both contractions on the INT8 tensor cores:
//   K1 (oz_k1_kernel)   U[P][(i,x)][b] = sum_j Loo[(P,i)][j] zt[x][b][j]; U never exists in fp64: the epilogue writes its S int8 digit
//                       planes (the A operand of K2) directly, under an a-priori power-of-two scale per (row, group of aux functions)
//   K2 (tcgen05.mma kind::i8, TMEM)   SIG[x][i][a] += w sum_P sum_b U[P][(i,x)][b] Lvv[P][a][b]   against the int8 planes of Lvv
// Block-weighted terms (XSF Delta A): the wide second virtual block [col0, nv) is emulated -- one half-transform per occupied
// row block ib with the trial vectors scaled by w(ib, 1, :, :), each filling its rows of the A planes, then ONE contraction
// against the planes of Lvv[col0:, :]; the narrow first block was done by the DMMA narrow pass of run_k.
static int run_k_emulated(xtd_engine* h, const KTermRec& k, int nvec) {
  cudaStream_t s = h->stream;
  Channel* ch = h->ch[k.ch];
  const long naux = h->naux[k.tensor];
  const int S = h->oz_slices, G = ch->oz_group;
  const int col0 = ch->oz_col0[k.tensor];
  struct RowPass { int i_lo, i_hi; BlockSplit bs; };
  std::vector<RowPass> passes;
  if (k.uniform) {
    passes.push_back({0, ch->no, BlockSplit()});
  } else {
    const int o2off = ch->o_blocks.size() > 1 ? ch->o_blocks[1].first : ch->no;
    const int v2off = ch->v_blocks.size() > 1 ? ch->v_blocks[1].first : ch->nv;
    const int ab = col0 > 0 ? 1 : 0;
    const int nib = ch->o_blocks.size() > 1 ? 2 : 1;
    for (int ib = 0; ib < nib; ++ib) {
      RowPass rp;
      rp.i_lo = ib == 0 ? 0 : o2off;
      rp.i_hi = (ib == 0 && nib == 2) ? o2off : ch->no;
      rp.bs.o2off = o2off; rp.bs.v2off = v2off;       // scale_blocks_kernel on the transposed vectors zt[x][b][j], as in run_k
      for (int j = 0; j < 2; ++j)
        for (int b = 0; b < 2; ++b) rp.bs.w[j][b] = k.w[ib][ab][j < k.nob ? j : 0][b < k.nvb ? b : 0];
      passes.push_back(rp);
    }
  }
  const int npass = (int)passes.size();
  OzShape shA, shZt;
  shA.set(nvec * ch->no, OZ_BM, ch->nv);          // rows m = x no + i of the contraction's A operand
  shZt.set(ch->nv, OZ_BN, ch->no);                // zt[x][b][j]: one q-slice per trial vector
  const OzShape &shB = ch->ozB, &shL = ch->ozL;
  const int tiles = shA.nrt * shB.nrt;
  int splits_max = std::min<long>(64, std::max<long>(1, cdiv(naux, G)));
  size_t w_doubles = (size_t)splits_max * shA.rows_pad * shB.rows_pad;
  while (splits_max > 1 && w_doubles * 4 > h->scratch_doubles) { splits_max /= 2; w_doubles = (size_t)splits_max * shA.rows_pad * shB.rows_pad; }
  const size_t zt_one = shZt.slice_bytes(nvec, S) / 8 + (size_t)nvec * shZt.rows_pad + nvec + 128;
  const size_t zt_doubles = npass * zt_one + (size_t)nvec * shZt.rows_pad + (k.uniform ? 0 : (size_t)nvec * ch->nv * ch->ldzt) + 256;
  const size_t a_per_p = shA.slice_bytes(1, S) / 8;
  const size_t per_p = a_per_p + (size_t)cdiv(shA.rows_pad, G) + 1;
  XTD_REQUIRE(h->scratch_doubles > w_doubles + zt_doubles + (size_t)G * per_p + 4096, XTD_ERR_NOMEM,
              "workspace too small for one group of the emulated exchange contraction");
  long pc = (long)((h->scratch_doubles - w_doubles - zt_doubles - 4096) / per_p);
  pc = std::min<long>(pc, naux);
  if (pc > 32768) pc = 32768;
  if (h->env.max_pc > 0) pc = std::min<long>(pc, h->env.max_pc);
  if (pc < naux) pc = std::max<long>(pc / G * G, G);
  h->last_aux_chunks = std::max<long>(h->last_aux_chunks, cdiv(naux, pc));
  double* cur = h->scratch;
  auto take = [&](size_t n) { double* p = cur; cur += (n + 31) & ~(size_t)31; return p; };
  double* W = take(w_doubles);
  double* ztNorm = take((size_t)nvec * shZt.rows_pad);
  double* zts_tmp = k.uniform ? nullptr : take((size_t)nvec * ch->nv * ch->ldzt);
  int8_t* ztS[2]; double* ztScale[2]; double* zmax[2];
  for (int ip = 0; ip < npass; ++ip) {
    ztS[ip] = reinterpret_cast<int8_t*>(take(shZt.slice_bytes(nvec, S) / 8));
    ztScale[ip] = take((size_t)nvec * shZt.rows_pad);
    zmax[ip] = take(nvec);
  }
  int8_t* As = reinterpret_cast<int8_t*>(take((size_t)pc * a_per_p));
  double* so = take((size_t)cdiv(pc, G) * shA.rows_pad);
  {
    PhaseTimer t(h, XTD_T_K2_SLICE);
    for (int ip = 0; ip < npass; ++ip) {
      const double* zt = h->ZT[k.ch];
      if (!k.uniform) {
        scale_blocks_kernel<<<dim3((unsigned)cdiv(ch->no, 128), ch->nv, nvec), 128, 0, s>>>(zts_tmp, h->ZT[k.ch], ch->ldzt, (long)ch->nv * ch->ldzt,
                                                                                          ch->nv, ch->no, passes[ip].bs);
        LAUNCH_CHECK();
        zt = zts_tmp;
      }
      XTD_TRY(oz_slice(S, ztS[ip], ztScale[ip], shZt, zt, ch->ldzt, (long)ch->nv * ch->ldzt, nvec, 1, s));
      oz_rownorm_kernel<<<dim3(shZt.rows_pad, nvec), 128, 0, s>>>(ztNorm, shZt.rows_pad, zt, ch->ldzt, (long)ch->nv * ch->ldzt, ch->nv, ch->no);
      LAUNCH_CHECK();
      oz_colmax_kernel<<<nvec, 256, 0, s>>>(zmax[ip], ztNorm, shZt.rows_pad, ch->nv);
      LAUNCH_CHECK();
    }
  }
  for (long P0 = 0; P0 < naux; P0 += pc) {
    const int pn = (int)std::min<long>(pc, naux - P0);
    const int ng = (int)cdiv(pn, G);
    {
      PhaseTimer t(h, XTD_T_K1);
      for (int ip = 0; ip < npass; ++ip) {
        const RowPass& rp = passes[ip];
        oz_bound_scale_kernel<<<dim3((unsigned)cdiv(shA.rows_pad, 256), ng), 256, 0, s>>>(so, shA.rows_pad, ch->LooNorm[k.tensor] + (size_t)P0 * ch->no,
                                                                                          ch->no, zmax[ip], pn, G, nvec, ch->no, rp.i_lo, rp.i_hi);
        LAUNCH_CHECK();
        // the packed row tiles of every group that hold the rows of this pass (P0 is a group boundary: pc is a multiple of G)
        const int o2 = ch->oz_row_split();
        OzK1Params q;
        q.A = ch->LooS[k.tensor] + shL.slice_bytes(P0 / G, S); q.B = ztS[ip];
        q.sa = ch->LooScale[k.tensor] + (size_t)(P0 / G) * shL.rows_pad; q.sb = ztScale[ip]; q.so = so; q.out = As;
        q.np = pn; q.ntg = shL.nrt; q.nbt = shZt.nrt; q.nkb1 = shL.nkb; q.nvec = nvec; q.no = ch->no; q.o2 = o2; q.group = G;
        q.nmt2 = shA.nrt; q.nkb2 = shA.nkb; q.Mpad2 = shA.rows_pad;
        q.i_lo = rp.i_lo; q.i_hi = rp.i_hi;
        q.t0 = oz_packed_row_lo(rp.i_lo, G, o2) / OZ_BM;
        q.nt_run = (int)cdiv(oz_packed_row_hi(rp.i_hi, G, o2, ch->no), OZ_BM) - q.t0;
        q.npairs = (long)ng * q.nt_run * cdiv((long)nvec * q.nbt, 2);
        XTD_TRY(oz_k1(S, q, s));
        h->gemm.flops += 2.0 * pn * (double)(rp.i_hi - rp.i_lo) * ch->no * ch->nv * nvec;
      }
    }
    {
      PhaseTimer t(h, XTD_T_K2);
      OzGemmParams p;
      p.A = As; p.B = ch->LvvS[k.tensor]; p.sa = so; p.sb = ch->LvvScale[k.tensor];
      p.nmt = shA.nrt; p.nnt = shB.nrt; p.nkb = shA.nkb; p.nq = pn; p.group = G; p.b_q0 = (int)P0;
      p.Mpad = shA.rows_pad; p.Npad = shB.rows_pad;
      p.splits = std::min(splits_max, oz_choose_splits(tiles, ng, h->gemm.num_sms));
      p.W = W; p.alpha = k.uniform ? k.w[0][0][0][0] : 1.0;
      XTD_TRY(oz_gemm(S, p, s));
      const int M = nvec * ch->no, N = ch->nv - col0;
      const long nblk = cdiv((long)M * N, 256);
      reduce_splits_kernel<<<dim3((unsigned)(nblk > 4096 ? 4096 : nblk), 1), 256, 0, s>>>(
          h->SIG + h->sig_base[k.ch] + col0, ch->ldz, 0, W, shB.rows_pad, 0, (long)shA.rows_pad * shB.rows_pad, p.splits, M, N, 1, 0, 0, 0);
      LAUNCH_CHECK();
      h->gemm.flops += 2.0 * M * N * (double)ch->nv * pn;
    }
  }
  return XTD_OK;
}

static int run_k(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  for (const KTermRec& k : h->kterms) {
    Channel* ch = h->ch[k.ch];
    const long naux = h->naux[k.tensor];
    if (naux == 0) continue;
    const double* Loo = ch->Loo[k.tensor].p;
    const double* Lvv = ch->Lvv[k.tensor].p;
    if (ch->use_oz[k.tensor] && k.uniform) {
      XTD_TRY(run_k_emulated(h, k, nvec));
      continue;
    }
    // aux chunk so that U[pc][nvec][no][ldz] fits the scratch region
    const size_t per_p = (size_t)nvec * ch->no * ch->ldz;
    long pc = (long)(h->scratch_doubles / per_p);
    XTD_REQUIRE(pc >= 1, XTD_ERR_NOMEM, "workspace too small for the exchange intermediate of one aux function");
    pc = std::min<long>(pc, naux);
    if ((long)pc * nvec > 65535) pc = 65535 / nvec;
    if (h->env.max_pc > 0) pc = std::min<long>(pc, h->env.max_pc);
    h->last_aux_chunks = std::max<long>(h->last_aux_chunks, cdiv(naux, pc));
    double* U = h->scratch;
    std::vector<std::pair<int, int>> iblks, ablks;
    const int o2off = ch->o_blocks.size() > 1 ? ch->o_blocks[1].first : ch->no;
    const int v2off = ch->v_blocks.size() > 1 ? ch->v_blocks[1].first : ch->nv;
    if (k.uniform) { iblks.push_back({0, ch->no}); ablks.push_back({0, ch->nv}); }
    else {
      // block ranges extended over the zero pad position so every row / column of U and SIG is written
      iblks.push_back({0, o2off});
      if (ch->o_blocks.size() > 1) iblks.push_back({o2off, ch->no - o2off});
      ablks.push_back({0, v2off});
      if (ch->v_blocks.size() > 1) ablks.push_back({v2off, ch->nv - v2off});
    }
    // Narrow first virtual block (the open-shell columns of a spin-flip channel, a handful wide): contract the trial
    // vectors with those few rows of Lvv first,
    //   R[x][P][a'][j] = sum_b Lvo[(P,a')][b] (w z)[x][j][b]        (aux index flattened into the GEMM rows)
    //   sigma[x][i in iblk][a'] += sum_P sum_j Loo[P][i][j] R[x][P][a'][j]
    // instead of a full half-transform U plus a 128-wide output tile for a few columns.
    size_t ab_first = 0;
    const long ldj = ch->ldzt;
    const size_t zs_doubles = (size_t)nvec * ch->no * ch->ldz;
    const int wmax = std::max(v2off, ch->tail_w);
    if (!k.uniform && ch->need_narrow[k.tensor] && ablks.size() == 2 &&
        zs_doubles + (size_t)nvec * naux * wmax * ldj <= h->scratch_doubles && (long)nvec * naux < (1L << 30) && !h->env.no_narrow) {
      double* Zs = h->scratch;
      double* R = h->scratch + zs_doubles;
      // (rows of Lvv gathered per aux function, first output column, width, column block whose weights apply)
      struct Narrow { const double* L; int col0, w, ab; };
      std::vector<Narrow> passes;
      passes.push_back({ch->Lvo[k.tensor].p, 0, v2off, 0});
      if (ch->tail_w > 0) passes.push_back({ch->Lvt[k.tensor].p, ch->tail_start, ch->tail_w, 1});
      for (const Narrow& nw : passes)
        for (size_t ib = 0; ib < iblks.size(); ++ib) {
          PhaseTimer t(h, XTD_T_K1);
          BlockSplit bs;                       // the kernel is written for the transposed layout: roles of rows / columns swap
          bs.o2off = v2off; bs.v2off = o2off;
          for (int j = 0; j < 2; ++j)
            for (int b = 0; b < 2; ++b) bs.w[b][j] = k.w[ib][nw.ab][j < k.nob ? j : 0][b < k.nvb ? b : 0];
          scale_blocks_kernel<<<dim3((unsigned)cdiv(ch->nv, 128), ch->no, nvec), 128, 0, s>>>(Zs, h->Z[k.ch], ch->ldz, (long)ch->no * ch->ldz,
                                                                                            ch->no, ch->nv, bs);
          LAUNCH_CHECK();
          GemmDesc d;
          d.A = view2d(nw.L, ch->ldvv, (int)(naux * nw.w), ch->nv);
          d.B = view3d(Zs, ch->ldz, (long)ch->no * ch->ldz, nvec, ch->no, ch->nv);
          d.M = (int)(naux * nw.w); d.N = ch->no; d.K = ch->nv; d.batches = nvec; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
          d.C = R; d.ldc = ldj; d.c_batch_stride = naux * nw.w * ldj;
          XTD_TRY(gemm(h->gemm, d, s));
          const int i0 = iblks[ib].first, nr = iblks[ib].second;
          GemmDesc e;
          e.A = view3d(Loo, ch->ldoo, (long)ch->no * ch->ldoo, (int)naux, nr, ch->no, i0, 0);
          e.B = view3d(R, ldj, (long)nw.w * ldj, (int)(nvec * naux), nw.w, ch->no);
          e.M = nr; e.N = nw.w; e.K = ch->no; e.nouter = (int)naux; e.batches = nvec; e.z_div = 1; e.a_hi = 0; e.b_hi = (int)naux;
          e.C = h->SIG + h->sig_base[k.ch] + (long)i0 * ch->ldz + nw.col0; e.ldc = ch->ldz; e.c_batch_stride = (long)ch->no * ch->ldz;
          e.accumulate = true;
          XTD_TRY(gemm(h->gemm, e, s));
        }
      ab_first = 1;
      if (ch->tail_w > 0) ablks[1].second = ch->tail_start - v2off;     // the general pass stops at the last full 128-column tile
    }
    if (ch->use_oz[k.tensor]) {
      // block weights on the emulated path: the narrow first block is done (or there is none); the wide block is emulated
      XTD_REQUIRE(ab_first == (size_t)(ch->oz_col0[k.tensor] > 0 ? 1 : 0), XTD_ERR_NOMEM,
                  "workspace too small for the narrow-output exchange pass that the emulated path relies on");
      XTD_TRY(run_k_emulated(h, k, nvec));
      continue;
    }
    for (size_t ab = ab_first; ab < ablks.size(); ++ab) {
      for (long P0 = 0; P0 < naux; P0 += pc) {
        const int pn = (int)std::min<long>(pc, naux - P0);
        if (k.uniform) {
          // Uniform weights: flatten (P, i) into the row index so the small occupied dimension is not padded to the
          // 128-row tile per aux function.  U[P][i][x][b] = sum_j Loo[(P,i)][j] zt[x][b][j]; the contraction below
          // then reads rows m = (i, x) of slice P and scatters them to sigma[x][i][:] through the two-level row map.
          {
            PhaseTimer t(h, XTD_T_K1);
            GemmDesc d;
            d.A = view2d(Loo + P0 * ch->no * ch->ldoo, ch->ldoo, pn * ch->no, ch->no);
            d.B = view3d(h->ZT[k.ch], ch->ldzt, (long)ch->nv * ch->ldzt, nvec, ch->nv, ch->no);
            d.M = pn * ch->no; d.N = ch->nv; d.K = ch->no;
            d.batches = nvec; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
            d.C = U; d.ldc = (long)nvec * ch->ldz; d.c_batch_stride = ch->ldz;
            XTD_TRY(gemm(h->gemm, d, s));
          }
          {
            PhaseTimer t(h, XTD_T_K2);
            // SIG[x][i][a] += w * sum_P sum_b U[P][(i,x)][b] Lvv[P][a][b]
            GemmDesc d;
            d.A = view3d(U, ch->ldz, (long)nvec * ch->no * ch->ldz, pn, nvec * ch->no, ch->nv);
            d.B = view3d(Lvv, ch->ldvv, (long)ch->nv * ch->ldvv, (int)(naux - P0), ch->nv, ch->nv, 0, 0, (int)P0);
            d.M = nvec * ch->no; d.N = ch->nv; d.K = ch->nv; d.nouter = pn;
            d.C = h->SIG + h->sig_base[k.ch]; d.ldc = ch->ldz; d.accumulate = true;
            d.c_row_div = nvec; d.c_row_hi = ch->ldz; d.c_row_lo = (long)ch->no * ch->ldz;
            d.alpha = k.w[0][0][0][0];
            XTD_TRY(gemm(h->gemm, d, s));
          }
          continue;
        }
        // Block weights: one half-transform per (row block, column block) pair with the trial vectors scaled by
        // w(iblk, ablk, :, :); rows (P, i in block) are flattened as in the uniform case and land in U[P][i][x][b].
        {
          PhaseTimer t(h, XTD_T_K1);
          for (size_t ib = 0; ib < iblks.size(); ++ib) {
            BlockSplit bs;
            bs.o2off = o2off; bs.v2off = v2off;
            for (int j = 0; j < 2; ++j)
              for (int b = 0; b < 2; ++b) bs.w[j][b] = k.w[ib][ab][j < k.nob ? j : 0][b < k.nvb ? b : 0];
            scale_blocks_kernel<<<dim3((unsigned)cdiv(ch->no, 128), ch->nv, nvec), 128, 0, s>>>(h->ZTs[k.ch], h->ZT[k.ch], ch->ldzt,
                                                                                              (long)ch->nv * ch->ldzt, ch->nv, ch->no, bs);
            LAUNCH_CHECK();
            const int i0 = iblks[ib].first, nr = iblks[ib].second;
            const double* lrows = ch->need_split[k.tensor] ? ch->Loob[k.tensor][ib].p : Loo;   // single row block: Loo itself
            GemmDesc d;
            d.A = view2d(lrows + P0 * nr * ch->ldoo, ch->ldoo, pn * nr, ch->no);
            d.B = view3d(h->ZTs[k.ch], ch->ldzt, (long)ch->nv * ch->ldzt, nvec, ch->nv, ch->no);
            d.M = pn * nr; d.N = ch->nv; d.K = ch->no;
            d.batches = nvec; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
            d.C = U + (long)i0 * nvec * ch->ldz; d.ldc = (long)nvec * ch->ldz; d.c_batch_stride = ch->ldz;
            d.c_row_div = nr; d.c_row_hi = (long)ch->no * nvec * ch->ldz; d.c_row_lo = (long)nvec * ch->ldz;
            XTD_TRY(gemm(h->gemm, d, s));
          }
        }
        {
          PhaseTimer t(h, XTD_T_K2);
          // SIG[x][i][a in block] += sum_P sum_b U[P][(i,x)][b] Lvv[P][a][b]
          GemmDesc d;
          d.A = view3d(U, ch->ldz, (long)nvec * ch->no * ch->ldz, pn, nvec * ch->no, ch->nv);
          d.B = view3d(Lvv, ch->ldvv, (long)ch->nv * ch->ldvv, (int)(naux - P0), ablks[ab].second, ch->nv, ablks[ab].first, 0, (int)P0);
          d.M = nvec * ch->no; d.N = ablks[ab].second; d.K = ch->nv; d.nouter = pn;
          d.C = h->SIG + h->sig_base[k.ch] + ablks[ab].first; d.ldc = ch->ldz; d.accumulate = true;
          d.c_row_div = nvec; d.c_row_hi = ch->ldz; d.c_row_lo = (long)ch->no * ch->ldz;
          XTD_TRY(gemm(h->gemm, d, s));
        }
      }
    }
  }
  return XTD_OK;
}

// Exchange of the transposed trial density (hermi = 1 response of the Z-vector operator; grad_hb/tdroks_sfu.py:284-298):
//   sigma[x][i][a] += w sum_P sum_j Lov[P][j][a] W[P][i][x][j],   W[P][i][x][j] = sum_b Lov[P][i][b] z[x][j][b]
// 4 naux no^2 nv flops per vector -- no / nv of the direct exchange term -- as two DMMA GEMMs per aux chunk.
static int run_kt(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  for (const KTermTRec& k : h->ktterms) {
    Channel* ch = h->ch[k.ch];
    const long naux = h->naux[k.tensor];
    if (naux == 0 || k.w == 0.0) continue;
    const double* Lov = ch->Lov[k.tensor].p;
    const long ldw = ch->ldzt;                                   // pad_ld(no)
    const size_t per_p = (size_t)nvec * ch->no * ldw;
    long pc = (long)(h->scratch_doubles / per_p);
    XTD_REQUIRE(pc >= 1, XTD_ERR_NOMEM, "workspace too small for the transposed-exchange intermediate of one aux function");
    pc = std::min<long>(pc, naux);
    if (h->env.max_pc > 0) pc = std::min<long>(pc, h->env.max_pc);
    h->last_aux_chunks = std::max<long>(h->last_aux_chunks, cdiv(naux, pc));
    double* W = h->scratch;
    for (long P0 = 0; P0 < naux; P0 += pc) {
      const int pn = (int)std::min<long>(pc, naux - P0);
      {
        PhaseTimer t(h, XTD_T_K1);
        // rows (P, i) flattened; W[(P,i)][x][j]
        GemmDesc d;
        d.A = view2d(Lov + P0 * ch->no * ch->ldz, ch->ldz, pn * ch->no, ch->nv);
        d.B = view3d(h->Z[k.ch], ch->ldz, (long)ch->no * ch->ldz, nvec, ch->no, ch->nv);
        d.M = pn * ch->no; d.N = ch->no; d.K = ch->nv;
        d.batches = nvec; d.z_div = 1; d.a_hi = 0; d.b_hi = 1;
        d.C = W; d.ldc = (long)nvec * ldw; d.c_batch_stride = ldw;
        XTD_TRY(gemm(h->gemm, d, s));
      }
      {
        PhaseTimer t(h, XTD_T_K2);
        GemmDesc d;
        d.b_kc = false;
        d.A = view3d(W, ldw, (long)nvec * ch->no * ldw, pn, nvec * ch->no, ch->no);
        d.B = view3d(Lov, ch->ldz, (long)ch->no * ch->ldz, (int)(naux - P0), ch->no, ch->nv, 0, 0, (int)P0);
        d.M = nvec * ch->no; d.N = ch->nv; d.K = ch->no; d.nouter = pn;
        d.C = h->SIG + h->sig_base[k.ch]; d.ldc = ch->ldz; d.accumulate = true;
        d.c_row_div = nvec; d.c_row_hi = ch->ldz; d.c_row_lo = (long)ch->no * ch->ldz;
        d.alpha = k.w;
        XTD_TRY(gemm(h->gemm, d, s));
      }
    }
  }
  return XTD_OK;
}

static int run_j(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  const int njb = (int)h->jblocks.size();
  const long naux = h->naux[0];
  if (!njb || naux == 0) return XTD_OK;
  PhaseTimer t(h, XTD_T_J);
  const long nap = naux + (naux & 1);        // per-block row of the aux-space vectors, even for the GEMM route
  // A block that spans the full width of its channel is contiguous in (i, a) for every aux function and vector, so both
  // Coulomb steps are plain GEMMs over the flattened pair index (the streaming kernels re-read all trial vectors from L2
  // once per aux function); sub-blocks (XSF Delta A) keep the streaming kernels.
  auto flat = [&](const JBlockRec* j) {      // (the flattened pair index is the N dimension of the second GEMM: grid.y limit)
    return !h->env.j_stream && j->c0 == 0 && j->ld == h->ch[j->ch]->ldz && (long)j->nr * j->ld <= 65535L * 128;
  };
  for (int b = 0; b < njb; ++b) {
    JBlockRec* j = h->jblocks[b];
    Channel* ch = h->ch[j->ch];
    if (flat(j)) {
      // R[x][b][P] = sum_(i,a) Z[x][(r0+i, a)] L_b[P][(i, a)]
      GemmDesc d;
      d.A = view2d(h->Z[j->ch] + (long)j->r0 * ch->ldz, (long)ch->no * ch->ldz, nvec, (int)(j->nr * ch->ldz));
      d.B = view2d(j->L.p, (long)j->nr * j->ld, (int)naux, (int)(j->nr * j->ld));
      d.M = nvec; d.N = (int)naux; d.K = (int)(j->nr * ch->ldz);
      d.C = h->jR + (long)b * nap; d.ldc = (long)njb * nap;
      XTD_TRY(gemm(h->gemm, d, s));
    } else {
      j_rho_kernel<8><<<(unsigned)naux, 256, 0, s>>>(h->jR + (long)b * nap, (long)njb * nap, j->L.p, j->ld, (long)j->nr * j->ld,
                                                    h->Z[j->ch] + (long)j->r0 * ch->ldz + j->c0, ch->ldz, (long)ch->no * ch->ldz, j->nr, j->nc,
                                                    nvec);
      LAUNCH_CHECK();
    }
  }
  j_mix_kernel<<<dim3((unsigned)cdiv(naux, 128), nvec), 128, 0, s>>>(h->jRm, h->jR, h->jmix_dev.p, njb, naux, nap, nvec);
  LAUNCH_CHECK();
  for (int b = 0; b < njb; ++b) {
    JBlockRec* j = h->jblocks[b];
    Channel* ch = h->ch[j->ch];
    if (flat(j)) {
      // SIG[x][(r0+i, a)] += sum_P Rm[x][b][P] L_b[P][(i, a)]
      GemmDesc d;
      d.b_kc = false;
      d.A = view2d(h->jRm + (long)b * nap, (long)njb * nap, nvec, (int)naux);
      d.B = view2d(j->L.p, (long)j->nr * j->ld, (int)naux, (int)(j->nr * j->ld));
      d.M = nvec; d.N = (int)(j->nr * j->ld); d.K = (int)naux;
      d.C = h->SIG + h->sig_base[j->ch] + (long)j->r0 * ch->ldz; d.ldc = (long)ch->no * ch->ldz; d.accumulate = true;
      XTD_TRY(gemm(h->gemm, d, s));
    } else {
      j_apply_kernel<8><<<dim3((unsigned)cdiv((long)j->nr * j->nc, 256), (unsigned)cdiv(nvec, 8)), 256, 0, s>>>(
          h->SIG + h->sig_base[j->ch] + (long)j->r0 * ch->ldz + j->c0, ch->ldz, (long)ch->no * ch->ldz, j->L.p, j->ld, (long)j->nr * j->ld,
          h->jRm + (long)b * nap, (long)njb * nap, naux, j->nr, j->nc, nvec);
      LAUNCH_CHECK();
    }
  }
  return XTD_OK;
}

static int run_local(xtd_engine* h, int nvec) {
  cudaStream_t s = h->stream;
  PhaseTimer t(h, XTD_T_LOCAL);
  const bool batched = h->small_local && (h->lt_dev || h->ld_dev);
  if (batched) {
    LocalSmallArgs a;
    a.terms = h->lt_dev; a.nterms = (int)h->lgemms.size(); a.diags = h->ld_dev; a.ndiags = (int)h->diags.size();
    a.sig = h->SIG;
    long max_elems = 0;
    for (int c = 0; c < 2; ++c) {
      const bool on = c < (int)h->ch.size();
      a.z[c] = on ? h->Z[c] : nullptr; a.sig_base[c] = on ? h->sig_base[c] : 0; a.ldz[c] = on ? h->ch[c]->ldz : 0;
      a.vec_stride[c] = on ? (long)h->ch[c]->no * h->ch[c]->ldz : 0; a.no[c] = on ? h->ch[c]->no : 0; a.nv[c] = on ? h->ch[c]->nv : 0;
      if (on) max_elems = std::max<long>(max_elems, (long)h->ch[c]->no * h->ch[c]->nv);
    }
    local_small_kernel<<<dim3((unsigned)cdiv(max_elems, 128), nvec, (unsigned)h->ch.size()), 128, 0, s>>>(a);
    LAUNCH_CHECK();
  }
  for (auto* l : h->lgemms) {
    if (batched) break;
    Channel *dc = h->ch[l->dch], *sc = h->ch[l->sch];
    double* dst = h->SIG + h->sig_base[l->dch] + (long)l->r0 * dc->ldz + l->c0;
    GemmDesc d;
    d.alpha = l->alpha; d.accumulate = true; d.ldc = dc->ldz;
    if (l->side == XTD_SIDE_RIGHT) {
      const bool flat = (l->r0 == 0 && l->nr == dc->no && l->sr0 == 0 && sc->no == dc->no);
      d.b_kc = false;
      d.B = view2d(l->M.p, l->ldm, l->mrows, l->mcols);
      d.N = l->nc; d.K = l->mrows;
      if (flat) {
        d.A = view2d(h->Z[l->sch], sc->ldz, nvec * sc->no, l->mrows, 0, l->sc0);
        d.M = nvec * dc->no; d.C = dst;
      } else {
        d.A = view3d(h->Z[l->sch], sc->ldz, (long)sc->no * sc->ldz, nvec, l->nr, l->mrows, l->sr0, l->sc0);
        d.M = l->nr; d.batches = nvec; d.a_hi = 1; d.b_hi = 0; d.C = dst; d.c_batch_stride = (long)dc->no * dc->ldz;
      }
    } else if (l->side == XTD_SIDE_LEFT) {
      d.A = view2d(l->M.p, l->ldm, l->mrows, l->mcols);
      d.b_kc = false;
      d.B = view3d(h->Z[l->sch], sc->ldz, (long)sc->no * sc->ldz, nvec, l->mcols, l->nc, l->sr0, l->sc0);
      d.M = l->nr; d.N = l->nc; d.K = l->mcols; d.batches = nvec; d.a_hi = 0; d.b_hi = 1;
      d.C = dst; d.c_batch_stride = (long)dc->no * dc->ldz;
    } else if (l->side == XTD_SIDE_LEFT_T) {
      // dst[r][c] += alpha sum_k M[r][k] src[c][k]: the source block enters transposed (both operands K-contiguous)
      d.A = view2d(l->M.p, l->ldm, l->mrows, l->mcols);
      d.B = view3d(h->Z[l->sch], sc->ldz, (long)sc->no * sc->ldz, nvec, l->nc, l->mcols, l->sr0, l->sc0);
      d.M = l->nr; d.N = l->nc; d.K = l->mcols; d.batches = nvec; d.a_hi = 0; d.b_hi = 1;
      d.C = dst; d.c_batch_stride = (long)dc->no * dc->ldz;
    } else {
      // dst[r][c] += alpha sum_j src[j][r] M[j][c]: neither operand K-contiguous
      d.a_kc = false; d.b_kc = false;
      d.A = view3d(h->Z[l->sch], sc->ldz, (long)sc->no * sc->ldz, nvec, l->mrows, l->nr, l->sr0, l->sc0);
      d.B = view2d(l->M.p, l->ldm, l->mrows, l->mcols);
      d.M = l->nr; d.N = l->nc; d.K = l->mrows; d.batches = nvec; d.a_hi = 1; d.b_hi = 0;
      d.C = dst; d.c_batch_stride = (long)dc->no * dc->ldz;
    }
    XTD_TRY(gemm(h->gemm, d, s));
  }
  for (auto* r : h->rank1s) {
    Channel *dc = h->ch[r->dch], *sc = h->ch[r->sch];
    block_dot_kernel<<<nvec, 256, 0, s>>>(h->r1d, r->V.p, h->Z[r->sch], sc->ldz, (long)sc->no * sc->ldz, sc->no, sc->nv);
    LAUNCH_CHECK();
    block_axpy_kernel<<<dim3((unsigned)cdiv((long)dc->no * dc->nv, 256), nvec), 256, 0, s>>>(h->SIG + h->sig_base[r->dch], r->U.p, h->r1d,
                                                                                           dc->ldz, (long)dc->no * dc->ldz, dc->no, dc->nv);
    LAUNCH_CHECK();
  }
  for (auto* dg : h->diags) {
    if (batched) break;
    Channel* c = h->ch[dg->ch];
    block_diag_kernel<<<dim3((unsigned)cdiv((long)c->no * c->nv, 256), nvec), 256, 0, s>>>(h->SIG + h->sig_base[dg->ch], dg->D.p, h->Z[dg->ch],
                                                                                         c->ldz, (long)c->no * c->ldz, c->no, c->nv);
    LAUNCH_CHECK();
  }
  return XTD_OK;
}

extern "C" {

int xtd_sigma_partial(xtd_handle h, int nvec, const double* z_dev) {
  XTD_REQUIRE(h && h->finalized, XTD_ERR_STATE, "xtd_sigma before xtd_finalize");
  XTD_REQUIRE(nvec >= 1 && nvec <= h->max_nvec && z_dev, XTD_ERR_ARG, "xtd_sigma: nvec %d outside 1..%d", nvec, h->max_nvec);
  cudaStream_t s = h->stream;
  h->ev_used = 0;
  for (int i = 0; i < 12; ++i) h->phase_flops[i] = 0.0;
  h->last_aux_chunks = h->last_grid_chunks = 0;
  if (h->env.prof_phase == XTD_T_TOTAL && !h->capturing) cudaProfilerStart();
  if (h->ev_ok && !h->capturing) cudaEventRecord(h->ev_total[0], s);
  XTD_TRY(setup_call_buffers(h, nvec));
  long base[2], total;
  sig_layout(h, nvec, base, &total);
  {
    PhaseTimer t(h, XTD_T_PACK);
    XTD_CUDA(cudaMemsetAsync(h->SIG, 0, (size_t)total * 8, s));
    XTD_CUDA(cudaMemsetAsync(h->Z[0], 0, (size_t)total * 8, s));
    for (size_t c = 0; c < h->ch.size(); ++c) {
      Channel* ch = h->ch[c];
      const long nrows = (long)ch->no * ch->nv;
      const bool need_zt = !h->kterms.empty() || ch->xc_oz_split;
      if (need_zt && h->small_local) {
        // small problems: gather and transposed copy in one launch
        XTD_CUDA(cudaMemsetAsync(h->ZT[c], 0, (size_t)nvec * ch->nv * ch->ldzt * 8, s));
        pack_t_kernel<<<dim3((unsigned)cdiv(nrows, 256), nvec), 256, 0, s>>>(h->Z[c], ch->ldz, (long)ch->no * ch->ldz, h->ZT[c], ch->ldzt,
                                                                           (long)ch->nv * ch->ldzt, ch->nv, nrows, ch->g_indptr, ch->g_cols,
                                                                           ch->g_vals, z_dev, h->ext_dim, nvec);
        LAUNCH_CHECK();
        continue;
      }
      pack_kernel<<<dim3((unsigned)cdiv(nrows, 256), nvec), 256, 0, s>>>(h->Z[c], ch->ldz, (long)ch->no * ch->ldz, ch->nv, nrows, ch->g_indptr,
                                                                         ch->g_cols, ch->g_vals, z_dev, h->ext_dim, nvec);
      LAUNCH_CHECK();
      if (need_zt) {
        XTD_CUDA(cudaMemsetAsync(h->ZT[c], 0, (size_t)nvec * ch->nv * ch->ldzt * 8, s));
        transpose_kernel<<<dim3((unsigned)cdiv(ch->nv, 32), (unsigned)cdiv(ch->no, 32), nvec), dim3(32, 8), 0, s>>>(
            h->ZT[c], ch->ldzt, (long)ch->nv * ch->ldzt, h->Z[c], ch->ldz, (long)ch->no * ch->ldz, ch->no, ch->nv);
        LAUNCH_CHECK();
      }
    }
  }
  if (h->fxc_kind != XTD_FXC_NONE && h->ng > 0) XTD_TRY(run_xc(h, nvec));
  XTD_TRY(run_k(h, nvec));
  XTD_TRY(run_kt(h, nvec));
  XTD_TRY(run_j(h, nvec));
  return XTD_OK;
}

int xtd_partial_buffer(xtd_handle h, int nvec, double** ptr, long* nelem) {
  XTD_REQUIRE(h && h->finalized && h->cur_nvec == nvec, XTD_ERR_STATE, "xtd_partial_buffer: call xtd_sigma_partial(nvec) first");
  long base[2], total;
  sig_layout(h, nvec, base, &total);
  if (ptr) *ptr = h->SIG;
  if (nelem) *nelem = total;
  return XTD_OK;
}

int xtd_sigma_finish(xtd_handle h, int nvec, double* hz_dev) {
  XTD_REQUIRE(h && h->finalized && h->cur_nvec == nvec && hz_dev, XTD_ERR_STATE, "xtd_sigma_finish: call xtd_sigma_partial(nvec) first");
  cudaStream_t s = h->stream;
  XTD_TRY(run_local(h, nvec));
  {
    PhaseTimer t(h, XTD_T_UNPACK);
    UnpackChan uc;
    for (int c = 0; c < 2; ++c) {
      uc.base[c] = c < (int)h->ch.size() ? h->sig_base[c] : 0;
      uc.vec_stride[c] = c < (int)h->ch.size() ? (long)h->ch[c]->no * h->ch[c]->ldz : 0;
    }
    unpack_kernel<<<dim3((unsigned)cdiv(h->ext_dim, 256), nvec), 256, 0, s>>>(hz_dev, h->ext_dim, nvec, h->s_indptr, h->s_offs, h->s_chans,
                                                                             h->s_vals, h->SIG, uc);
    LAUNCH_CHECK();
  }
  if (h->ev_ok && !h->capturing) cudaEventRecord(h->ev_total[1], s);
  if (h->env.prof_phase == XTD_T_TOTAL && !h->capturing) cudaProfilerStop();
  return XTD_OK;
}

static int sigma_eager(xtd_handle h, int nvec, const double* z_dev, double* hz_dev) {
  XTD_TRY(xtd_sigma_partial(h, nvec, z_dev));
  return xtd_sigma_finish(h, nvec, hz_dev);
}

static int launch_graph(xtd_engine* h, const xtd_engine::GraphRec& g) {
  cudaStream_t s = h->stream;
  h->ev_used = 0;                                    // no per-phase events inside a graph: only the total is timed
  if (h->ev_ok) cudaEventRecord(h->ev_total[0], s);
  XTD_CUDA(cudaGraphLaunch(g.exec, s));
  if (h->ev_ok) cudaEventRecord(h->ev_total[1], s);
  for (int i = 0; i < 12; ++i) h->phase_flops[i] = g.phase_flops[i];
  XTD_TRY(setup_call_buffers(h, g.nvec));            // same (deterministic) arena layout the recorded call used: channel bases,
  return XTD_OK;                                     // Z / SIG pointers for xtd_partial_buffer / xtd_sigma_finish after a replay
}

int xtd_sigma(xtd_handle h, int nvec, const double* z_dev, double* hz_dev) {
  XTD_REQUIRE(h && h->finalized, XTD_ERR_STATE, "xtd_sigma before xtd_finalize");
  if (h->graphs_off || h->env.prof_phase >= 0) return sigma_eager(h, nvec, z_dev, hz_dev);
  for (const auto& g : h->graphs)
    if (g.nvec == nvec && g.z == z_dev && g.hz == hz_dev) {
      g_launch_count += g.launches;                  // the kernels of the recorded call run again
      h->gemm.flops += g.flops;
      return launch_graph(h, g);
    }
  // second call with the same arguments, and the first one was launch-bound: capture it
  const bool repeat = h->last_eager_nvec == nvec && h->last_eager_z == z_dev && h->last_eager_hz == hz_dev;
  if (repeat && h->last_eager_flops < 2e10 && h->graphs.size() < 64) {
    if (!h->cap_stream && cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess) h->cap_stream = nullptr;
    cudaStream_t s = h->cap_stream, user_stream = h->stream;
    const unsigned long long l0 = g_launch_count;
    const double f0 = h->gemm.flops;
    cudaGraph_t graph = nullptr;
    if (s && cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
      h->capturing = true;
      h->stream = s;
      const int rc = sigma_eager(h, nvec, z_dev, hz_dev);
      h->stream = user_stream;
      h->capturing = false;
      const cudaError_t ce = cudaStreamEndCapture(s, &graph);
      xtd_engine::GraphRec g;
      g.nvec = nvec; g.z = z_dev; g.hz = hz_dev; g.exec = nullptr;
      g.launches = g_launch_count - l0; g.flops = h->gemm.flops - f0;
      for (int i = 0; i < 12; ++i) g.phase_flops[i] = h->phase_flops[i];
      if (rc == XTD_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess) {
        cudaGraphDestroy(graph);
        h->graphs.push_back(g);
        return launch_graph(h, h->graphs.back());    // the capture recorded the work without running it: run it now
      }
      // capture not possible for this call: undo the bookkeeping, never try again, run eagerly
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      g_launch_count = l0; h->gemm.flops = f0;
      h->graphs_off = true;
    } else {
      cudaGetLastError();
      h->graphs_off = true;
    }
  }
  const double f0 = h->gemm.flops;
  const int rc = sigma_eager(h, nvec, z_dev, hz_dev);
  h->last_eager_nvec = nvec; h->last_eager_z = z_dev; h->last_eager_hz = hz_dev; h->last_eager_flops = h->gemm.flops - f0;
  return rc;
}

int xtd_sigma_host(xtd_handle h, int nvec, const double* z_host, double* hz_host) {
  XTD_REQUIRE(h && h->finalized && z_host && hz_host, XTD_ERR_ARG, "xtd_sigma_host: bad arguments");
  XTD_REQUIRE(nvec >= 1 && nvec <= h->max_nvec, XTD_ERR_ARG, "xtd_sigma_host: nvec %d outside 1..%d", nvec, h->max_nvec);
  const size_t n = (size_t)nvec * h->ext_dim;
  if (n > h->pin_doubles) {
    if (h->pin_in) cudaFreeHost(h->pin_in);
    if (h->pin_out) cudaFreeHost(h->pin_out);
    if (h->dev_in) cudaFree(h->dev_in);
    if (h->dev_out) cudaFree(h->dev_out);
    const size_t cap = (size_t)h->max_nvec * h->ext_dim;
    XTD_CUDA(cudaMallocHost((void**)&h->pin_in, cap * 8));
    XTD_CUDA(cudaMallocHost((void**)&h->pin_out, cap * 8));
    XTD_CUDA(cudaMalloc((void**)&h->dev_in, cap * 8));
    XTD_CUDA(cudaMalloc((void**)&h->dev_out, cap * 8));
    h->pin_doubles = cap;
  }
  memcpy(h->pin_in, z_host, n * 8);
  XTD_CUDA(cudaMemcpyAsync(h->dev_in, h->pin_in, n * 8, cudaMemcpyHostToDevice, h->stream));
  XTD_TRY(xtd_sigma(h, nvec, h->dev_in, h->dev_out));
  XTD_CUDA(cudaMemcpyAsync(h->pin_out, h->dev_out, n * 8, cudaMemcpyDeviceToHost, h->stream));
  XTD_CUDA(cudaStreamSynchronize(h->stream));
  memcpy(hz_host, h->pin_out, n * 8);
  return XTD_OK;
}

int xtd_get_stats(xtd_handle h, xtd_stats* out) {
  XTD_REQUIRE(h && out, XTD_ERR_ARG, "xtd_get_stats: bad arguments");
  XTD_CUDA(cudaStreamSynchronize(h->stream));
  out->flops_gemm = h->gemm.flops - h->flops0;
  out->launches = g_launch_count - h->launches0;
  for (int i = 0; i < 12; ++i) { out->ms[i] = 0.0; out->flops[i] = h->phase_flops[i]; }
  for (size_t i = 0; i < h->ev_used; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->evpool[i].a, h->evpool[i].b) == cudaSuccess) out->ms[h->evpool[i].id] += ms;
    else cudaGetLastError();
  }
  float tot = 0.f;
  if (cudaEventElapsedTime(&tot, h->ev_total[0], h->ev_total[1]) == cudaSuccess) out->ms[XTD_T_TOTAL] = tot;
  else cudaGetLastError();
  return XTD_OK;
}

int xtd_last_chunks(xtd_handle h, long* aux_chunks, long* grid_chunks) {
  XTD_REQUIRE(h, XTD_ERR_ARG, "null handle");
  if (aux_chunks) *aux_chunks = h->last_aux_chunks;
  if (grid_chunks) *grid_chunks = h->last_grid_chunks;
  return XTD_OK;
}

int xtd_xc_split_form(xtd_handle h, int nvec) {
  XTD_REQUIRE(h && h->finalized && nvec >= 1, XTD_ERR_STATE, "xtd_xc_split_form: finalize first");
  if (h->fxc_kind == XTD_FXC_NONE || h->ng == 0) return 0;
  return xc_use_split(h, nvec) ? 1 : 0;
}

int xtd_reset_stats(xtd_handle h) {
  XTD_REQUIRE(h, XTD_ERR_ARG, "null handle");
  h->flops0 = h->gemm.flops;
  h->launches0 = g_launch_count;
  return XTD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Davidson vector primitives
// ---------------------------------------------------------------------------------------------------------
int xtd_vec_dots(void* stream, double* g, int ldg, const double* a, long lda, int m, const double* b, long ldb, int k, long n) {
  if (m <= 0 || k <= 0) return XTD_OK;
  vec_dots_kernel<<<dim3(k, m), 512, 0, (cudaStream_t)stream>>>(g, ldg, a, lda, b, ldb, n);
  LAUNCH_CHECK();
  return XTD_OK;
}
int xtd_vec_lincomb(void* stream, double* y, long ldy, const double* x, long ldx, const double* c, int ldc, int m, int k, long n,
                    double beta) {
  if (m <= 0) return XTD_OK;
  vec_lincomb_kernel<8><<<dim3((unsigned)cdiv(n, 256), (unsigned)cdiv(m, 8)), 256, 0, (cudaStream_t)stream>>>(y, ldy, x, ldx, c, ldc, m, k, n,
                                                                                                         beta);
  LAUNCH_CHECK();
  return XTD_OK;
}
int xtd_vec_residual(void* stream, double* r, const double* ax, const double* x, long ld, const double* e, double* nrm2, int k, long n) {
  if (k <= 0) return XTD_OK;
  vec_residual_kernel<<<k, 512, 0, (cudaStream_t)stream>>>(r, ax, x, ld, e, nrm2, n);
  LAUNCH_CHECK();
  return XTD_OK;
}
int xtd_vec_precond(void* stream, double* x, long ld, const double* hdiag, const double* shift, double* nrm2, int k, long n) {
  if (k <= 0) return XTD_OK;
  vec_precond_kernel<<<k, 512, 0, (cudaStream_t)stream>>>(x, ld, hdiag, shift, nrm2, n);
  LAUNCH_CHECK();
  return XTD_OK;
}
int xtd_vec_scale(void* stream, double* x, long ld, const double* sc, int k, long n) {
  if (k <= 0) return XTD_OK;
  vec_scale_kernel<<<dim3((unsigned)cdiv(n, 256), k), 256, 0, (cudaStream_t)stream>>>(x, ld, sc, n);
  LAUNCH_CHECK();
  return XTD_OK;
}

int xtd_dgemm(void* stream, int m, int n, int k, double alpha, const double* a, long lda, int a_kc, const double* b, long ldb, int b_kc,
              double* c, long ldc, int accumulate) {
  static GemmContext ctxs[64];                 // one context + split-K workspace per device
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  GemmContext& ctx = ctxs[dev & 63];
  if (!ctx.encode) {
    double* ws = nullptr;
    XTD_TRY(gemm_context_init(ctx));
    XTD_CUDA(cudaMalloc((void**)&ws, (size_t)256 << 20));
    ctx.split_ws = ws; ctx.split_ws_bytes = (size_t)256 << 20;
  }
  GemmDesc d;
  d.a_kc = a_kc != 0; d.b_kc = b_kc != 0;
  d.A = d.a_kc ? view2d(a, lda, m, k) : view2d(a, lda, k, m);
  d.B = d.b_kc ? view2d(b, ldb, n, k) : view2d(b, ldb, k, n);
  d.M = m; d.N = n; d.K = k; d.C = c; d.ldc = ldc; d.alpha = alpha; d.accumulate = accumulate != 0;
  return gemm(ctx, d, (cudaStream_t)stream);
}

// Emulated-FP64 contraction on the INT8 tensor cores (ozaki.cuh), self-contained: slices both operands, runs the tcgen05 kernel,
// reduces the split partials.  Temporary buffers are allocated per call: a test / benchmark entry, not the engine path.
int xtd_ozaki_gemm(void* stream, int m, int n, int k, int nq, int slices, int group, const double* a_dev, long lda, long sqa,
                   const double* b_dev, long ldb, long sqb, double* c_dev, long ldc, double alpha, int accumulate, double* ms_out) {
  XTD_REQUIRE(m > 0 && n > 0 && k > 0 && nq > 0 && a_dev && b_dev && c_dev, XTD_ERR_ARG, "xtd_ozaki_gemm: bad arguments");
  XTD_REQUIRE(slices >= OZ_MIN_S && slices <= OZ_MAX_S, XTD_ERR_ARG, "xtd_ozaki_gemm: slices %d outside %d..%d", slices, OZ_MIN_S, OZ_MAX_S);
  if (group <= 0) group = std::min(4, oz_max_group(k, slices));
  XTD_REQUIRE(group >= 1 && group <= oz_max_group(k, slices), XTD_ERR_ARG, "xtd_ozaki_gemm: K = %d too long for one int32 group (max group %d)", k,
              oz_max_group(k, slices));
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 148;
  XTD_CUDA(cudaGetDevice(&dev));
  XTD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  OzShape sa, sb;
  sa.set(m, OZ_BM, k);
  sb.set(n, OZ_BN, k);
  const int ngroups = (int)cdiv(nq, group);
  const int splits = oz_choose_splits(sa.nrt * sb.nrt, ngroups, sms);
  int8_t *As = nullptr, *Bs = nullptr;
  double *sca = nullptr, *scb = nullptr, *W = nullptr;
  XTD_CUDA(cudaMalloc((void**)&As, sa.slice_bytes(nq, slices)));
  XTD_CUDA(cudaMalloc((void**)&Bs, sb.slice_bytes(nq, slices)));
  XTD_CUDA(cudaMalloc((void**)&sca, sa.scale_doubles(nq, group) * 8));
  XTD_CUDA(cudaMalloc((void**)&scb, sb.scale_doubles(nq, group) * 8));
  XTD_CUDA(cudaMalloc((void**)&W, (size_t)splits * sa.rows_pad * sb.rows_pad * 8));
  cudaEvent_t ev[4];
  for (auto& e : ev) cudaEventCreate(&e);
  int rc = XTD_OK;
  cudaEventRecord(ev[0], st);
  for (int q0 = 0; q0 < nq && rc == XTD_OK; q0 += 32768 / group * group) {     // grid.z limit of the slicing kernel
    const int qn = std::min(nq - q0, 32768 / group * group);
    rc = oz_slice(slices, As + sa.slice_bytes(q0, slices), sca + (size_t)(q0 / group) * sa.rows_pad, sa, a_dev + (long)q0 * sqa, lda, sqa, qn, group, st);
  }
  cudaEventRecord(ev[1], st);
  for (int q0 = 0; q0 < nq && rc == XTD_OK; q0 += 32768 / group * group) {
    const int qn = std::min(nq - q0, 32768 / group * group);
    rc = oz_slice(slices, Bs + sb.slice_bytes(q0, slices), scb + (size_t)(q0 / group) * sb.rows_pad, sb, b_dev + (long)q0 * sqb, ldb, sqb, qn, group, st);
  }
  cudaEventRecord(ev[2], st);
  if (rc == XTD_OK) {
    OzGemmParams p;
    p.A = As; p.B = Bs; p.sa = sca; p.sb = scb;
    p.nmt = sa.nrt; p.nnt = sb.nrt; p.nkb = sa.nkb; p.nq = nq; p.group = group; p.b_q0 = 0;
    p.Mpad = sa.rows_pad; p.Npad = sb.rows_pad; p.splits = splits; p.W = W; p.alpha = alpha;
    rc = oz_gemm(slices, p, st);
    if (rc == XTD_OK) {
      long nblk = cdiv((long)m * n, 256);
      reduce_splits_kernel<<<dim3((unsigned)(nblk > 4096 ? 4096 : nblk), 1), 256, 0, st>>>(c_dev, ldc, 0, W, sb.rows_pad, 0,
                                                                                          (long)sa.rows_pad * sb.rows_pad, splits, m, n,
                                                                                          accumulate ? 1 : 0, 0, 0, 0);
      XTD_COUNT_LAUNCH();
      if (cudaGetLastError() != cudaSuccess) rc = XTD_ERR_CUDA;
    }
  }
  cudaEventRecord(ev[3], st);
  cudaError_t se = cudaStreamSynchronize(st);
  if (se != cudaSuccess) { XTD_SET_ERR("xtd_ozaki_gemm: %s", cudaGetErrorString(se)); rc = XTD_ERR_CUDA; }
  if (ms_out && rc == XTD_OK)
    for (int i = 0; i < 3; ++i) {
      float t = 0.f;
      cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
      ms_out[i] = t;
    }
  for (auto& e : ev) cudaEventDestroy(e);
  cudaFree(As); cudaFree(Bs); cudaFree(sca); cudaFree(scb); cudaFree(W);
  return rc;
}

int xtd_dgemm_tn(void* stream, int m, int n, int k, double alpha, const double* a, long lda, const double* b, long ldb, double* c,
                 long ldc, int accumulate) {
  return xtd_dgemm(stream, m, n, k, alpha, a, lda, 1, b, ldb, 1, c, ldc, accumulate);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Davidson solver (host control flow in C++; algorithm of xtddft_b200/davidson.py / the reference's utils/Davidson.py:21-298)
// ---------------------------------------------------------------------------------------------------------
namespace {
struct DavBuf {
  double* d = nullptr;
  int alloc(size_t n) { XTD_CUDA(cudaMalloc((void**)&d, std::max<size_t>(n, 2) * 8)); return XTD_OK; }
  ~DavBuf() { if (d) cudaFree(d); }
};
struct DavPinned {
  double* p = nullptr;
  int alloc(size_t n) { XTD_CUDA(cudaMallocHost((void**)&p, std::max<size_t>(n, 2) * 8)); return XTD_OK; }
  ~DavPinned() { if (p) cudaFreeHost(p); }
};
}  // namespace

extern "C" int xtd_davidson(xtd_handle h, int nroots, const xtd_solver_opts* o, const double* hdiag_dev, const double* x0_dev, int n0,
                            double* e_host, double* x_dev, int* conv_host, int* ncycle, int* nsigma_out) {
  XTD_REQUIRE(h && h->finalized && o && hdiag_dev && x0_dev && e_host && x_dev && conv_host, XTD_ERR_ARG, "xtd_davidson: bad arguments");
  const long dim = h->ext_dim;
  XTD_REQUIRE(nroots >= 1 && nroots <= dim && n0 >= 1, XTD_ERR_ARG, "xtd_davidson: nroots %d / initial vectors %d", nroots, n0);
  cudaStream_t s = h->stream;
  const double tol = o->tol, toloose = o->tol_residual > 0.0 ? o->tol_residual : std::sqrt(o->tol), lindep = o->lindep;
  // nroots close to dim (core-valence-separated spaces): the subspace may grow to the whole space, so it never restarts and never
  // takes more new vectors than there are dimensions left
  const bool whole = (long)o->max_space + (nroots - 1) * 4 >= dim;
  const int max_space = (int)std::min<long>(o->max_space + (nroots - 1) * 4, dim);
  const int cap = max_space + nroots + 40;
  const int nxt = std::max(std::max(n0, nroots), 40);
  DavBuf xs, ax, xt, axt, ritz, aritz, tmp, gdev, cdev, ndev, sdev;
  XTD_TRY(xs.alloc((size_t)cap * dim)); XTD_TRY(ax.alloc((size_t)cap * dim)); XTD_TRY(xt.alloc((size_t)nxt * dim));
  XTD_TRY(ritz.alloc((size_t)nroots * dim)); XTD_TRY(aritz.alloc((size_t)nroots * dim)); XTD_TRY(tmp.alloc((size_t)nxt * dim));
  XTD_TRY(axt.alloc((size_t)nxt * dim));       // sigma lands in a FIXED buffer: (nvec, z, hz) then repeat and the call replays as a CUDA graph
  XTD_TRY(gdev.alloc((size_t)cap * cap)); XTD_TRY(cdev.alloc((size_t)cap * cap)); XTD_TRY(ndev.alloc(cap)); XTD_TRY(sdev.alloc(cap));
  DavPinned gh;
  XTD_TRY(gh.alloc((size_t)cap * cap));
  XTD_CUDA(cudaMemcpyAsync(xt.d, x0_dev, (size_t)n0 * dim * 8, cudaMemcpyDeviceToDevice, s));
  int nt = n0;

  auto rows = [&](DavBuf& b, long r) { return b.d + r * dim; };
  auto fetch = [&](const double* dev, size_t n) -> int {          // device -> pinned host, synchronous
    XTD_CUDA(cudaMemcpyAsync(gh.p, dev, n * 8, cudaMemcpyDeviceToHost, s));
    XTD_CUDA(cudaStreamSynchronize(s));
    return XTD_OK;
  };
  auto dots = [&](const double* a, int m, const double* b, int k) -> int {      // gh.p[m][k] = <a_i, b_j>
    XTD_TRY(xtd_vec_dots(s, gdev.d, k, a, dim, m, b, dim, k, dim));
    return fetch(gdev.d, (size_t)m * k);
  };
  auto lincomb = [&](double* y, const double* x, const double* c_host, int m, int k, double beta) -> int {
    XTD_CUDA(cudaMemcpyAsync(cdev.d, c_host, (size_t)m * std::max(k, 1) * 8, cudaMemcpyHostToDevice, s));
    // (c_host is overwritten only after a later synchronising fetch, or is a live vector: the pageable copy is staged at once)
    return xtd_vec_lincomb(s, y, dim, x, dim, cdev.d, std::max(k, 1), m, k, dim, beta);
  };
  auto transform = [&](double* work, int n_in, const std::vector<double>& t, int n_out) -> int {      // work[:n_out] = t work[:n_in]
    if (n_out == 0) return XTD_OK;
    XTD_TRY(lincomb(tmp.d, work, t.data(), n_out, n_in, 0.0));
    XTD_CUDA(cudaMemcpyAsync(work, tmp.d, (size_t)n_out * dim * 8, cudaMemcpyDeviceToDevice, s));
    return XTD_OK;
  };
  std::vector<double> tco;
  auto orthonormalise = [&](double* work, int n_in, int* n_out) -> int {
    int nv = n_in;
    for (int it = 0; it < 2 && nv > 0; ++it) {
      XTD_TRY(dots(work, nv, work, nv));
      const int nk = gs_coefficients(gh.p, nv, lindep, tco);
      XTD_TRY(transform(work, nv, tco, nk));
      nv = nk;
    }
    *n_out = nv;
    return XTD_OK;
  };
  auto sigma = [&](const double* z, double* hz, int n) -> int {
    for (int x0 = 0; x0 < n; x0 += h->max_nvec) {
      const int nx = std::min(h->max_nvec, n - x0);
      if (!o->allreduce) {
        XTD_TRY(xtd_sigma(h, nx, z + (long)x0 * dim, hz + (long)x0 * dim));
      } else {
        XTD_TRY(xtd_sigma_partial(h, nx, z + (long)x0 * dim));
        double* part = nullptr;
        long np_ = 0;
        XTD_TRY(xtd_partial_buffer(h, nx, &part, &np_));
        XTD_REQUIRE(o->allreduce(o->allreduce_ctx, part, np_) == 0, XTD_ERR_CUDA, "xtd_davidson: the all-reduce callback failed");
        XTD_TRY(xtd_sigma_finish(h, nx, hz + (long)x0 * dim));
      }
    }
    return XTD_OK;
  };

  std::vector<double> heff((size_t)cap * cap, 0.0), hsub, w, e, elast, v, vlast, de, dxn, sel;
  std::vector<char> conv, conv_last;
  bool fresh = true, xt_orth = false;
  int space = 0, nsigma = 0, nritz = 0, icyc = 0, vrows = 0, vlast_rows = 0;
  for (icyc = 0; icyc < o->max_cycle; ++icyc) {
    if (fresh) {
      space = 0;
      XTD_TRY(orthonormalise(xt.d, nt, &nt));
      XTD_REQUIRE(nt > 0, XTD_ERR_ARG, "xtd_davidson: %s", icyc == 0 ? "initial guess is empty or zero" : "no more linearly independent basis vectors");
    } else if (nt > 1 && !xt_orth) {
      XTD_TRY(orthonormalise(xt.d, nt, &nt));
      nt = std::min(nt, 40);
    }
    xt_orth = false;
    XTD_REQUIRE(nt > 0, XTD_ERR_ARG, "xtd_davidson: no linearly independent basis found");
    XTD_REQUIRE(space + nt <= cap, XTD_ERR_STATE, "xtd_davidson: subspace overflow");
    XTD_TRY(sigma(xt.d, axt.d, nt));
    XTD_CUDA(cudaMemcpyAsync(rows(ax, space), axt.d, (size_t)nt * dim * 8, cudaMemcpyDeviceToDevice, s));
    XTD_CUDA(cudaMemcpyAsync(rows(xs, space), xt.d, (size_t)nt * dim * 8, cudaMemcpyDeviceToDevice, s));
    nsigma += nt;
    const int head = space;
    space += nt;
    elast = e; vlast = v; vlast_rows = vrows; conv_last = conv;
    // projected matrix: new rows / columns from one Gram product
    XTD_TRY(dots(rows(xs, head), nt, ax.d, space));
    for (int ip = 0; ip < nt; ++ip) {
      for (int jp = 0; jp < ip; ++jp) heff[(size_t)(head + ip) * cap + head + jp] = heff[(size_t)(head + jp) * cap + head + ip] = gh.p[(size_t)ip * space + head + jp];
      heff[(size_t)(head + ip) * cap + head + ip] = gh.p[(size_t)ip * space + head + ip];
      for (int j = 0; j < head; ++j) heff[(size_t)(head + ip) * cap + j] = heff[(size_t)j * cap + head + ip] = gh.p[(size_t)ip * space + j];
    }
    hsub.assign((size_t)space * space, 0.0);
    for (int i = 0; i < space; ++i)
      for (int j = 0; j < space; ++j) hsub[(size_t)i * space + j] = heff[(size_t)i * cap + j];
    XTD_REQUIRE(sym_eig(hsub, space, w) == 0, XTD_ERR_STATE, "xtd_davidson: the projected eigenproblem did not converge");
    // pick: positive eigenvalues only (XTDA.py:769-772), then the lowest nroots
    std::vector<int> idx;
    for (int k = 0; k < space; ++k)
      if (!o->pick_positive || w[k] > 1e-3) idx.push_back(k);
    XTD_REQUIRE(!idx.empty(), XTD_ERR_STATE, "xtd_davidson: not enough eigenvalues");
    nritz = std::min<int>(nroots, (int)idx.size());
    e.assign(nritz, 0.0);
    v.assign((size_t)space * nritz, 0.0);
    vrows = space;
    for (int k = 0; k < nritz; ++k) {
      e[k] = w[idx[k]];
      for (int r = 0; r < space; ++r) v[(size_t)r * nritz + k] = hsub[(size_t)r * space + idx[k]];
    }
    conv.assign(nritz, 0);
    if (!fresh && !elast.empty()) {
      // `_sort_elast`: match the previous roots to the new ones by the overlap of their subspace coefficients
      const int nprev = (int)elast.size();
      std::vector<double> e2(nritz, 0.0);
      std::vector<char> c2(nritz, 0);
      for (int k = 0; k < nritz; ++k) {
        int best = 0;
        double bo = -1.0;
        bool found = false;
        for (int q = 0; q < nprev; ++q) {
          double ov = 0.0;
          for (int r = 0; r < vlast_rows; ++r) ov += v[(size_t)r * nritz + k] * vlast[(size_t)r * nprev + q];
          ov = std::fabs(ov);
          if (ov > bo) { bo = ov; best = q; }
          if (ov > 0.5) found = true;
        }
        e2[k] = found ? elast[best] : 0.0;
        c2[k] = found ? conv_last[best] : 0;
      }
      elast = e2; conv_last = c2;
    }
    de.assign(nritz, 0.0);
    for (int k = 0; k < nritz; ++k) de[k] = ((int)elast.size() == nritz) ? e[k] - elast[k] : e[k];
    // Ritz vectors, their images, residuals
    {
      std::vector<double> vt((size_t)nritz * space);
      for (int k = 0; k < nritz; ++k)
        for (int r = 0; r < space; ++r) vt[(size_t)k * space + r] = v[(size_t)r * nritz + k];
      XTD_TRY(lincomb(ritz.d, xs.d, vt.data(), nritz, space, 0.0));
      XTD_CUDA(cudaStreamSynchronize(s));                 // vt is reused by the second upload
      XTD_TRY(lincomb(aritz.d, ax.d, vt.data(), nritz, space, 0.0));
      XTD_CUDA(cudaMemcpyAsync(sdev.d, e.data(), (size_t)nritz * 8, cudaMemcpyHostToDevice, s));
      XTD_TRY(xtd_vec_residual(s, xt.d, aritz.d, ritz.d, dim, sdev.d, ndev.d, nritz, dim));
      XTD_TRY(fetch(ndev.d, nritz));
    }
    dxn.assign(nritz, 0.0);
    bool all_conv = true;
    for (int k = 0; k < nritz; ++k) {
      dxn[k] = std::sqrt(gh.p[k]);
      conv[k] = (std::fabs(de[k]) < tol && dxn[k] < toloose) ? 1 : 0;
      all_conv = all_conv && conv[k];
    }
    if (all_conv) { ++icyc; break; }
    // precondition the unconverged residuals, normalise, project against the subspace, drop dependent ones
    std::vector<int> keep;
    for (int k = 0; k < nritz; ++k)
      if (!conv[k] && dxn[k] * dxn[k] > lindep) keep.push_back(k);
    for (size_t dst = 0; dst < keep.size(); ++dst)
      if ((int)dst != keep[dst]) XTD_CUDA(cudaMemcpyAsync(rows(xt, (long)dst), rows(xt, keep[dst]), (size_t)dim * 8, cudaMemcpyDeviceToDevice, s));
    nt = (int)keep.size();
    if (nt) {
      std::vector<double> shift(nt, e[0] - o->level_shift);
      XTD_CUDA(cudaMemcpyAsync(sdev.d, shift.data(), (size_t)nt * 8, cudaMemcpyHostToDevice, s));
      XTD_CUDA(cudaStreamSynchronize(s));
      XTD_TRY(xtd_vec_precond(s, xt.d, dim, hdiag_dev, sdev.d, ndev.d, nt, dim));
      dav_rsqrt_kernel<<<1, 64, 0, s>>>(ndev.d, ndev.d, nt);
      LAUNCH_CHECK();
      XTD_TRY(xtd_vec_scale(s, xt.d, dim, ndev.d, nt, dim));
      XTD_TRY(xtd_vec_dots(s, gdev.d, space, xt.d, dim, nt, xs.d, dim, space, dim));
      dav_negate_kernel<<<(unsigned)cdiv((long)nt * space, 256), 256, 0, s>>>(gdev.d, (long)nt * space);
      LAUNCH_CHECK();
      XTD_TRY(xtd_vec_lincomb(s, xt.d, dim, xs.d, dim, gdev.d, space, nt, space, dim, 1.0));
      // one Gram matrix: `_normalize_xt_` filter (diagonal), normalisation, first Gram-Schmidt pass of the next cycle's `_qr`
      XTD_TRY(dots(xt.d, nt, xt.d, nt));
      std::vector<int> good;
      for (int k = 0; k < nt; ++k)
        if (gh.p[(size_t)k * nt + k] > lindep) good.push_back(k);
      const int ng = (int)good.size();
      if (ng) {
        std::vector<double> inv(ng);
        for (int a = 0; a < ng; ++a) inv[a] = 1.0 / std::sqrt(gh.p[(size_t)good[a] * nt + good[a]]);
        const bool will_restart = space + nroots > max_space && !whole;
        if (ng > 1 && !will_restart) {
          std::vector<double> gs((size_t)ng * ng);
          for (int a = 0; a < ng; ++a)
            for (int b = 0; b < ng; ++b) gs[(size_t)a * ng + b] = gh.p[(size_t)good[a] * nt + good[b]] * inv[a] * inv[b];
          std::vector<double> t1;
          const int n1 = gs_coefficients(gs.data(), ng, lindep, t1);
          sel.assign((size_t)n1 * nt, 0.0);                 // t1 composed with the selection / normalisation
          for (int r = 0; r < n1; ++r)
            for (int a = 0; a < ng; ++a) sel[(size_t)r * nt + good[a]] = t1[(size_t)r * ng + a] * inv[a];
          XTD_TRY(transform(xt.d, nt, sel, n1));
          XTD_CUDA(cudaStreamSynchronize(s));
          nt = n1;
          if (nt > 1) {
            XTD_TRY(dots(xt.d, nt, xt.d, nt));
            const int n2 = gs_coefficients(gh.p, nt, lindep, tco);
            XTD_TRY(transform(xt.d, nt, tco, n2));
            XTD_CUDA(cudaStreamSynchronize(s));
            nt = n2;
          }
          nt = std::min(nt, 40);
          xt_orth = true;
        } else {
          sel.assign((size_t)ng * nt, 0.0);
          for (int a = 0; a < ng; ++a) sel[(size_t)a * nt + good[a]] = inv[a];
          XTD_TRY(transform(xt.d, nt, sel, ng));
          XTD_CUDA(cudaStreamSynchronize(s));
          nt = ng;
        }
      } else {
        nt = 0;
      }
    }
    if (whole) nt = (int)std::min<long>(nt, dim - space);
    if (nt == 0) {
      for (int k = 0; k < nritz; ++k) conv[k] = dxn[k] < toloose ? 1 : 0;
      ++icyc;
      break;
    }
    fresh = space + nroots > max_space && !whole;
    if (fresh) {
      XTD_CUDA(cudaMemcpyAsync(xt.d, ritz.d, (size_t)nritz * dim * 8, cudaMemcpyDeviceToDevice, s));
      nt = nritz;
    }
  }
  for (int k = 0; k < nroots; ++k) {
    e_host[k] = k < nritz ? e[k] : 0.0;
    conv_host[k] = k < nritz ? (int)conv[k] : 0;
  }
  XTD_CUDA(cudaMemcpyAsync(x_dev, ritz.d, (size_t)nritz * dim * 8, cudaMemcpyDeviceToDevice, s));
  XTD_CUDA(cudaStreamSynchronize(s));
  if (ncycle) *ncycle = std::min(icyc, o->max_cycle);
  if (nsigma_out) *nsigma_out = nsigma;
  return nritz;
}

// Host-only pieces of the native solver, exported so the CPU test suite can hold them to NumPy (no device needed):
// symmetric eigenproblem (a[n][n] row-major in, eigenvectors in columns out, w ascending) and the Gram-Schmidt coefficients.
extern "C" int xtd_host_sym_eig(double* a, int n, double* w) {
  XTD_REQUIRE(a && w && n >= 1, XTD_ERR_ARG, "xtd_host_sym_eig: bad arguments");
  std::vector<double> m(a, a + (size_t)n * n), ev;
  XTD_REQUIRE(sym_eig(m, n, ev) == 0, XTD_ERR_STATE, "xtd_host_sym_eig: no convergence");
  std::copy(m.begin(), m.end(), a);
  std::copy(ev.begin(), ev.end(), w);
  return XTD_OK;
}
extern "C" int xtd_host_gs_coefficients(const double* g, int n, double lindep, double* t_out) {
  XTD_REQUIRE(g && t_out && n >= 1, XTD_ERR_ARG, "xtd_host_gs_coefficients: bad arguments");
  std::vector<double> t;
  const int nk = gs_coefficients(g, n, lindep, t);
  std::copy(t.begin(), t.end(), t_out);
  return nk;
}

// ---------------------------------------------------------------------------------------------------------
// Response of symmetric MO-block densities on the resident blocks (xtd_block_response): the right-hand side and the W matrix of
// the Z-vector equation.  Per channel c the density D_c has an occupied-occupied block, a virtual-virtual block and an
// occupied-virtual block (the virtual-occupied one is its transpose); the outputs are the occupied-occupied and occupied-virtual
// blocks of  c_J J[D_0 + D_1] + c_xc f_xc[D_c] + sum_t c_K[t] K_t[D_c].  With L[P] = [[Loo, Lov], [Lvo, Lvv]] per aux function:
//   A[P] = Loo Doo + Lov Dov^T,  B[P] = Loo Dov + Lov Dvv       K_oo = sum_P A Loo + B Lov^T,   K_ov = sum_P A Lov + B Lvv
// ---------------------------------------------------------------------------------------------------------
namespace {

// occupied-virtual block of `tensor` in channel ci: the transposed-density exchange copy, or a full-channel Coulomb block
const double* ov_block(const xtd_engine* h, int ci, int tensor, long* ld) {
  const Channel* c = h->ch[ci];
  if (c->need_kt[tensor]) { *ld = c->ldz; return c->Lov[tensor].p; }
  if (tensor == 0)
    for (auto* j : h->jblocks)
      if (j->ch == ci && j->r0 == 0 && j->nr == c->no && j->c0 == 0 && j->nc == c->nv) { *ld = j->ld; return j->L.p; }
  return nullptr;
}

int mm(xtd_engine* h, const MatView& A, bool akc, const MatView& B, bool bkc, int M, int N, int K, int nouter, int batches, double* Cp,
       long ldc, long cbs, double alpha, bool acc) {
  GemmDesc d;
  d.A = A; d.B = B; d.a_kc = akc; d.b_kc = bkc; d.M = M; d.N = N; d.K = K; d.nouter = nouter;
  d.batches = batches; d.z_div = 1; d.a_hi = batches > 1 ? 1 : 0; d.b_hi = 0;
  d.C = Cp; d.ldc = ldc; d.c_batch_stride = cbs; d.alpha = alpha; d.accumulate = acc;
  return gemm(h->gemm, d, h->stream);
}

struct BlockBufs {
  double *Doo, *Dvv, *Dov, *Ooo, *Oov;
};

int block_response_df(xtd_engine* h, const BlockBufs* bb, const double* coef, const double* X, double* const* XO, double* scratch,
                      size_t scratch_doubles) {
  cudaStream_t s = h->stream;
  const double cj = coef[0], cx = coef[4];
  for (int t = 0; t < 2; ++t) {
    const double ck = coef[1 + t];
    const bool doJ = t == 0 && cj != 0.0, doK = ck != 0.0, doX = t == 0 && X && cx != 0.0;
    if (!(doJ || doK || doX) || h->naux[t] == 0) continue;
    const long naux = h->naux[t];
    const double* Lov[2];
    long ldov[2];
    size_t per_p = 8;
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      Lov[ci] = ov_block(h, ci, t, &ldov[ci]);
      XTD_REQUIRE(oovv_resident(h, c, t) && Lov[ci], XTD_ERR_STATE,
                  "xtd_block_response: channel %d holds no MO blocks of tensor %d (call xtd_enable_block_response before xtd_df_begin)", ci, t);
      XTD_REQUIRE(!c->use_oz[t] || c->oz_col0[t] == 0, XTD_ERR_UNSUPPORTED, "xtd_block_response: block-weighted emulated exchange image");
      per_p += (size_t)c->no * c->ldoo + (size_t)c->no * c->ldz + (c->use_oz[t] ? (size_t)c->nv * c->ldvv : 0);
    }
    Channel *c0 = h->ch[0], *c1 = h->ch[1];
    if (doX) per_p += (size_t)c1->no * c0->ldz + (size_t)c1->nv * c0->ldz;
    long pc = (long)(scratch_doubles / (per_p + 64));
    if (h->env.max_pc > 0) pc = std::min<long>(pc, h->env.max_pc);
    pc = std::min<long>(pc, naux);
    XTD_REQUIRE(pc >= 1, XTD_ERR_NOMEM, "xtd_block_response: workspace too small for one aux function (%zu doubles)", per_p);
    double* cur = scratch;
    auto take = [&](size_t n) { double* p = cur; cur += (n + 31) & ~(size_t)31; return p; };
    double *Ab[2], *Bb[2], *Ldec[2] = {nullptr, nullptr};
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      Ab[ci] = take((size_t)pc * c->no * c->ldoo);
      Bb[ci] = take((size_t)pc * c->no * c->ldz);
      if (c->use_oz[t]) Ldec[ci] = take((size_t)pc * c->nv * c->ldvv);
    }
    double* U = doX ? take((size_t)pc * c1->no * c0->ldz) : nullptr;
    double* V = doX ? take((size_t)pc * c1->nv * c0->ldz) : nullptr;
    double* R = take((size_t)6 * pc);
    double* rho = take((size_t)pc);
    h->last_aux_chunks = std::max<long>(h->last_aux_chunks, cdiv(naux, pc));
    for (long P0 = 0; P0 < naux; P0 += pc) {
      const int pn = (int)std::min<long>(pc, naux - P0);
      const double *Loo[2], *Lvv[2], *Lo[2];
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        Loo[ci] = c->Loo[t].p + P0 * c->no * c->ldoo;
        Lo[ci] = Lov[ci] + P0 * c->no * ldov[ci];
        if (c->use_oz[t]) {
          PhaseTimer tm(h, XTD_T_K2_SLICE);
          oz_unslice_b_kernel<<<dim3((unsigned)cdiv((long)c->nv * c->nv, 256), pn), 256, 0, s>>>(
              Ldec[ci], c->ldvv, (long)c->nv * c->ldvv, c->LvvS[t], c->LvvScale[t], h->oz_slices, c->nv, c->ozB.rows_pad, c->nv, c->ozB.nkb,
              c->oz_group, P0, pn);
          LAUNCH_CHECK();
          Lvv[ci] = Ldec[ci];
        } else {
          Lvv[ci] = c->Lvv[t].p + P0 * c->nv * c->ldvv;
        }
      }
      if (doJ) {
        PhaseTimer tm(h, XTD_T_J);
        // rho_P = sum_c <Loo, Doo> + <Lvv, Dvv> + 2 <Lov, Dov>;  Ooo += c_J sum_P rho_P Loo[P],  Oov += c_J sum_P rho_P Lov[P]
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          j_rho_kernel<1><<<pn, 256, 0, s>>>(R + (3 * ci) * pc, 0, Loo[ci], c->ldoo, (long)c->no * c->ldoo, bb[ci].Doo, c->ldoo, 0, c->no, c->no, 1);
          LAUNCH_CHECK();
          j_rho_kernel<1><<<pn, 256, 0, s>>>(R + (3 * ci + 1) * pc, 0, Lvv[ci], c->ldvv, (long)c->nv * c->ldvv, bb[ci].Dvv, c->ldvv, 0, c->nv, c->nv, 1);
          LAUNCH_CHECK();
          j_rho_kernel<1><<<pn, 256, 0, s>>>(R + (3 * ci + 2) * pc, 0, Lo[ci], ldov[ci], (long)c->no * ldov[ci], bb[ci].Dov, c->ldz, 0, c->no, c->nv, 1);
          LAUNCH_CHECK();
        }
        RhoWeights w = {{cj, cj, 2.0 * cj, cj, cj, 2.0 * cj}};
        rho_combine_kernel<<<grid1d(pn, 256), 256, 0, s>>>(rho, R, pc, 6, pn, w);
        LAUNCH_CHECK();
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          j_apply_kernel<1><<<dim3((unsigned)cdiv((long)c->no * c->no, 256), 1), 256, 0, s>>>(bb[ci].Ooo, c->ldoo, 0, Loo[ci], c->ldoo,
                                                                                           (long)c->no * c->ldoo, rho, 0, pn, c->no, c->no, 1);
          LAUNCH_CHECK();
          j_apply_kernel<1><<<dim3((unsigned)cdiv((long)c->no * c->nv, 256), 1), 256, 0, s>>>(bb[ci].Oov, c->ldz, 0, Lo[ci], ldov[ci],
                                                                                           (long)c->no * ldov[ci], rho, 0, pn, c->no, c->nv, 1);
          LAUNCH_CHECK();
        }
      }
      if (doK)
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          const int no = c->no, nv = c->nv;
          const long soo = (long)no * c->ldoo, sov = (long)no * ldov[ci], svv = (long)nv * c->ldvv, sA = (long)no * c->ldoo, sB = (long)no * c->ldz;
          {
            PhaseTimer tm(h, XTD_T_K1);
            XTD_TRY(mm(h, view3d(Loo[ci], c->ldoo, soo, pn, no, no), true, view2d(bb[ci].Doo, c->ldoo, no, no), false, no, no, no, 1, pn, Ab[ci], c->ldoo, sA, 1.0, false));
            XTD_TRY(mm(h, view3d(Lo[ci], ldov[ci], sov, pn, no, nv), true, view2d(bb[ci].Dov, c->ldz, no, nv), true, no, no, nv, 1, pn, Ab[ci], c->ldoo, sA, 1.0, true));
            XTD_TRY(mm(h, view3d(Loo[ci], c->ldoo, soo, pn, no, no), true, view2d(bb[ci].Dov, c->ldz, no, nv), false, no, nv, no, 1, pn, Bb[ci], c->ldz, sB, 1.0, false));
            XTD_TRY(mm(h, view3d(Lo[ci], ldov[ci], sov, pn, no, nv), true, view2d(bb[ci].Dvv, c->ldvv, nv, nv), false, no, nv, nv, 1, pn, Bb[ci], c->ldz, sB, 1.0, true));
          }
          PhaseTimer tm(h, XTD_T_K2);
          const MatView Av = view3d(Ab[ci], c->ldoo, sA, pn, no, no), Bv = view3d(Bb[ci], c->ldz, sB, pn, no, nv);
          XTD_TRY(mm(h, Av, true, view3d(Loo[ci], c->ldoo, soo, pn, no, no), false, no, no, no, pn, 1, bb[ci].Ooo, c->ldoo, 0, ck, true));
          XTD_TRY(mm(h, Bv, true, view3d(Lo[ci], ldov[ci], sov, pn, no, nv), true, no, no, nv, pn, 1, bb[ci].Ooo, c->ldoo, 0, ck, true));
          XTD_TRY(mm(h, Av, true, view3d(Lo[ci], ldov[ci], sov, pn, no, nv), false, no, nv, no, pn, 1, bb[ci].Oov, c->ldz, 0, ck, true));
          XTD_TRY(mm(h, Bv, true, view3d(Lvv[ci], c->ldvv, svv, pn, nv, nv), false, no, nv, nv, pn, 1, bb[ci].Oov, c->ldz, 0, ck, true));
        }
      if (doX) {
        // mixed-spin K[X], X on (channel-1 occupied) x (channel-0 virtual):  U[P] = Loo1 X,  V[P] = Lov1^T X
        //   XO_oo += c_X sum_P U Lov0^T,  XO_ov += c_X sum_P U Lvv0,  XO_vo += c_X sum_P V Lov0^T,  XO_vv += c_X sum_P V Lvv0
        const int no1 = c1->no, nv1 = c1->nv, no0 = c0->no, nv0 = c0->nv;
        const long sU = (long)no1 * c0->ldz, sV = (long)nv1 * c0->ldz, sov0 = (long)no0 * ldov[0], svv0 = (long)nv0 * c0->ldvv;
        {
          PhaseTimer tm(h, XTD_T_K1);
          XTD_TRY(mm(h, view3d(Loo[1], c1->ldoo, (long)no1 * c1->ldoo, pn, no1, no1), true, view2d(X, c0->ldz, no1, nv0), false, no1, nv0, no1, 1, pn, U,
                     c0->ldz, sU, 1.0, false));
          XTD_TRY(mm(h, view3d(Lo[1], ldov[1], (long)no1 * ldov[1], pn, no1, nv1), false, view2d(X, c0->ldz, no1, nv0), false, nv1, nv0, no1, 1, pn, V,
                     c0->ldz, sV, 1.0, false));
        }
        PhaseTimer tm(h, XTD_T_K2);
        const MatView Uv = view3d(U, c0->ldz, sU, pn, no1, nv0), Vv = view3d(V, c0->ldz, sV, pn, nv1, nv0);
        const MatView Lov0 = view3d(Lo[0], ldov[0], sov0, pn, no0, nv0), Lvv0 = view3d(Lvv[0], c0->ldvv, svv0, pn, nv0, nv0);
        XTD_TRY(mm(h, Uv, true, Lov0, true, no1, no0, nv0, pn, 1, XO[0], c0->ldoo, 0, cx, true));
        XTD_TRY(mm(h, Uv, true, Lvv0, false, no1, nv0, nv0, pn, 1, XO[1], c0->ldz, 0, cx, true));
        XTD_TRY(mm(h, Vv, true, Lov0, true, nv1, no0, nv0, pn, 1, XO[2], c0->ldoo, 0, cx, true));
        XTD_TRY(mm(h, Vv, true, Lvv0, false, nv1, nv0, nv0, pn, 1, XO[3], c0->ldz, 0, cx, true));
      }
    }
  }
  return XTD_OK;
}

// grid term: Wo = phi Doo + phiv Dov^T, Wv = phiv Dvv + phi Dov (value component; all four with tau), xc_block_weight_kernel,
// then Ooo += c_xc sum_c Bo_c^T phi_c, Oov += c_xc sum_c Bo_c^T phiv_c
int block_response_xc(xtd_engine* h, const BlockBufs* bb, double cxc, double* scratch, size_t scratch_doubles) {
  cudaStream_t s = h->stream;
  XTD_REQUIRE(h->fxc_kind == XTD_FXC_UKS, XTD_ERR_UNSUPPORTED, "xtd_block_response: the grid term needs the UKS kernel tables");
  const int nve = h->nvar_eff, nf = h->tau ? 4 : 1;
  size_t per_g = 0;
  for (auto* c : h->ch) {
    XTD_REQUIRE(c->phiv.p && c->phi.p, XTD_ERR_STATE,
                "xtd_block_response: fp64 virtual MO values not kept on the grid (call xtd_enable_block_response before the grid commit)");
    per_g += (size_t)nve * (c->ldoo + c->ldvv);
  }
  long GB = (long)(scratch_doubles / per_g) - 64;
  GB = std::min<long>(GB, 1 << 16);
  if (h->env.max_gb > 0) GB = std::min<long>(GB, std::max<long>(h->env.max_gb, 128));
  GB = (GB / 128) * 128;
  XTD_REQUIRE(GB >= 128, XTD_ERR_NOMEM, "xtd_block_response: workspace too small for a 128-point grid chunk");
  h->last_grid_chunks = cdiv(h->ng, GB);
  for (long g0 = 0; g0 < h->ng; g0 += GB) {
    const int gb = (int)std::min<long>(GB, h->ng - g0);
    double *Wo[2], *Wv[2];
    double* cur = scratch;
    for (int ci = 0; ci < 2; ++ci) {
      Wo[ci] = cur; cur += (size_t)nve * gb * h->ch[ci]->ldoo;
      Wv[ci] = cur; cur += (size_t)nve * gb * h->ch[ci]->ldvv;
    }
    {
      PhaseTimer tm(h, XTD_T_XC_GEMM);
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        const int no = c->no, nv = c->nv;
        const MatView ph = view3d(c->phi.p, c->ldphi, h->ng * c->ldphi, nf, gb, no, (int)g0, 0);
        const MatView pv = view3d(c->phiv.p, c->ldphiv, h->ng * c->ldphiv, nf, gb, nv, (int)g0, 0);
        const long so = (long)gb * c->ldoo, sv = (long)gb * c->ldvv;
        XTD_TRY(mm(h, ph, true, view2d(bb[ci].Doo, c->ldoo, no, no), false, gb, no, no, 1, nf, Wo[ci], c->ldoo, so, 1.0, false));
        XTD_TRY(mm(h, pv, true, view2d(bb[ci].Dov, c->ldz, no, nv), true, gb, no, nv, 1, nf, Wo[ci], c->ldoo, so, 1.0, true));
        XTD_TRY(mm(h, pv, true, view2d(bb[ci].Dvv, c->ldvv, nv, nv), false, gb, nv, nv, 1, nf, Wv[ci], c->ldvv, sv, 1.0, false));
        XTD_TRY(mm(h, ph, true, view2d(bb[ci].Dov, c->ldz, no, nv), false, gb, nv, no, 1, nf, Wv[ci], c->ldvv, sv, 1.0, true));
      }
    }
    {
      PhaseTimer tm(h, XTD_T_XC_STREAM);
      XcBlockArgs a;
      a.gb = gb; a.g0 = g0; a.wf = h->wf.p;
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        a.Wo[ci] = Wo[ci]; a.Wv[ci] = Wv[ci]; a.ldWo[ci] = c->ldoo; a.ldWv[ci] = c->ldvv;
        a.phi[ci] = c->phi.p; a.phiv[ci] = c->phiv.p; a.ldphi[ci] = c->ldphi; a.ldphiv[ci] = c->ldphiv;
        a.phi_comp[ci] = h->ng * c->ldphi; a.phiv_comp[ci] = h->ng * c->ldphiv;
        a.no[ci] = c->no; a.nv[ci] = c->nv;
      }
      const unsigned grid = (unsigned)cdiv(gb, 8);
      if (nve == 1) xc_block_weight_kernel<1, false><<<grid, 256, 0, s>>>(a);
      else if (h->tau) xc_block_weight_kernel<4, true><<<grid, 256, 0, s>>>(a);
      else xc_block_weight_kernel<4, false><<<grid, 256, 0, s>>>(a);
      LAUNCH_CHECK();
    }
    PhaseTimer tm(h, XTD_T_XC_GEMM);
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      const int no = c->no, nv = c->nv;
      const MatView Bo = view3d(Wo[ci], c->ldoo, (long)gb * c->ldoo, nve, gb, no);
      XTD_TRY(mm(h, Bo, false, view3d(c->phi.p, c->ldphi, h->ng * c->ldphi, nve, gb, no, (int)g0, 0), false, no, no, gb, nve, 1, bb[ci].Ooo, c->ldoo, 0,
                 cxc, true));
      XTD_TRY(mm(h, Bo, false, view3d(c->phiv.p, c->ldphiv, h->ng * c->ldphiv, nve, gb, nv, (int)g0, 0), false, no, nv, gb, nve, 1, bb[ci].Oov, c->ldz,
                 0, cxc, true));
    }
  }
  return XTD_OK;
}

int copy_block(double* dst, long ldd, const double* src, long lds, int rows, int cols, cudaStream_t s) {
  if (rows > 0 && cols > 0)
    XTD_CUDA(cudaMemcpy2DAsync(dst, (size_t)ldd * 8, src, (size_t)lds * 8, (size_t)cols * 8, rows, cudaMemcpyDeviceToDevice, s));
  return XTD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// xtd_block_response_batch: kb densities per pass over the resident blocks.  Each aux chunk is read (and its int8 Lvv decoded) once
// for all kb densities, and every GEMM carries the kb densities in one dimension:
//   stage 1 (per P, rows stacked over the densities)  [A_1^T; ..; A_kb^T] = [Doo_1; ..] Loo + [Dov_1; ..] Lov^T
//                                                      [B_1^T; ..; B_kb^T] = [Dov_1^T; ..] Loo + [Dvv_1; ..] Lov^T
//   stored transposed through the two-level output rows, so that density x owns columns [x ldoo, x ldoo + no) of SA[P] / SB[P];
//   stage 2 (sum over P, M = kb ldoo)  Ooo += SA^T Loo + SB^T Lov^T,  Oov += SA^T Lov + SB^T Lvv  with density x on rows x ldoo + i.
// K[X] in the same way with U_x^T = X_x^T Loo1, V_x^T = X_x^T Lov1.  Row-stacked (_r) inputs put density x at row x n; the
// column-stacked copies (_c) of Dov and X put it at column x nv.
// ---------------------------------------------------------------------------------------------------------
int mmx(xtd_engine* h, const MatView& A, bool akc, const MatView& B, bool bkc, int M, int N, int K, int nouter, int batches, int a_hi, int b_hi,
        double* Cp, long ldc, long cbs, double alpha, bool acc, int row_div = 0, long row_hi = 0, long row_lo = 0) {
  GemmDesc d;
  d.A = A; d.B = B; d.a_kc = akc; d.b_kc = bkc; d.M = M; d.N = N; d.K = K; d.nouter = nouter;
  d.batches = batches; d.z_div = 1; d.a_hi = a_hi; d.b_hi = b_hi;
  d.C = Cp; d.ldc = ldc; d.c_batch_stride = cbs; d.alpha = alpha; d.accumulate = acc;
  d.c_row_div = row_div; d.c_row_hi = row_hi; d.c_row_lo = row_lo;
  return gemm(h->gemm, d, h->stream);
}

struct BatchBufs {
  double *Doo_r, *Dvv_r, *Dov_r, *Dov_c;   // [kb no][ldoo], [kb nv][ldvv], [kb no][ldz], [no][ldc]
  double *Ooo, *Oov;                       // [kb ldoo][ldoo], [kb ldoo][ldz]: density x from row x ldoo
  long ldc;                                // pad_ld(kb nv)
};
struct BatchX {
  double* X_c = nullptr;                   // [no1][ldx], density x at column x nv0
  double* XO[4] = {nullptr, nullptr, nullptr, nullptr};   // oo, ov: density x from row x su;  vo, vv: from row x sv
  long ldx = 0, su = 0, sv = 0;
};

// fixed buffers of a pass over kb densities; false when the arena cannot hold them
bool batch_take(xtd_engine* h, Arena& ar, int kb, bool with_x, BatchBufs* bb, BatchX* bx) {
  bool ok = true;
  auto take = [&](size_t n) { double* p = ar.take(n); ok = ok && p; return p; };
  for (int ci = 0; ci < 2; ++ci) {
    Channel* c = h->ch[ci];
    bb[ci].ldc = pad_ld((long)kb * c->nv);
    bb[ci].Doo_r = take((size_t)kb * c->no * c->ldoo);
    bb[ci].Dvv_r = take((size_t)kb * c->nv * c->ldvv);
    bb[ci].Dov_r = take((size_t)kb * c->no * c->ldz);
    bb[ci].Dov_c = take((size_t)c->no * bb[ci].ldc);
    bb[ci].Ooo = take((size_t)kb * c->ldoo * c->ldoo);
    bb[ci].Oov = take((size_t)kb * c->ldoo * c->ldz);
  }
  if (with_x) {
    Channel *c0 = h->ch[0], *c1 = h->ch[1];
    bx->ldx = pad_ld((long)kb * c0->nv);
    bx->su = c1->ldoo;
    bx->sv = c1->ldz;
    bx->X_c = take((size_t)c1->no * bx->ldx);
    bx->XO[0] = take((size_t)kb * bx->su * c0->ldoo);
    bx->XO[1] = take((size_t)kb * bx->su * c0->ldz);
    bx->XO[2] = take((size_t)kb * bx->sv * c0->ldoo);
    bx->XO[3] = take((size_t)kb * bx->sv * c0->ldz);
  }
  return ok;
}

// per aux function scratch of tensor t for kb densities (SA, SB, decoded Lvv per channel; SU, SV; rho rows)
size_t batch_per_aux(const xtd_engine* h, int t, int kb, bool doX) {
  size_t per_p = 8 * (size_t)kb + 64;
  for (int ci = 0; ci < 2; ++ci) {
    const Channel* c = h->ch[ci];
    per_p += (size_t)(c->no + c->nv) * kb * c->ldoo + (c->use_oz[t] ? (size_t)c->nv * c->ldvv : 0) + 96;
  }
  if (doX) {
    const Channel *c0 = h->ch[0], *c1 = h->ch[1];
    per_p += (size_t)c0->nv * kb * (c1->ldoo + c1->ldz) + 64;
  }
  return per_p;
}

size_t batch_per_point(const xtd_engine* h, int kb) {
  size_t per_g = 0;
  for (auto* c : h->ch) per_g += (size_t)h->nvar_eff * (pad_ld((long)kb * c->no) + pad_ld((long)kb * c->nv));
  return per_g;
}

int block_response_batch_df(xtd_engine* h, int kb, const BatchBufs* bb, const double* coef, const BatchX* bx, double* scratch,
                            size_t scratch_doubles) {
  cudaStream_t s = h->stream;
  const double cj = coef[0], cx = coef[4];
  Channel *c0 = h->ch[0], *c1 = h->ch[1];
  for (int t = 0; t < 2; ++t) {
    const double ck = coef[1 + t];
    const bool doJ = t == 0 && cj != 0.0, doK = ck != 0.0, doX = t == 0 && bx->X_c && cx != 0.0;
    if (!(doJ || doK || doX) || h->naux[t] == 0) continue;
    const long naux = h->naux[t];
    const double* Lov[2];
    long ldov[2];
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      Lov[ci] = ov_block(h, ci, t, &ldov[ci]);
      XTD_REQUIRE(oovv_resident(h, c, t) && Lov[ci], XTD_ERR_STATE,
                  "xtd_block_response_batch: channel %d holds no MO blocks of tensor %d (call xtd_enable_block_response before xtd_df_begin)",
                  ci, t);
      XTD_REQUIRE(!c->use_oz[t] || c->oz_col0[t] == 0, XTD_ERR_UNSUPPORTED, "xtd_block_response_batch: block-weighted emulated exchange image");
    }
    long pc = (long)(scratch_doubles / batch_per_aux(h, t, kb, doX));
    if (h->env.max_pc > 0) pc = std::min<long>(pc, h->env.max_pc);
    pc = std::min<long>(pc, naux);
    XTD_REQUIRE(pc >= 1, XTD_ERR_NOMEM, "xtd_block_response_batch: workspace too small for one aux function");
    double* cur = scratch;
    auto take = [&](size_t n) { double* p = cur; cur += (n + 31) & ~(size_t)31; return p; };
    double *SA[2], *SB[2], *Ldec[2] = {nullptr, nullptr};
    long ldS[2], sSA[2], sSB[2];
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      ldS[ci] = (long)kb * c->ldoo;
      sSA[ci] = (long)c->no * ldS[ci];
      sSB[ci] = (long)c->nv * ldS[ci];
      SA[ci] = take((size_t)pc * sSA[ci]);
      SB[ci] = take((size_t)pc * sSB[ci]);
      if (c->use_oz[t]) Ldec[ci] = take((size_t)pc * c->nv * c->ldvv);
    }
    const long ldU = (long)kb * bx->su, ldV = (long)kb * bx->sv, sSU = (long)c0->nv * ldU, sSV = (long)c0->nv * ldV;
    double* SU = doX ? take((size_t)pc * sSU) : nullptr;
    double* SV = doX ? take((size_t)pc * sSV) : nullptr;
    // the stage-1 GEMMs write only the live columns of each density's slot: the padding between slots stays zero
    XTD_CUDA(cudaMemsetAsync(scratch, 0, (size_t)(cur - scratch) * 8, s));
    double* R = take((size_t)6 * kb * pc);
    double* rho = take((size_t)kb * pc);
    h->last_aux_chunks = std::max<long>(h->last_aux_chunks, cdiv(naux, pc));
    for (long P0 = 0; P0 < naux; P0 += pc) {
      const int pn = (int)std::min<long>(pc, naux - P0);
      const double *Loo[2], *Lvv[2], *Lo[2];
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        Loo[ci] = c->Loo[t].p + P0 * c->no * c->ldoo;
        Lo[ci] = Lov[ci] + P0 * c->no * ldov[ci];
        if (c->use_oz[t]) {
          PhaseTimer tm(h, XTD_T_K2_SLICE);
          oz_unslice_b_kernel<<<dim3((unsigned)cdiv((long)c->nv * c->nv, 256), pn), 256, 0, s>>>(
              Ldec[ci], c->ldvv, (long)c->nv * c->ldvv, c->LvvS[t], c->LvvScale[t], h->oz_slices, c->nv, c->ozB.rows_pad, c->nv, c->ozB.nkb,
              c->oz_group, P0, pn);
          LAUNCH_CHECK();
          Lvv[ci] = Ldec[ci];
        } else {
          Lvv[ci] = c->Lvv[t].p + P0 * c->nv * c->ldvv;
        }
      }
      if (doJ) {
        PhaseTimer tm(h, XTD_T_J);
        // R[blk][x][P] for the six blocks (Doo, Dvv, Dov of each channel); rho[x][P]; every L element read once per 4 densities
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          j_rho_kernel<4><<<pn, 256, 0, s>>>(R + (size_t)(3 * ci) * kb * pc, pc, Loo[ci], c->ldoo, (long)c->no * c->ldoo, bb[ci].Doo_r, c->ldoo,
                                             (long)c->no * c->ldoo, c->no, c->no, kb);
          LAUNCH_CHECK();
          j_rho_kernel<4><<<pn, 256, 0, s>>>(R + (size_t)(3 * ci + 1) * kb * pc, pc, Lvv[ci], c->ldvv, (long)c->nv * c->ldvv, bb[ci].Dvv_r, c->ldvv,
                                             (long)c->nv * c->ldvv, c->nv, c->nv, kb);
          LAUNCH_CHECK();
          j_rho_kernel<4><<<pn, 256, 0, s>>>(R + (size_t)(3 * ci + 2) * kb * pc, pc, Lo[ci], ldov[ci], (long)c->no * ldov[ci], bb[ci].Dov_r, c->ldz,
                                             (long)c->no * c->ldz, c->no, c->nv, kb);
          LAUNCH_CHECK();
        }
        RhoWeights w = {{cj, cj, 2.0 * cj, cj, cj, 2.0 * cj}};
        rho_combine_kernel<<<grid1d((long)kb * pc, 256), 256, 0, s>>>(rho, R, (long)kb * pc, 6, (long)kb * pc, w);
        LAUNCH_CHECK();
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          j_apply_kernel<4><<<dim3((unsigned)cdiv((long)c->no * c->no, 256), (unsigned)cdiv(kb, 4)), 256, 0, s>>>(
              bb[ci].Ooo, c->ldoo, (long)c->ldoo * c->ldoo, Loo[ci], c->ldoo, (long)c->no * c->ldoo, rho, pc, pn, c->no, c->no, kb);
          LAUNCH_CHECK();
          j_apply_kernel<4><<<dim3((unsigned)cdiv((long)c->no * c->nv, 256), (unsigned)cdiv(kb, 4)), 256, 0, s>>>(
              bb[ci].Oov, c->ldz, (long)c->ldoo * c->ldz, Lo[ci], ldov[ci], (long)c->no * ldov[ci], rho, pc, pn, c->no, c->nv, kb);
          LAUNCH_CHECK();
        }
      }
      if (doK)
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          const int no = c->no, nv = c->nv, Mo = (kb - 1) * c->ldoo + no;
          const long soo = (long)no * c->ldoo, sov = (long)no * ldov[ci], svv = (long)nv * c->ldvv;
          const MatView LooV = view3d(Loo[ci], c->ldoo, soo, pn, no, no), LovV = view3d(Lo[ci], ldov[ci], sov, pn, no, nv);
          {
            PhaseTimer tm(h, XTD_T_K1);
            XTD_TRY(mmx(h, view2d(bb[ci].Doo_r, c->ldoo, kb * no, no), true, LooV, false, kb * no, no, no, 1, pn, 0, 1, SA[ci], ldS[ci], sSA[ci], 1.0,
                        false, no, c->ldoo, ldS[ci]));
            XTD_TRY(mmx(h, view2d(bb[ci].Dov_r, c->ldz, kb * no, nv), true, LovV, true, kb * no, no, nv, 1, pn, 0, 1, SA[ci], ldS[ci], sSA[ci], 1.0,
                        true, no, c->ldoo, ldS[ci]));
            XTD_TRY(mmx(h, view2d(bb[ci].Dov_c, bb[ci].ldc, no, kb * nv), false, LooV, false, kb * nv, no, no, 1, pn, 0, 1, SB[ci], ldS[ci], sSB[ci],
                        1.0, false, nv, c->ldoo, ldS[ci]));
            XTD_TRY(mmx(h, view2d(bb[ci].Dvv_r, c->ldvv, kb * nv, nv), true, LovV, true, kb * nv, no, nv, 1, pn, 0, 1, SB[ci], ldS[ci], sSB[ci], 1.0,
                        true, nv, c->ldoo, ldS[ci]));
          }
          PhaseTimer tm(h, XTD_T_K2);
          const MatView Av = view3d(SA[ci], ldS[ci], sSA[ci], pn, no, Mo), Bv = view3d(SB[ci], ldS[ci], sSB[ci], pn, nv, Mo);
          XTD_TRY(mmx(h, Av, false, LooV, false, Mo, no, no, pn, 1, 0, 0, bb[ci].Ooo, c->ldoo, 0, ck, true));
          XTD_TRY(mmx(h, Bv, false, LovV, true, Mo, no, nv, pn, 1, 0, 0, bb[ci].Ooo, c->ldoo, 0, ck, true));
          XTD_TRY(mmx(h, Av, false, LovV, false, Mo, nv, no, pn, 1, 0, 0, bb[ci].Oov, c->ldz, 0, ck, true));
          XTD_TRY(mmx(h, Bv, false, view3d(Lvv[ci], c->ldvv, svv, pn, nv, nv), false, Mo, nv, nv, pn, 1, 0, 0, bb[ci].Oov, c->ldz, 0, ck, true));
        }
      if (doX) {
        const int no1 = c1->no, nv1 = c1->nv, no0 = c0->no, nv0 = c0->nv;
        const int Mu = (kb - 1) * (int)bx->su + no1, Mv = (kb - 1) * (int)bx->sv + nv1;
        const MatView Xv = view2d(bx->X_c, bx->ldx, no1, kb * nv0);
        {
          PhaseTimer tm(h, XTD_T_K1);
          XTD_TRY(mmx(h, Xv, false, view3d(Loo[1], c1->ldoo, (long)no1 * c1->ldoo, pn, no1, no1), false, kb * nv0, no1, no1, 1, pn, 0, 1, SU, ldU,
                      sSU, 1.0, false, nv0, bx->su, ldU));
          XTD_TRY(mmx(h, Xv, false, view3d(Lo[1], ldov[1], (long)no1 * ldov[1], pn, no1, nv1), false, kb * nv0, nv1, no1, 1, pn, 0, 1, SV, ldV,
                      sSV, 1.0, false, nv0, bx->sv, ldV));
        }
        PhaseTimer tm(h, XTD_T_K2);
        const MatView Uv = view3d(SU, ldU, sSU, pn, nv0, Mu), Vv = view3d(SV, ldV, sSV, pn, nv0, Mv);
        const MatView Lov0 = view3d(Lo[0], ldov[0], (long)no0 * ldov[0], pn, no0, nv0);
        const MatView Lvv0 = view3d(Lvv[0], c0->ldvv, (long)nv0 * c0->ldvv, pn, nv0, nv0);
        XTD_TRY(mmx(h, Uv, false, Lov0, true, Mu, no0, nv0, pn, 1, 0, 0, bx->XO[0], c0->ldoo, 0, cx, true));
        XTD_TRY(mmx(h, Uv, false, Lvv0, false, Mu, nv0, nv0, pn, 1, 0, 0, bx->XO[1], c0->ldz, 0, cx, true));
        XTD_TRY(mmx(h, Vv, false, Lov0, true, Mv, no0, nv0, pn, 1, 0, 0, bx->XO[2], c0->ldoo, 0, cx, true));
        XTD_TRY(mmx(h, Vv, false, Lvv0, false, Mv, nv0, nv0, pn, 1, 0, 0, bx->XO[3], c0->ldz, 0, cx, true));
      }
    }
  }
  return XTD_OK;
}

// grid term for kb densities: Wo = phi [Doo_1 ..] + phiv [Dov_1^T ..],  Wv = phiv [Dvv_1 ..] + phi [Dov_1 ..] (density x at column
// x no / x nv), xc_block_weight_batch_kernel, then  Ooo_x += c_xc sum_c Bo_x^T phi_c,  Oov_x += c_xc sum_c Bo_x^T phiv_c  as one GEMM
// each with M = kb no (output rows placed at x ldoo + i)
int block_response_batch_xc(xtd_engine* h, int kb, const BatchBufs* bb, double cxc, double* scratch, size_t scratch_doubles) {
  cudaStream_t s = h->stream;
  XTD_REQUIRE(h->fxc_kind == XTD_FXC_UKS, XTD_ERR_UNSUPPORTED, "xtd_block_response_batch: the grid term needs the UKS kernel tables");
  const int nve = h->nvar_eff, nf = h->tau ? 4 : 1;
  for (auto* c : h->ch)
    XTD_REQUIRE(c->phiv.p && c->phi.p, XTD_ERR_STATE,
                "xtd_block_response_batch: fp64 virtual MO values not kept on the grid (call xtd_enable_block_response before the grid commit)");
  long ldWo[2], ldWv[2];
  for (int ci = 0; ci < 2; ++ci) {
    ldWo[ci] = pad_ld((long)kb * h->ch[ci]->no);
    ldWv[ci] = pad_ld((long)kb * h->ch[ci]->nv);
  }
  long GB = (long)(scratch_doubles / batch_per_point(h, kb)) - 64;
  GB = std::min<long>(GB, 1 << 16);
  if (h->env.max_gb > 0) GB = std::min<long>(GB, std::max<long>(h->env.max_gb, 128));
  GB = (GB / 128) * 128;
  XTD_REQUIRE(GB >= 128, XTD_ERR_NOMEM, "xtd_block_response_batch: workspace too small for a 128-point grid chunk");
  h->last_grid_chunks = std::max<long>(h->last_grid_chunks, cdiv(h->ng, GB));
  for (long g0 = 0; g0 < h->ng; g0 += GB) {
    const int gb = (int)std::min<long>(GB, h->ng - g0);
    double *Wo[2], *Wv[2];
    double* cur = scratch;
    for (int ci = 0; ci < 2; ++ci) {
      Wo[ci] = cur; cur += (size_t)nve * gb * ldWo[ci];
      Wv[ci] = cur; cur += (size_t)nve * gb * ldWv[ci];
    }
    {
      PhaseTimer tm(h, XTD_T_XC_GEMM);
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        const int no = c->no, nv = c->nv;
        const MatView ph = view3d(c->phi.p, c->ldphi, h->ng * c->ldphi, nf, gb, no, (int)g0, 0);
        const MatView pv = view3d(c->phiv.p, c->ldphiv, h->ng * c->ldphiv, nf, gb, nv, (int)g0, 0);
        const long so = (long)gb * ldWo[ci], sv = (long)gb * ldWv[ci];
        XTD_TRY(mm(h, ph, true, view2d(bb[ci].Doo_r, c->ldoo, kb * no, no), true, gb, kb * no, no, 1, nf, Wo[ci], ldWo[ci], so, 1.0, false));
        XTD_TRY(mm(h, pv, true, view2d(bb[ci].Dov_r, c->ldz, kb * no, nv), true, gb, kb * no, nv, 1, nf, Wo[ci], ldWo[ci], so, 1.0, true));
        XTD_TRY(mm(h, pv, true, view2d(bb[ci].Dvv_r, c->ldvv, kb * nv, nv), true, gb, kb * nv, nv, 1, nf, Wv[ci], ldWv[ci], sv, 1.0, false));
        XTD_TRY(mm(h, ph, true, view2d(bb[ci].Dov_c, bb[ci].ldc, no, kb * nv), false, gb, kb * nv, no, 1, nf, Wv[ci], ldWv[ci], sv, 1.0, true));
      }
    }
    {
      PhaseTimer tm(h, XTD_T_XC_STREAM);
      XcBlockArgs a;
      a.gb = gb; a.g0 = g0; a.wf = h->wf.p;
      for (int ci = 0; ci < 2; ++ci) {
        Channel* c = h->ch[ci];
        a.Wo[ci] = Wo[ci]; a.Wv[ci] = Wv[ci]; a.ldWo[ci] = ldWo[ci]; a.ldWv[ci] = ldWv[ci];
        a.phi[ci] = c->phi.p; a.phiv[ci] = c->phiv.p; a.ldphi[ci] = c->ldphi; a.ldphiv[ci] = c->ldphiv;
        a.phi_comp[ci] = h->ng * c->ldphi; a.phiv_comp[ci] = h->ng * c->ldphiv;
        a.no[ci] = c->no; a.nv[ci] = c->nv;
      }
      const unsigned grid = (unsigned)cdiv(gb, 8);
      if (nve == 1) xc_block_weight_batch_kernel<1, false, 4><<<grid, 256, 0, s>>>(a, kb);
      else if (h->tau) xc_block_weight_batch_kernel<4, true, 4><<<grid, 256, 0, s>>>(a, kb);
      else xc_block_weight_batch_kernel<4, false, 4><<<grid, 256, 0, s>>>(a, kb);
      LAUNCH_CHECK();
    }
    PhaseTimer tm(h, XTD_T_XC_GEMM);
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      const int no = c->no, nv = c->nv;
      const MatView Bo = view3d(Wo[ci], ldWo[ci], (long)gb * ldWo[ci], nve, gb, kb * no);
      XTD_TRY(mmx(h, Bo, false, view3d(c->phi.p, c->ldphi, h->ng * c->ldphi, nve, gb, no, (int)g0, 0), false, kb * no, no, gb, nve, 1, 0, 0,
                  bb[ci].Ooo, c->ldoo, 0, cxc, true, no, (long)c->ldoo * c->ldoo, c->ldoo));
      XTD_TRY(mmx(h, Bo, false, view3d(c->phiv.p, c->ldphiv, h->ng * c->ldphiv, nve, gb, nv, (int)g0, 0), false, kb * no, nv, gb, nve, 1, 0, 0,
                  bb[ci].Oov, c->ldz, 0, cxc, true, no, (long)c->ldoo * c->ldz, c->ldz));
    }
  }
  return XTD_OK;
}

}  // namespace

extern "C" int xtd_enable_block_response(xtd_handle h) {
  XTD_REQUIRE(h && !h->finalized && !h->grid_committed && h->naux[0] == 0 && h->naux[1] == 0, XTD_ERR_STATE,
              "xtd_enable_block_response must precede xtd_grid_commit, xtd_df_begin and xtd_finalize");
  h->block_resp = true;
  return XTD_OK;
}

extern "C" int xtd_block_response(xtd_handle h, const double* dens_dev, double* out_dev, const double* coef_host, const double* x_dev,
                                  double* xout_dev) {
  XTD_REQUIRE(h && h->finalized, XTD_ERR_STATE, "xtd_block_response before xtd_finalize");
  XTD_REQUIRE(dens_dev && out_dev && coef_host && (!x_dev || xout_dev), XTD_ERR_ARG, "xtd_block_response: bad arguments");
  XTD_REQUIRE(h->ch.size() == 2, XTD_ERR_UNSUPPORTED, "xtd_block_response needs a two-channel plan");
  cudaStream_t s = h->stream;
  h->ev_used = 0;
  for (int i = 0; i < 12; ++i) h->phase_flops[i] = 0.0;
  h->last_aux_chunks = h->last_grid_chunks = 0;
  if (h->ev_ok) cudaEventRecord(h->ev_total[0], s);
  h->arena.used = 0;
  BlockBufs bb[2];
  for (int ci = 0; ci < 2; ++ci) {
    Channel* c = h->ch[ci];
    bb[ci].Doo = h->arena.take((size_t)c->no * c->ldoo);
    bb[ci].Dvv = h->arena.take((size_t)c->nv * c->ldvv);
    bb[ci].Dov = h->arena.take((size_t)c->no * c->ldz);
    bb[ci].Ooo = h->arena.take((size_t)c->no * c->ldoo);
    bb[ci].Oov = h->arena.take((size_t)c->no * c->ldz);
    XTD_REQUIRE(bb[ci].Doo && bb[ci].Dvv && bb[ci].Dov && bb[ci].Ooo && bb[ci].Oov, XTD_ERR_NOMEM, "xtd_block_response: workspace exhausted");
  }
  Channel *c0 = h->ch[0], *c1 = h->ch[1];
  double* X = nullptr;
  double* XO[4] = {nullptr, nullptr, nullptr, nullptr};
  if (x_dev) {
    X = h->arena.take((size_t)c1->no * c0->ldz);
    XO[0] = h->arena.take((size_t)c1->no * c0->ldoo);
    XO[1] = h->arena.take((size_t)c1->no * c0->ldz);
    XO[2] = h->arena.take((size_t)c1->nv * c0->ldoo);
    XO[3] = h->arena.take((size_t)c1->nv * c0->ldz);
    XTD_REQUIRE(X && XO[0] && XO[1] && XO[2] && XO[3], XTD_ERR_NOMEM, "xtd_block_response: workspace exhausted");
  }
  const size_t fixed = h->arena.used;
  {
    PhaseTimer tm(h, XTD_T_PACK);
    XTD_CUDA(cudaMemsetAsync(h->arena.base, 0, fixed, s));
    const double* src = dens_dev;
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      XTD_TRY(copy_block(bb[ci].Doo, c->ldoo, src, c->no, c->no, c->no, s)); src += (size_t)c->no * c->no;
      XTD_TRY(copy_block(bb[ci].Dvv, c->ldvv, src, c->nv, c->nv, c->nv, s)); src += (size_t)c->nv * c->nv;
      XTD_TRY(copy_block(bb[ci].Dov, c->ldz, src, c->nv, c->no, c->nv, s)); src += (size_t)c->no * c->nv;
    }
    if (X) XTD_TRY(copy_block(X, c0->ldz, x_dev, c0->nv, c1->no, c0->nv, s));
  }
  size_t split_bytes = std::min<size_t>(h->arena.left() / 4, (size_t)1 << 30);
  h->gemm.split_ws = h->arena.take(split_bytes / 8);
  h->gemm.split_ws_bytes = split_bytes;
  const size_t scratch_doubles = h->arena.left() / 8 - 64;
  double* scratch = h->arena.take(scratch_doubles);
  XTD_REQUIRE(scratch, XTD_ERR_NOMEM, "xtd_block_response: workspace exhausted (chunk scratch)");
  XTD_TRY(block_response_df(h, bb, coef_host, X, XO, scratch, scratch_doubles));
  if (coef_host[3] != 0.0 && h->fxc_kind != XTD_FXC_NONE && h->ng > 0) XTD_TRY(block_response_xc(h, bb, coef_host[3], scratch, scratch_doubles));
  {
    PhaseTimer tm(h, XTD_T_UNPACK);
    double* dst = out_dev;
    for (int ci = 0; ci < 2; ++ci) {
      Channel* c = h->ch[ci];
      XTD_TRY(copy_block(dst, c->no, bb[ci].Ooo, c->ldoo, c->no, c->no, s)); dst += (size_t)c->no * c->no;
      XTD_TRY(copy_block(dst, c->nv, bb[ci].Oov, c->ldz, c->no, c->nv, s)); dst += (size_t)c->no * c->nv;
    }
    if (X) {
      const long w = (long)c0->no + c0->nv;
      XTD_TRY(copy_block(xout_dev, w, XO[0], c0->ldoo, c1->no, c0->no, s));
      XTD_TRY(copy_block(xout_dev + c0->no, w, XO[1], c0->ldz, c1->no, c0->nv, s));
      XTD_TRY(copy_block(xout_dev + (size_t)c1->no * w, w, XO[2], c0->ldoo, c1->nv, c0->no, s));
      XTD_TRY(copy_block(xout_dev + (size_t)c1->no * w + c0->no, w, XO[3], c0->ldz, c1->nv, c0->nv, s));
    }
  }
  if (h->ev_ok) cudaEventRecord(h->ev_total[1], s);
  return XTD_OK;
}

extern "C" int xtd_block_response_batch(xtd_handle h, int ndens, const double* dens_dev, double* out_dev, const double* coef_host,
                                        const double* x_dev, double* xout_dev) {
  XTD_REQUIRE(h && h->finalized, XTD_ERR_STATE, "xtd_block_response_batch before xtd_finalize");
  XTD_REQUIRE(ndens >= 1 && dens_dev && out_dev && coef_host && (!x_dev || xout_dev), XTD_ERR_ARG, "xtd_block_response_batch: bad arguments");
  XTD_REQUIRE(h->ch.size() == 2, XTD_ERR_UNSUPPORTED, "xtd_block_response_batch needs a two-channel plan");
  cudaStream_t s = h->stream;
  h->ev_used = 0;
  for (int i = 0; i < 12; ++i) h->phase_flops[i] = 0.0;
  h->last_aux_chunks = h->last_grid_chunks = 0;
  if (h->ev_ok) cudaEventRecord(h->ev_total[0], s);
  Channel *c0 = h->ch[0], *c1 = h->ch[1];
  const bool with_x = x_dev != nullptr;
  const bool doxc = coef_host[3] != 0.0 && h->fxc_kind != XTD_FXC_NONE && h->ng > 0;
  size_t nin = 0, nout = 0;
  for (auto* c : h->ch) {
    nin += (size_t)c->no * c->no + (size_t)c->nv * c->nv + (size_t)c->no * c->nv;
    nout += (size_t)c->no * c->no + (size_t)c->no * c->nv;
  }
  const size_t nxin = (size_t)c1->no * c0->nv, nxout = (size_t)(c1->no + c1->nv) * (c0->no + c0->nv);
  // densities per pass: the largest kb (of ceil(ndens / n) for n = 1, 2, ..) whose fixed buffers, split-K partials and one aux function
  // / one 128-point grid chunk of scratch fit the workspace; the passes are counted in last_dens_batches
  int kb = 0;
  for (int n = 1; n <= ndens && !kb; ++n) {
    const int k = (int)cdiv(ndens, n);
    if (n > 1 && k == (int)cdiv(ndens, n - 1)) continue;
    Arena ar = h->arena;
    ar.used = 0;
    BatchBufs bb[2];
    BatchX bx;
    if (!batch_take(h, ar, k, with_x, bb, &bx)) continue;
    const size_t left = ar.left() - std::min<size_t>(ar.left() / 4, (size_t)1 << 30);
    const size_t scratch = left / 8 > 64 + 512 ? left / 8 - 64 - 512 : 0;
    bool fits = true;
    for (int t = 0; t < 2; ++t)
      if (h->naux[t] > 0) fits = fits && scratch >= batch_per_aux(h, t, k, with_x && t == 0);
    if (doxc) fits = fits && (long)(scratch / batch_per_point(h, k)) - 64 >= 128;
    if (fits) kb = k;
  }
  XTD_REQUIRE(kb >= 1, XTD_ERR_NOMEM, "xtd_block_response_batch: workspace too small for one density");
  h->last_dens_batches = cdiv(ndens, kb);
  for (int x0 = 0; x0 < ndens; x0 += kb) {
    const int nb = std::min(kb, ndens - x0);
    h->arena.used = 0;
    BatchBufs bb[2];
    BatchX bx;
    XTD_REQUIRE(batch_take(h, h->arena, nb, with_x, bb, &bx), XTD_ERR_NOMEM, "xtd_block_response_batch: workspace exhausted");
    const size_t fixed = h->arena.used;
    {
      PhaseTimer tm(h, XTD_T_PACK);
      XTD_CUDA(cudaMemsetAsync(h->arena.base, 0, fixed, s));
      for (int x = 0; x < nb; ++x) {
        const double* src = dens_dev + (size_t)(x0 + x) * nin;
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          XTD_TRY(copy_block(bb[ci].Doo_r + (size_t)x * c->no * c->ldoo, c->ldoo, src, c->no, c->no, c->no, s)); src += (size_t)c->no * c->no;
          XTD_TRY(copy_block(bb[ci].Dvv_r + (size_t)x * c->nv * c->ldvv, c->ldvv, src, c->nv, c->nv, c->nv, s)); src += (size_t)c->nv * c->nv;
          XTD_TRY(copy_block(bb[ci].Dov_r + (size_t)x * c->no * c->ldz, c->ldz, src, c->nv, c->no, c->nv, s));
          XTD_TRY(copy_block(bb[ci].Dov_c + (size_t)x * c->nv, bb[ci].ldc, src, c->nv, c->no, c->nv, s)); src += (size_t)c->no * c->nv;
        }
        if (with_x) XTD_TRY(copy_block(bx.X_c + (size_t)x * c0->nv, bx.ldx, x_dev + (size_t)(x0 + x) * nxin, c0->nv, c1->no, c0->nv, s));
      }
    }
    size_t split_bytes = std::min<size_t>(h->arena.left() / 4, (size_t)1 << 30);
    h->gemm.split_ws = h->arena.take(split_bytes / 8);
    h->gemm.split_ws_bytes = split_bytes;
    const size_t scratch_doubles = h->arena.left() / 8 - 64;
    double* scratch = h->arena.take(scratch_doubles);
    XTD_REQUIRE(scratch, XTD_ERR_NOMEM, "xtd_block_response_batch: workspace exhausted (chunk scratch)");
    XTD_TRY(block_response_batch_df(h, nb, bb, coef_host, &bx, scratch, scratch_doubles));
    if (doxc) XTD_TRY(block_response_batch_xc(h, nb, bb, coef_host[3], scratch, scratch_doubles));
    {
      PhaseTimer tm(h, XTD_T_UNPACK);
      for (int x = 0; x < nb; ++x) {
        double* dst = out_dev + (size_t)(x0 + x) * nout;
        for (int ci = 0; ci < 2; ++ci) {
          Channel* c = h->ch[ci];
          XTD_TRY(copy_block(dst, c->no, bb[ci].Ooo + (size_t)x * c->ldoo * c->ldoo, c->ldoo, c->no, c->no, s)); dst += (size_t)c->no * c->no;
          XTD_TRY(copy_block(dst, c->nv, bb[ci].Oov + (size_t)x * c->ldoo * c->ldz, c->ldz, c->no, c->nv, s)); dst += (size_t)c->no * c->nv;
        }
        if (with_x) {
          const long w = (long)c0->no + c0->nv;
          double* xo = xout_dev + (size_t)(x0 + x) * nxout;
          XTD_TRY(copy_block(xo, w, bx.XO[0] + (size_t)x * bx.su * c0->ldoo, c0->ldoo, c1->no, c0->no, s));
          XTD_TRY(copy_block(xo + c0->no, w, bx.XO[1] + (size_t)x * bx.su * c0->ldz, c0->ldz, c1->no, c0->nv, s));
          XTD_TRY(copy_block(xo + (size_t)c1->no * w, w, bx.XO[2] + (size_t)x * bx.sv * c0->ldoo, c0->ldoo, c1->nv, c0->no, s));
          XTD_TRY(copy_block(xo + (size_t)c1->no * w + c0->no, w, bx.XO[3] + (size_t)x * bx.sv * c0->ldz, c0->ldz, c1->nv, c0->nv, s));
        }
      }
    }
  }
  if (h->ev_ok) cudaEventRecord(h->ev_total[1], s);
  return XTD_OK;
}

extern "C" int xtd_last_density_batches(xtd_handle h, long* nbatches) {
  XTD_REQUIRE(h && nbatches, XTD_ERR_ARG, "xtd_last_density_batches: bad arguments");
  *nbatches = h->last_dens_batches;
  return XTD_OK;
}
