// cs_b200.cu -- host side of libcsb200.so (C ABI in include/cs_b200.h).
// Plain CUDA runtime, no torch.  One handle = one connected component's operator
// resident on one B200 + a panel workspace for the batched PCG.
#include "../../include/cs_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "amg_host.hpp"
#include "win_host.hpp"
#include "kernels.cuh"
#include "raster_assembly.cuh"
#include "components.cuh"
#include "setup_device.hpp"

using namespace csb;

namespace {

thread_local std::string g_create_error;

struct GraphSlot {
  cudaGraphExec_t exec = nullptr;
  int chunk = 0;
  int64_t kernels = 0, spmms = 0;   // launches inside one graph replay
  cudaGraphExec_t loop_exec = nullptr;        // whole PCG loop as a device-side WHILE graph
  int64_t loop_kernels = 0, loop_spmms = 0;   // launches per loop iteration
};

}  // namespace

// one CSR resident on the device, with its row-block partition (type-erased values)
struct DevCsr {
  int* rowptr = nullptr;
  int* colidx = nullptr;
  void* vals = nullptr;
  int* bstart = nullptr;
  int nblocks = 0;
  int nrows = 0;
  int64_t nnz = 0;
  int lpr = 1;  // lanes per row used by k_spmm for this matrix
  // windowed row-block form for the TMA-staged kernel (win_host.hpp); null => plain kernel
  WinMeta* win_meta = nullptr;
  unsigned char* blob = nullptr;   // per-block records [values | 1/diag | local columns | row offsets]
  int has_dinv = 0;
  int64_t win_blocks = 0;
  int win_nblocks = 0;
  // stencil (DIA) form (kernels.cuh k_stencil): 9 diagonals, ld apart; null => CSR kernels
  void* dia = nullptr;
  size_t dia_ld = 0;
  int dia_nr = 0;
  // ELL-4 copy of a prolongator with <= 4 entries per row (k_stencil_prolong_jacobi); null otherwise
  int* ell_col = nullptr;
  void* ell_val = nullptr;
  size_t ell_ld = 0;
};

// one multigrid level below the finest (the finest level aliases the handle's own CSR)
struct DevLevel {
  int64_t n = 0, n_pad = 0;
  DevCsr A, P, R;          // P: this level <- next coarser ; R = P^T
  void* dinv = nullptr;
  double omega = 2.0 / 3.0;
  void *x = nullptr, *b = nullptr, *t = nullptr, *y = nullptr;   // panels n_pad x ktmax
};

struct cs_b200_handle {
  int device = 0;
  int dtype = CS_B200_F64;
  int64_t n = 0, n_pad = 0, nnz = 0;
  int* d_rowptr = nullptr;
  int* d_colidx = nullptr;
  void* d_vals = nullptr;
  bool owns_matrix = true;
  void* d_vals0 = nullptr;           // pristine values while grounds are applied (cs_b200_set_grounds)
  bool grounds_applied = false;      // d_vals currently differ from the operator as created
  void* d_dinv = nullptr;
  int* d_bstart = nullptr;
  int nblocks = 0;
  int ktmax = 8;
  void *X = nullptr, *R = nullptr, *P = nullptr, *AP = nullptr, *B = nullptr, *stage = nullptr;
  void* Z = nullptr;                 // AMG: z = M^-1 r
  DevCsr A0;                         // view of the finest operator (aliases d_rowptr/...)
  std::vector<DevLevel> lv;          // lv[0] = finest (A aliases A0), lv.back() = coarsest
  double* d_pinv = nullptr;          // dense pseudo-inverse of the coarsest operator
  double amg_opc = 0.0;              // operator complexity
  bool amg = false;
  // mixed precision: fp64 CG around an fp32 V-cycle.  lv32 = float copies of every level's
  // operators and panels (the finest included); R32/X32/T32/Z32 = finest-level float panels.
  bool mixed = false;
  std::vector<DevLevel> lv32;
  void *R32 = nullptr, *X32 = nullptr, *T32 = nullptr, *Z32 = nullptr;
  void *d_cum = nullptr, *d_max = nullptr;
  PanelCtl* d_ctl = nullptr;
  PanelCtl* h_ctl = nullptr;  // pinned
  double* d_partials = nullptr;
  float* d_flush = nullptr;
  size_t flush_elems = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
  // solve_rhs host<->device pipeline: panel i+1 uploads and panel i-1 downloads on two copy
  // streams while panel i solves (column-major staging buffers, double-buffered; lazy)
  // cs_b200_solve_sources scratch (grown on demand)
  long long* d_sp_rows = nullptr;
  double* d_sp_vals = nullptr;
  int* d_sp_ptr = nullptr;
  size_t sp_cap = 0;
  long long* d_probe = nullptr;
  void* d_probe_out = nullptr;
  size_t probe_cap = 0;
  cudaStream_t s_in = nullptr, s_out = nullptr;
  void* io_in[2] = {nullptr, nullptr};
  void* io_out[2] = {nullptr, nullptr};
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr};
  cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
  int num_sms = 148;
  int grid_spmm = 148, grid_ew = 148;
  cs_b200_opts opts{};
  cs_b200_stats stats{};
  GraphSlot graphs[4];  // KT = 1,2,4,8
  // optional per-launch SpMM timing (cs_b200_profile_spmm): event pairs harvested at
  // every host poll, so the pool only has to cover one chunk of iterations.
  int profile = 0;
  std::vector<cudaEvent_t> prof_ev;
  size_t prof_used = 0;
  double prof_ms = 0.0;
  double prof_bytes = 0.0;   // algorithmic bytes of the timed launches (DESIGN.md §4 formula)
  int64_t prof_launches = 0;
  // the same per kernel class: slot = 2 * MODE + (fp32 ? 1 : 0), MODE 7 = fused prolongation + sweep
  std::vector<int> prof_slot;           // one entry per event pair in flight
  std::vector<double> prof_pair_bytes;
  double prof_slot_ms[16] = {}, prof_slot_bytes[16] = {};
  int64_t prof_slot_launches[16] = {};
  std::string err;
  size_t esize() const { return dtype == CS_B200_F64 ? 8 : 4; }
};

namespace {

// CS_B200_VERBOSE=1: one stderr line per setup phase (host hierarchy, windows, uploads)
struct Tick {
  bool on = std::getenv("CS_B200_VERBOSE") != nullptr;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  void operator()(const char* what) {
    if (!on) return;
    const auto t1 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[cs_b200 setup] %-28s %8.1f ms\n", what,
                 std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

int set_err(cs_b200_handle* h, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CK(h, call)                                                                      \
  do {                                                                                   \
    cudaError_t _e = (call);                                                             \
    if (_e != cudaSuccess)                                                               \
      return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s at %s:%d (%s)",                 \
                     cudaGetErrorString(_e), __FILE__, __LINE__, #call);                 \
  } while (0)

// Host->device upload ordered on the handle's (non-blocking) stream.  NOT cudaMemcpy:
// for pageable sources that call may return before the DMA of the last staged chunk has
// landed and is only ordered against the legacy default stream -- a kernel on h->stream
// launched right after could read a stale tail.
cudaError_t h2d(cs_b200_handle* h, void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return cudaSuccess;
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream);
  if (e != cudaSuccess) return e;
  return cudaStreamSynchronize(h->stream);   // the source buffers are short-lived host vectors
}

int kt_index(int kt) { return kt == 1 ? 0 : kt == 2 ? 1 : kt == 4 ? 2 : 3; }

// greedy row blocks: <= NNZ_CAP nnz and <= NT rows; an over-long row stands alone.
void build_row_blocks(const std::vector<int>& rowptr, int64_t n, std::vector<int>& bstart,
                      int max_rows = NT) {
  bstart.clear();
  bstart.push_back(0);
  int64_t r = 0;
  while (r < n) {
    int64_t r1 = r + 1;
    const int64_t base = rowptr[r];
    while (r1 < n && (r1 - r) < max_rows && (int64_t)rowptr[r1 + 1] - base <= NNZ_CAP) ++r1;
    bstart.push_back((int)r1);
    r = r1;
  }
}

template <typename T>
int build_windowed(cs_b200_handle* h, DevCsr& d, const int* rowptr, const int* colidx, int64_t ncols_pad,
                   const T* d_dinv = nullptr);

// upload one host CSR (double values) as a device CSR of T with its row blocks
// debugging aid: CS_B200_WIN_MASK bit 0 = finest A, 1 = coarse A, 2 = P, 3 = R (default all)
int win_mask() {
  const char* e = getenv("CS_B200_WIN_MASK");
  return e ? atoi(e) : 15;
}

template <typename T>
int upload_csr(cs_b200_handle* h, const csb_amg::Csr& m, DevCsr& d, bool windowed, const T* d_dinv = nullptr) {
  d.nrows = (int)m.nrows;
  d.nnz = m.nnz();
  d.lpr = (m.nrows > 0 && (double)d.nnz / (double)m.nrows >= 20.0) ? 4 : 1;
  // small operators (coarse levels): shrink the row blocks so that >= 4 CTAs per SM exist --
  // their kernels are latency-bound chains of dependent gathers, not bandwidth-bound
  const int unit = d.lpr == 4 ? 8 : 32;          // rows per pass of k_spmm at KT = 8
  int max_rows = (int)((m.nrows + 4 * h->num_sms - 1) / (4 * h->num_sms));
  max_rows = std::min(NT, std::max(unit, (max_rows + unit - 1) / unit * unit));
  std::vector<int> bstart;
  build_row_blocks(m.ptr, m.nrows, bstart, max_rows);
  d.nblocks = (int)bstart.size() - 1;
  std::vector<T> v(m.val.begin(), m.val.end());
  CK(h, cudaMalloc(&d.rowptr, (size_t)(m.nrows + 1) * sizeof(int)));
  CK(h, cudaMalloc(&d.colidx, std::max<size_t>(1, (size_t)d.nnz) * sizeof(int)));
  CK(h, cudaMalloc(&d.vals, std::max<size_t>(1, (size_t)d.nnz) * sizeof(T)));
  CK(h, cudaMalloc(&d.bstart, bstart.size() * sizeof(int)));
  CK(h, h2d(h, d.rowptr, m.ptr.data(), (size_t)(m.nrows + 1) * sizeof(int)));
  CK(h, h2d(h, d.colidx, m.idx.data(), (size_t)d.nnz * sizeof(int)));
  CK(h, h2d(h, d.vals, v.data(), (size_t)d.nnz * sizeof(T)));
  CK(h, h2d(h, d.bstart, bstart.data(), bstart.size() * sizeof(int)));
  if (h->opts.window >= 0 && windowed) {
    const int64_t ncols_pad = (m.ncols + 3) / 4 * 4;
    return build_windowed<T>(h, d, m.ptr.data(), m.idx.data(), ncols_pad, d_dinv);
  }
  return CS_B200_OK;
}

void free_win(DevCsr& d) {
  cudaFree(d.win_meta); cudaFree(d.blob); cudaFree(d.dia); cudaFree(d.ell_col); cudaFree(d.ell_val);
  d.win_meta = nullptr; d.blob = nullptr; d.dia = nullptr; d.ell_col = nullptr; d.ell_val = nullptr;
}

void free_csr(DevCsr& d) {
  cudaFree(d.rowptr); cudaFree(d.colidx); cudaFree(d.vals); cudaFree(d.bstart);
  free_win(d);
  d = DevCsr{};
}

// Build + upload the windowed row-block form of a CSR already resident in `d`.
// rowptr/colidx: host copies; ncols_pad: rows of the input panel (n_pad of the column space).
template <typename T>
int build_windowed(cs_b200_handle* h, DevCsr& d, const int* rowptr, const int* colidx, int64_t ncols_pad,
                   const T* d_dinv) {
  static_assert(sizeof(WinMeta) == sizeof(csb_win::BlockMeta), "meta layout");
  static_assert(W_RB == csb_win::RB && W_WCAP == csb_win::WCAP && W_WCAP_WIDE == csb_win::WCAP_WIDE && W_NNZ == csb_win::NNZ_CAP &&
                W_MAXSEG == csb_win::MAXSEG, "window geometry");
  csb_win::Windowed w = csb_win::build(rowptr, colidx, d.nrows, ncols_pad, (int)sizeof(T),
                                       d.lpr == 4 ? csb_win::WCAP_WIDE : csb_win::WCAP, d_dinv != nullptr);
  d.has_dinv = d_dinv != nullptr ? 1 : 0;
  d.win_blocks = w.windowed_blocks;
  d.win_nblocks = (int)w.meta.size();
  if (w.windowed_blocks * 2 < (int64_t)w.meta.size()) return CS_B200_OK;   // mostly scattered: keep the plain kernel
  const size_t ne = w.lcol.size();
  int* d_perm = nullptr;
  int* d_roff_off = nullptr;
  unsigned short *d_lcol = nullptr, *d_roff = nullptr;
  CK(h, cudaMalloc(&d.win_meta, w.meta.size() * sizeof(WinMeta)));
  CK(h, cudaMalloc(&d.blob, (size_t)w.blob_bytes));
  CK(h, cudaMalloc(&d_lcol, ne * sizeof(unsigned short)));
  CK(h, cudaMalloc(&d_roff, w.roff.size() * sizeof(unsigned short)));
  CK(h, cudaMalloc(&d_roff_off, w.roff_off.size() * sizeof(int)));
  CK(h, cudaMalloc(&d_perm, ne * sizeof(int)));
  CK(h, h2d(h, d.win_meta, w.meta.data(), w.meta.size() * sizeof(WinMeta)));
  CK(h, h2d(h, d_lcol, w.lcol.data(), ne * sizeof(unsigned short)));
  CK(h, h2d(h, d_roff, w.roff.data(), w.roff.size() * sizeof(unsigned short)));
  CK(h, h2d(h, d_roff_off, w.roff_off.data(), w.roff_off.size() * sizeof(int)));
  CK(h, h2d(h, d_perm, w.perm_off.data(), ne * sizeof(int)));
  CK(h, cudaMemsetAsync(d.blob, 0, (size_t)w.blob_bytes, h->stream));
  k_pack_blob<T><<<std::max(1, std::min(d.win_nblocks, h->num_sms * 16)), 128, 0, h->stream>>>(
      d.win_nblocks, d.win_meta, d_perm, d_lcol, d_roff, d_roff_off, (const T*)d.vals, d_dinv, d.blob);
  CK(h, cudaGetLastError());
  CK(h, cudaStreamSynchronize(h->stream));
  cudaFree(d_lcol);
  cudaFree(d_roff);
  cudaFree(d_roff_off);
  cudaFree(d_perm);
  return CS_B200_OK;
}

// Upload a host hierarchy as device levels of type TV.  `own0`: the finest level gets its own
// device CSR (float copy for the mixed-precision cycle); otherwise it aliases the handle's.
template <typename TV>
int upload_levels(cs_b200_handle* h, const csb_amg::Hierarchy& hier, std::vector<DevLevel>& lv, bool own0) {
  const int nl = (int)hier.levels.size();
  lv.resize(nl);
  for (int l = 0; l < nl; ++l) {
    const csb_amg::HostLevel& hl = hier.levels[l];
    DevLevel& L = lv[l];
    L.n = hl.A.nrows;
    L.n_pad = (L.n + 3) / 4 * 4;
    L.omega = hl.omega;
    if (l == 0 && !own0) {
      L.A = h->A0;  // alias, not owned
      L.dinv = h->d_dinv;
    } else {
      std::vector<TV> dv(L.n_pad, TV(0));
      for (int64_t i = 0; i < L.n; ++i) dv[i] = (TV)hl.dinv[i];
      CK(h, cudaMalloc(&L.dinv, (size_t)L.n_pad * sizeof(TV)));
      CK(h, h2d(h, L.dinv, dv.data(), (size_t)L.n_pad * sizeof(TV)));
      const bool win = h->opts.window > 0 || (L.n >= 20000 && (win_mask() & (l == 0 ? 1 : 2)));
      int rc = upload_csr<TV>(h, hl.A, L.A, win, (const TV*)L.dinv);
      if (rc) return rc;
      if (l > 0) {
        const size_t pe = (size_t)L.n_pad * h->ktmax * sizeof(TV);
        void** bufs[] = {&L.x, &L.b, &L.t, &L.y};
        for (void** bp : bufs) {
          CK(h, cudaMalloc(bp, pe));
          CK(h, cudaMemsetAsync(*bp, 0, pe, h->stream));
        }
      }
    }
    if (l + 1 < nl) {
      int rc = upload_csr<TV>(h, hl.P, L.P, L.n >= 20000 && (win_mask() & 4));
      if (rc) return rc;
      rc = upload_csr<TV>(h, hl.R, L.R, L.n >= 20000 && (win_mask() & 8));
      if (rc) return rc;
    }
  }
  return CS_B200_OK;
}

// Smoothed-aggregation hierarchy: built on the host (amg_host.hpp), resident on the device.
template <typename T>
int setup_amg(cs_b200_handle* h, const std::vector<int>& rp, const std::vector<int>& ci,
              const T* vals_host) {
  csb_amg::Csr a0;
  a0.nrows = a0.ncols = h->n;
  a0.ptr = rp;
  a0.idx = ci;
  a0.val.assign(vals_host, vals_host + h->nnz);
  Tick tick;
  csb_amg::Hierarchy hier = csb_amg::build_hierarchy(std::move(a0));
  tick("host hierarchy");
  h->amg_opc = hier.operator_complexity();
  const int nl = (int)hier.levels.size();
  // fp64 handles run the V-cycle in fp32 (opts.mixed: 0 auto = on, -1 off): the preconditioner
  // only has to be a good approximate inverse, CG's own vectors stay fp64
  h->mixed = nl > 1 && sizeof(T) == 8 && h->opts.mixed >= 0;
  int rc = h->mixed ? upload_levels<float>(h, hier, h->lv32, true) : CS_B200_OK;
  if (rc) return rc;
  tick("levels: windows + upload");
  if (h->mixed) {
    // the fp64 side only needs level 0's omega / dinv (already on the handle)
    h->lv.resize(nl);
    for (int l = 0; l < nl; ++l) { h->lv[l].n = hier.levels[l].A.nrows; h->lv[l].omega = hier.levels[l].omega; }
    h->lv[0].A = h->A0;
    h->lv[0].dinv = h->d_dinv;
    const size_t pe = (size_t)h->n_pad * h->ktmax * sizeof(float);
    void** bufs[] = {&h->R32, &h->X32, &h->T32, &h->Z32};
    for (void** bp : bufs) {
      CK(h, cudaMalloc(bp, pe));
      CK(h, cudaMemsetAsync(*bp, 0, pe, h->stream));
    }
  } else {
    rc = upload_levels<T>(h, hier, h->lv, false);
    if (rc) return rc;
    const size_t pe = (size_t)h->n_pad * h->ktmax * sizeof(T);
    CK(h, cudaMalloc(&h->Z, pe));
    CK(h, cudaMemsetAsync(h->Z, 0, pe, h->stream));
  }
  const size_t nc = (size_t)hier.levels.back().A.nrows;
  if (hier.coarse_pinv.size() == nc * nc && nc > 0) {
    CK(h, cudaMalloc(&h->d_pinv, nc * nc * sizeof(double)));
    CK(h, h2d(h, h->d_pinv, hier.coarse_pinv.data(), nc * nc * sizeof(double)));
  }
  CK(h, cudaStreamSynchronize(h->stream));
  h->amg = nl > 1;
  return CS_B200_OK;
}

// panels, 1/diag, current vectors, control block: what every handle needs whatever built its operators
template <typename T>
int alloc_common(cs_b200_handle* h) {
  const size_t pe = (size_t)h->n_pad * h->ktmax;
  void** bufs[] = {&h->X, &h->R, &h->P, &h->AP, &h->B, &h->stage};
  const char* ve = std::getenv("CS_B200_VERBOSE");
  const bool v2 = ve && std::atoi(ve) >= 2;
  auto t0 = std::chrono::steady_clock::now();
  auto stamp = [&](const char* what) {
    if (!v2) return;
    cudaStreamSynchronize(h->stream);
    const auto t1 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[cs_b200 setup/stamp]        %-34s %8.2f ms\n", what,
                 std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  };
  stamp("alloc_common: entry (pending work)");
  for (void** b : bufs) {
    CK(h, cudaMalloc(b, pe * sizeof(T)));
    CK(h, cudaMemsetAsync(*b, 0, pe * sizeof(T), h->stream));
  }
  stamp("alloc_common: 6 panels");
  CK(h, cudaMalloc(&h->d_dinv, (size_t)h->n_pad * sizeof(T)));
  CK(h, cudaMalloc(&h->d_cum, (size_t)h->n_pad * sizeof(T)));
  CK(h, cudaMalloc(&h->d_max, (size_t)h->n_pad * sizeof(T)));
  CK(h, cudaMalloc(&h->d_ctl, sizeof(PanelCtl)));
  CK(h, cudaMemsetAsync(h->d_ctl, 0, sizeof(PanelCtl), h->stream));
  stamp("alloc_common: dinv/cum/max/ctl");
  CK(h, cudaMallocHost(&h->h_ctl, sizeof(PanelCtl)));
  stamp("alloc_common: cudaMallocHost");
  const int maxgrid = h->num_sms * 8;
  CK(h, cudaMalloc(&h->d_partials, (size_t)maxgrid * 2 * MAXKT * sizeof(double)));
  k_dinv<T><<<std::min<int64_t>((h->n_pad + 255) / 256, 4096), 256, 0, h->stream>>>(
      (int)h->n, (int)h->n_pad, h->d_rowptr, h->d_colidx, (const T*)h->d_vals, (T*)h->d_dinv);
  CK(h, cudaGetLastError());
  stamp("alloc_common: k_dinv");
  return CS_B200_OK;
}

template <typename T>
int finish_setup(cs_b200_handle* h, const std::vector<int>& h_rowptr, const std::vector<int>* h_colidx,
                 const T* h_vals) {
  std::vector<int> bstart;
  build_row_blocks(h_rowptr, h->n, bstart);
  h->nblocks = (int)bstart.size() - 1;
  CK(h, cudaMalloc(&h->d_bstart, bstart.size() * sizeof(int)));
  CK(h, cudaMemcpyAsync(h->d_bstart, bstart.data(), bstart.size() * sizeof(int),
                        cudaMemcpyHostToDevice, h->stream));
  h->A0 = DevCsr{h->d_rowptr, h->d_colidx, h->d_vals, h->d_bstart, h->nblocks, (int)h->n, h->nnz, 1};
  int rc0 = alloc_common<T>(h);
  if (rc0) return rc0;
  CK(h, cudaStreamSynchronize(h->stream));
  std::vector<int> ci_local;
  std::vector<T> v_local;
  const bool want_win = h->opts.window >= 0 && (h->opts.window > 0 || h->n >= 20000) && (win_mask() & 1);
  const bool want_amg = h->opts.precond == CS_B200_PRECOND_AMG;
  if (!h_colidx && (want_win || want_amg)) {  // matrix arrived on the device (NCCL broadcast)
    ci_local.resize(h->nnz);
    CK(h, cudaMemcpy(ci_local.data(), h->d_colidx, (size_t)h->nnz * sizeof(int), cudaMemcpyDeviceToHost));
    h_colidx = &ci_local;
    if (want_amg) {
      v_local.resize(h->nnz);
      CK(h, cudaMemcpy(v_local.data(), h->d_vals, (size_t)h->nnz * sizeof(T), cudaMemcpyDeviceToHost));
      h_vals = v_local.data();
    }
  }
  Tick tick;
  if (want_win) {
    int rc = build_windowed<T>(h, h->A0, h_rowptr.data(), h_colidx->data(), h->n_pad, (const T*)h->d_dinv);
    if (rc) return rc;
    tick("finest operator: windows");
  }
  if (want_amg) {
    int rc = setup_amg<T>(h, h_rowptr, *h_colidx, h_vals);
    if (rc) return rc;
  }
  return cs_b200_reset_currents(h);
}

// ---------------------------------------------------------------------------------------------
// device-side setup (setup_device.cu): row blocks, windowed records and the multigrid hierarchy are
// built on the GPU from the resident CSR; only the ordered aggregation seed pass runs on the host
// ---------------------------------------------------------------------------------------------
int rc_dev(cs_b200_handle* h, int rc) {   // csb_dev codes -> cs_b200 status (h->err already set)
  (void)h;
  if (rc == 0) return CS_B200_OK;
  return rc == -5 ? CS_B200_ERR_UNSUPPORTED : CS_B200_ERR_CUDA;
}

// plain-kernel row blocks of a device CSR (the partition build_row_blocks computes on the host)
int device_row_blocks(cs_b200_handle* h, DevCsr& d, int max_rows) {
  int* bs = nullptr;
  int nb = 0;
  int rc = csb_dev::row_blocks(h->stream, d.rowptr, d.nrows, max_rows, NNZ_CAP, &bs, &nb, h->err);
  if (rc) return rc_dev(h, rc);
  d.bstart = bs;
  d.nblocks = nb;
  return CS_B200_OK;
}

template <typename T>
int device_windows(cs_b200_handle* h, DevCsr& d, int64_t ncols_pad, const T* d_dinv) {
  csb_dev::DWin w;
  int rc = csb_dev::build_windowed<T>(h->stream, d.rowptr, d.colidx, (const T*)d.vals, d.nrows, ncols_pad,
                                      d.lpr == 4 ? W_WCAP_WIDE : W_WCAP, d_dinv, w, h->err);
  if (rc) return rc_dev(h, rc);
  d.has_dinv = d_dinv != nullptr ? 1 : 0;
  d.win_blocks = w.windowed_blocks;
  d.win_nblocks = w.nblocks;
  d.win_meta = reinterpret_cast<WinMeta*>(w.meta);
  d.blob = w.blob;
  return CS_B200_OK;
}

// stencil (DIA) form of a square operator, if its pattern allows it (opts.stencil: 0 auto, 1, -1 never)
template <typename T>
int device_stencil(cs_b200_handle* h, DevCsr& d) {
  static const bool env_off = std::getenv("CS_B200_NO_STENCIL") != nullptr;
  if (h->opts.stencil < 0 || env_off) return CS_B200_OK;
  if (h->opts.stencil == 0 && d.nrows < 20000) return CS_B200_OK;
  T* dia = nullptr;
  int nr = 0;
  size_t ld = 0;
  int rc = csb_dev::build_dia<T>(h->stream, d.rowptr, d.colidx, (const T*)d.vals, d.nrows, &dia, &nr, &ld, h->err);
  if (rc) return rc_dev(h, rc);
  d.dia = dia;
  d.dia_nr = nr;
  d.dia_ld = ld;
  return CS_B200_OK;
}

// take over a hierarchy operator as a device CSR of TV: the index arrays move (or are duplicated when
// the source is the handle's own matrix), the fp64 values move or are converted
template <typename TV>
int adopt_csr(cs_b200_handle* h, csb_dev::DCsr& src, bool duplicate, DevCsr& d, bool windowed, const TV* d_dinv) {
  d.nrows = (int)src.nrows;
  d.nnz = src.nnz;
  d.lpr = (src.nrows > 0 && (double)d.nnz / (double)src.nrows >= 20.0) ? 4 : 1;
  const size_t np = (size_t)src.nrows + 1, ne = std::max<size_t>(1, (size_t)src.nnz);
  if (duplicate) {
    CK(h, cudaMalloc(&d.rowptr, np * sizeof(int)));
    CK(h, cudaMalloc(&d.colidx, ne * sizeof(int)));
    CK(h, cudaMemcpyAsync(d.rowptr, src.ptr, np * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    CK(h, cudaMemcpyAsync(d.colidx, src.idx, (size_t)src.nnz * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
  } else {
    d.rowptr = src.ptr; src.ptr = nullptr;
    d.colidx = src.idx; src.idx = nullptr;
  }
  if (sizeof(TV) == 8 && !duplicate) {
    d.vals = src.val; src.val = nullptr;
  } else {
    CK(h, cudaMalloc(&d.vals, ne * sizeof(TV)));
    if (sizeof(TV) == 8) {
      CK(h, cudaMemcpyAsync(d.vals, src.val, (size_t)src.nnz * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    } else if (csb_dev::convert_values(h->stream, src.val, (float*)d.vals, src.nnz)) {
      return set_err(h, CS_B200_ERR_CUDA, "value conversion launch failed");
    }
    if (!duplicate) {
      CK(h, cudaStreamSynchronize(h->stream));
      cudaFree(src.val); src.val = nullptr;
    }
  }
  // small operators (coarse levels): shrink the row blocks so that >= 4 CTAs per SM exist
  const int unit = d.lpr == 4 ? 8 : 32;
  int max_rows = (int)((src.nrows + 4 * h->num_sms - 1) / (4 * h->num_sms));
  max_rows = std::min(NT, std::max(unit, (max_rows + unit - 1) / unit * unit));
  int rc = device_row_blocks(h, d, max_rows);
  if (rc) return rc;
  if (src.nrows == src.ncols && d_dinv != nullptr) {   // square level operator: stencil form if it has one
    rc = device_stencil<TV>(h, d);
    if (rc) return rc;
    if (d.dia) return CS_B200_OK;
  }
  if (h->opts.window >= 0 && windowed) {
    const int64_t ncols_pad = (src.ncols + 3) / 4 * 4;
    return device_windows<TV>(h, d, ncols_pad, d_dinv);
  }
  return CS_B200_OK;
}

template <typename TV>
int adopt_levels(cs_b200_handle* h, csb_dev::DHierarchy& hier, std::vector<DevLevel>& lv, bool own0) {
  const int nl = (int)hier.levels.size();
  lv.resize(nl);
  Tick lt;
  auto mark = [&](int l, const char* what) {
    if (!lt.on) return;
    cudaStreamSynchronize(h->stream);
    char buf[64];
    snprintf(buf, sizeof buf, "  L%d %s", l, what);
    lt(buf);
  };
  for (int l = 0; l < nl; ++l) {
    csb_dev::DLevel& hl = hier.levels[l];
    DevLevel& L = lv[l];
    L.n = hl.A.nrows;
    L.n_pad = (L.n + 3) / 4 * 4;
    L.omega = hl.omega;
    if (l == 0 && !own0) {
      L.A = h->A0;  // alias, not owned
      L.dinv = h->d_dinv;
    } else {
      CK(h, cudaMalloc(&L.dinv, (size_t)L.n_pad * sizeof(TV)));
      CK(h, cudaMemsetAsync(L.dinv, 0, (size_t)L.n_pad * sizeof(TV), h->stream));
      if (sizeof(TV) == 8) {
        CK(h, cudaMemcpyAsync(L.dinv, hl.dinv, (size_t)L.n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
      } else if (csb_dev::convert_values(h->stream, hl.dinv, (float*)L.dinv, L.n)) {
        return set_err(h, CS_B200_ERR_CUDA, "dinv conversion launch failed");
      }
      const bool win = h->opts.window > 0 || (L.n >= 20000 && (win_mask() & (l == 0 ? 1 : 2)));
      int rc = adopt_csr<TV>(h, hl.A, l == 0, L.A, win, (const TV*)L.dinv);
      if (rc) return rc;
      mark(l, "A: copy/convert, blocks, windows");
      if (l > 0) {
        const size_t pe = (size_t)L.n_pad * h->ktmax * sizeof(TV);
        void** bufs[] = {&L.x, &L.b, &L.t, &L.y};
        for (void** bp : bufs) {
          CK(h, cudaMalloc(bp, pe));
          CK(h, cudaMemsetAsync(*bp, 0, pe, h->stream));
        }
      }
    }
    if (l + 1 < nl) {
      int rc = adopt_csr<TV>(h, hl.P, false, L.P, L.n >= 20000 && (win_mask() & 4), (const TV*)nullptr);
      if (rc) return rc;
      if (L.A.dia) {          // the fused prolongation kernel of this level reads P as ELL-4 when it can
        int* ec = nullptr;
        TV* ev = nullptr;
        size_t eld = 0;
        int rce = csb_dev::build_ell4<TV>(h->stream, L.P.rowptr, L.P.colidx, (const TV*)L.P.vals, L.P.nrows, &ec, &ev, &eld, h->err);
        if (rce) return rc_dev(h, rce);
        L.P.ell_col = ec; L.P.ell_val = ev; L.P.ell_ld = eld;
      }
      mark(l, "P");
      rc = adopt_csr<TV>(h, hl.R, false, L.R, L.n >= 20000 && (win_mask() & 8), (const TV*)nullptr);
      if (rc) return rc;
      mark(l, "R");
    }
  }
  return CS_B200_OK;
}

template <typename T>
int setup_amg_device(cs_b200_handle* h, const csb_dev::HostPattern& hp, csb_dev::SeedJob* job,
                     const csb_dev::DeviceSeed* dseed) {
  const bool verbose = std::getenv("CS_B200_VERBOSE") != nullptr;
  csb_dev::DCsr a0;
  a0.nrows = a0.ncols = h->n;
  a0.nnz = h->nnz;
  a0.ptr = h->d_rowptr;
  a0.idx = h->d_colidx;
  double* tmp64 = nullptr;
  if (sizeof(T) == 8) {
    a0.val = (double*)h->d_vals;
  } else {   // the hierarchy is built in fp64 whatever the handle computes in
    cudaError_t e = cudaMalloc(&tmp64, std::max<size_t>(1, (size_t)h->nnz) * sizeof(double));
    if (e != cudaSuccess) {
      csb_dev::seed_discard(job);
      return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (fp64 copy of the matrix)", cudaGetErrorString(e));
    }
    csb_dev::convert_values(h->stream, (const float*)h->d_vals, tmp64, h->nnz);
    a0.val = tmp64;
  }
  Tick tick;
  csb_dev::DHierarchy hier;
  int rc = csb_dev::build_hierarchy(h->stream, a0, hp, job, dseed, 12, 200, hier, h->err, verbose);
  auto done = [&](int code) {
    cudaStreamSynchronize(h->stream);
    csb_dev::free_hierarchy(hier);
    cudaFree(tmp64);
    return code;
  };
  if (rc) return done(rc_dev(h, rc));
  tick("device hierarchy");
  h->amg_opc = hier.operator_complexity;
  const int nl = (int)hier.levels.size();
  h->mixed = nl > 1 && sizeof(T) == 8 && h->opts.mixed >= 0;
  if (h->mixed) {
    rc = adopt_levels<float>(h, hier, h->lv32, true);
    if (rc) return done(rc);
    h->lv.resize(nl);
    for (int l = 0; l < nl; ++l) { h->lv[l].n = hier.levels[l].A.nrows; h->lv[l].omega = hier.levels[l].omega; }
    h->lv[0].A = h->A0;
    h->lv[0].dinv = h->d_dinv;
    const size_t pe = (size_t)h->n_pad * h->ktmax * sizeof(float);
    void** bufs[] = {&h->R32, &h->X32, &h->T32, &h->Z32};
    for (void** bp : bufs) {
      cudaError_t e = cudaMalloc(bp, pe);
      if (e == cudaSuccess) e = cudaMemsetAsync(*bp, 0, pe, h->stream);
      if (e != cudaSuccess) return done(set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (fp32 panels)", cudaGetErrorString(e)));
    }
  } else {
    rc = adopt_levels<T>(h, hier, h->lv, false);
    if (rc) return done(rc);
    const size_t pe = (size_t)h->n_pad * h->ktmax * sizeof(T);
    cudaError_t e = cudaMalloc(&h->Z, pe);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->Z, 0, pe, h->stream);
    if (e != cudaSuccess) return done(set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (Z panel)", cudaGetErrorString(e)));
  }
  tick("levels: row blocks + windows");
  csb_dev::coarse_pinv_wait(hier);
  tick("coarse pseudo-inverse (wait)");
  const size_t nc = (size_t)hier.levels.back().A.nrows;
  if (hier.coarse_pinv.size() == nc * nc && nc > 0) {
    cudaError_t e = cudaMalloc(&h->d_pinv, nc * nc * sizeof(double));
    if (e == cudaSuccess) e = h2d(h, h->d_pinv, hier.coarse_pinv.data(), nc * nc * sizeof(double));
    if (e != cudaSuccess) return done(set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (coarse pseudo-inverse)", cudaGetErrorString(e)));
  }
  h->amg = nl > 1;
  return done(CS_B200_OK);
}

template <typename T>
int build_operators(cs_b200_handle* h, const csb_dev::HostPattern& hp, csb_dev::SeedJob* job,
                    const csb_dev::DeviceSeed* dseed);

template <typename T>
int finish_setup_device(cs_b200_handle* h, const csb_dev::HostPattern& hp, csb_dev::SeedJob* job,
                        const csb_dev::DeviceSeed* dseed = nullptr) {
  h->A0 = DevCsr{h->d_rowptr, h->d_colidx, h->d_vals, nullptr, 0, (int)h->n, h->nnz, 1};
  Tick tick0;
  int rc = device_row_blocks(h, h->A0, NT);
  if (rc) { csb_dev::seed_discard(job); return rc; }
  h->d_bstart = h->A0.bstart;
  h->nblocks = h->A0.nblocks;
  rc = alloc_common<T>(h);
  if (rc) { csb_dev::seed_discard(job); return rc; }
  if (tick0.on) { cudaStreamSynchronize(h->stream); tick0("row blocks + panels"); }
  rc = build_operators<T>(h, hp, job, dseed);
  if (rc) return rc;
  return cs_b200_reset_currents(h);
}

// 1/diag, the finest operator's stencil / window form, the multigrid hierarchy: everything that depends
// on the matrix VALUES (re-run by cs_b200_set_grounds after the values changed)
template <typename T>
int build_operators(cs_b200_handle* h, const csb_dev::HostPattern& hp, csb_dev::SeedJob* job,
                    const csb_dev::DeviceSeed* dseed) {
  int rc = CS_B200_OK;
  k_dinv<T><<<std::min<int64_t>((h->n_pad + 255) / 256, 4096), 256, 0, h->stream>>>(
      (int)h->n, (int)h->n_pad, h->d_rowptr, h->d_colidx, (const T*)h->d_vals, (T*)h->d_dinv);
  const bool want_win = h->opts.window >= 0 && (h->opts.window > 0 || h->n >= 20000) && (win_mask() & 1);
  const bool want_amg = h->opts.precond == CS_B200_PRECOND_AMG;
  Tick tick;
  if (want_win) {
    rc = device_stencil<T>(h, h->A0);
    if (!rc && !h->A0.dia) rc = device_windows<T>(h, h->A0, h->n_pad, (const T*)h->d_dinv);
    if (rc) { csb_dev::seed_discard(job); return rc; }
    tick(h->A0.dia ? "finest operator: stencil form" : "finest operator: windows");
  }
  if (want_amg) {
    rc = setup_amg_device<T>(h, hp, job, dseed);
    if (rc) return rc;
  } else {
    csb_dev::seed_discard(job);
  }
  Tick tick1;
  csb_dev::trim_pool(h->device);
  tick1("scratch pool released");
  return CS_B200_OK;
}

int common_create(cs_b200_handle* h, const cs_b200_opts* opts) {
  if (opts) h->opts = *opts;
  if (h->opts.panel_width == 0) h->opts.panel_width = 8;
  if (h->opts.check_every <= 0) h->opts.check_every = 16;
  if (h->opts.resid_gate <= 0) h->opts.resid_gate = 1e-4;
  if (h->opts.use_graph == 0) h->opts.use_graph = 1;  // 0 -> default on; pass -1 to disable
  const int pw = h->opts.panel_width;
  if (pw != 1 && pw != 2 && pw != 4 && pw != 8)
    return set_err(h, CS_B200_ERR_ARG, "panel_width must be 1, 2, 4 or 8 (got %d)", pw);
  h->ktmax = pw;
  if (h->opts.precond != CS_B200_PRECOND_JACOBI && h->opts.precond != CS_B200_PRECOND_AMG)
    return set_err(h, CS_B200_ERR_UNSUPPORTED, "unknown preconditioner %d", h->opts.precond);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return set_err(h, CS_B200_ERR_CUDA,
                   "no CUDA device available (%s): libcsb200 has no CPU fallback",
                   cudaGetErrorString(e));
  if (h->device < 0 || h->device >= ndev)
    return set_err(h, CS_B200_ERR_ARG, "device %d out of range (0..%d)", h->device, ndev - 1);
  CK(h, cudaSetDevice(h->device));
  cudaDeviceProp prop;
  CK(h, cudaGetDeviceProperties(&prop, h->device));
  h->num_sms = prop.multiProcessorCount;
  h->grid_spmm = h->num_sms * 8;
  h->grid_ew = h->num_sms * 4;
  CK(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(h, cudaEventCreate(&h->ev0));
  CK(h, cudaEventCreate(&h->ev1));
  CK(h, cudaEventCreate(&h->ev2));
  CK(h, cudaEventCreate(&h->ev3));
  h->n_pad = (h->n + 3) / 4 * 4;
  return CS_B200_OK;
}

template <typename I>
void narrow_indices(const I* src, int64_t count, int base, std::vector<int>& dst) {
  dst.resize(count);
  for (int64_t i = 0; i < count; ++i) dst[i] = (int)(src[i] - base);
}

// ---------------------------------------------------------------------------
// launch helpers (all on h->stream)
// ---------------------------------------------------------------------------
template <typename T>
CsrDev<T> view(const DevCsr& m) {
  return CsrDev<T>{m.rowptr, m.colidx, (const T*)m.vals, m.bstart, m.nblocks, m.nrows};
}

// Y = op(M X) with the fused epilogue MODE (kernels.cuh).  `timed`: counts as a launch of
// the dominant kernel for the per-launch profile (finest-level operator only).
template <typename T, int KT, int MODE>
void launch_spmm_on(cs_b200_handle* h, const DevCsr& m, const T* X, T* Y, const T* B, const T* dinv,
                    double omega, bool timed) {
  const int grid = std::max(1, std::min(h->grid_spmm, m.nblocks));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool prof = h->profile && timed;
  if (prof) {
    if (h->prof_used + 2 > h->prof_ev.size()) {
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e); }
    }
    e0 = h->prof_ev[h->prof_used++];
    e1 = h->prof_ev[h->prof_used++];
    // nnz (s_v + 4) + (n + 1) 4 + X once + Y once (+ B for the residual / sweep epilogues,
    // + 1/diag for the sweeps)
    double bytes = (double)m.nnz * (sizeof(T) + 4) + (double)(m.nrows + 1) * 4 +
                   2.0 * (double)m.nrows * KT * sizeof(T);
    if (MODE == SP_RESNORM || MODE == SP_RES || MODE == SP_JACOBI || MODE == SP_JACOBI_DOT)
      bytes += (double)m.nrows * KT * sizeof(T);
    if (MODE == SP_JACOBI || MODE == SP_JACOBI_DOT) bytes += (double)m.nrows * sizeof(T);
    h->prof_bytes += bytes;
    h->prof_slot.push_back(2 * MODE + (sizeof(T) == 4 ? 1 : 0));
    h->prof_pair_bytes.push_back(bytes);
    cudaEventRecord(e0, h->stream);
  }
  const SpmmEpi<T> ep{B, dinv, (T)omega, h->d_ctl, h->d_partials};
  if (m.dia && MODE != SP_ADD) {
    if constexpr (MODE != SP_ADD) {
      const DiaDev<T> a{(const T*)m.dia, m.dia_ld, m.nrows, m.dia_nr};
      constexpr int V16 = 16 / (int)sizeof(T);
      constexpr int CGn = KT / (KT < V16 ? KT : V16);
      const int rpp = NT / CGn;
      const long long ntiles = (long long)((m.dia_nr + rpp - 1) / rpp) *
                               ((((long long)m.nrows + m.dia_nr - 1) / m.dia_nr + ST_TC - 1) / ST_TC);
      const int sg = (int)std::max<long long>(1, std::min<long long>(h->grid_spmm, ntiles));
      k_stencil<T, KT, MODE><<<sg, NT, 0, h->stream>>>(a, X, Y, ep);
    }
  } else if (m.win_meta) {
    const WinCsr<T> w{m.win_meta, m.blob, m.has_dinv, m.rowptr, m.colidx, (const T*)m.vals, m.win_nblocks};
    if (m.lpr == 4) {
      constexpr int SMEM = WinSmem2<T, KT, MODE, true>::TOTAL;
      constexpr int SB = WinMap<T, KT, true>::SB;
      const int wg = std::max(1, std::min(h->num_sms, (m.win_nblocks + SB - 1) / SB));
      static bool once[64] = {};   // per device: the attribute lives in the device's context
      bool& set = once[h->device & 63];
      if (!set) { cudaFuncSetAttribute(k_spmm_win<T, KT, MODE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM); set = true; }
      k_spmm_win<T, KT, MODE, true><<<wg, WTT, SMEM, h->stream>>>(w, X, Y, ep);
    } else {
      constexpr int SMEM = WinSmem2<T, KT, MODE, false>::TOTAL;
      constexpr int SB = WinMap<T, KT, false>::SB;
      const int wg = std::max(1, std::min(h->num_sms, (m.win_nblocks + SB - 1) / SB));
      static bool once[64] = {};
      bool& set = once[h->device & 63];
      if (!set) { cudaFuncSetAttribute(k_spmm_win<T, KT, MODE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM); set = true; }
      k_spmm_win<T, KT, MODE, false><<<wg, WTT, SMEM, h->stream>>>(w, X, Y, ep);
    }
  } else if (m.lpr == 4 && KT * 4 <= 32) {
    k_spmm<T, KT, MODE, (KT * 4 <= 32 ? 4 : 1)><<<grid, NT, 0, h->stream>>>(view<T>(m), X, Y, ep);
  } else {
    k_spmm<T, KT, MODE, 1><<<grid, NT, 0, h->stream>>>(view<T>(m), X, Y, ep);
  }
  if (prof) cudaEventRecord(e1, h->stream);
  h->stats.kernel_launches++;
  if (timed) h->stats.spmm_launches++;
}

template <typename T, int KT, int MODE>
void launch_spmm(cs_b200_handle* h, const T* X, T* Y, const T* B) {
  launch_spmm_on<T, KT, MODE>(h, h->A0, X, Y, B, (const T*)h->d_dinv, 0.0, true);
}

// after a stream sync: fold the recorded SpMM event pairs into the profile totals
void harvest_profile(cs_b200_handle* h) {
  for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->prof_ev[i], h->prof_ev[i + 1]) == cudaSuccess) {
      h->prof_ms += ms;
      h->prof_launches++;
      if (i / 2 < h->prof_slot.size()) {
        const int sl = h->prof_slot[i / 2] & 15;
        h->prof_slot_ms[sl] += ms;
        h->prof_slot_bytes[sl] += h->prof_pair_bytes[i / 2];
        h->prof_slot_launches[sl]++;
      }
    }
  }
  h->prof_used = 0;
  h->prof_slot.clear();
  h->prof_pair_bytes.clear();
}

template <typename T, int KT>
int ew_grid(cs_b200_handle* h) {
  const size_t nelem = (size_t)h->n_pad * KT;
  const size_t per = (size_t)NT * Vec<T>::N;
  return (int)std::min<size_t>(h->grid_ew, (nelem + per - 1) / per);
}

template <typename T, int KT>
int ew_grid_n(cs_b200_handle* h, int64_t n_pad) {
  const size_t nelem = (size_t)n_pad * KT;
  const size_t per = (size_t)NT * Vec<T>::N;
  return (int)std::max<size_t>(1, std::min<size_t>(h->grid_ew, (nelem + per - 1) / per));
}

// stencil-form levels keep the zero-guess Jacobi sweep implicit: x0 = omega D^-1 b is formed on the fly
// by the residual kernel (SP_RES0) and by the fused upward kernel, never stored (CS_B200_NO_IMPLICIT_X0
// switches back to the stored form for A/B runs)
inline bool implicit_x0(const DevLevel& L) {
  static const bool off = std::getenv("CS_B200_NO_IMPLICIT_X0") != nullptr || std::getenv("CS_B200_NO_FUSED_PROLONG") != nullptr;
  return L.A.dia != nullptr && !off;
}

// T = B - A (omega D^-1 B) on a stencil-form level
template <typename T, int KT>
void launch_stencil_res0(cs_b200_handle* h, DevLevel& L, const T* B, T* Tout, bool timed) {
  const DevCsr& m = L.A;
  const DiaDev<T> a{(const T*)m.dia, m.dia_ld, m.nrows, m.dia_nr};
  const SpmmEpi<T> ep{B, (const T*)L.dinv, (T)L.omega, h->d_ctl, h->d_partials};
  constexpr int V16 = 16 / (int)sizeof(T);
  constexpr int CGn = KT / (KT < V16 ? KT : V16);
  const int rpp = NT / CGn;
  const long long ntiles = (long long)((m.dia_nr + rpp - 1) / rpp) *
                           ((((long long)m.nrows + m.dia_nr - 1) / m.dia_nr + ST_TC - 1) / ST_TC);
  const int sg = (int)std::max<long long>(1, std::min<long long>(h->grid_spmm, ntiles));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool prof = h->profile && timed;
  if (prof) {
    if (h->prof_used + 2 > h->prof_ev.size())
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e); }
    e0 = h->prof_ev[h->prof_used++];
    e1 = h->prof_ev[h->prof_used++];
    // what it replaces: the residual SpMM on A (X, B read, T written); the zero-guess sweep is folded in
    const double fb = (double)m.nnz * (sizeof(T) + 4) + (double)(m.nrows + 1) * 4 + 3.0 * (double)m.nrows * KT * sizeof(T);
    h->prof_bytes += fb;
    h->prof_slot.push_back(2 * (int)SP_RES + (sizeof(T) == 4 ? 1 : 0));
    h->prof_pair_bytes.push_back(fb);
    cudaEventRecord(e0, h->stream);
  }
  k_stencil<T, KT, SP_RES0><<<sg, NT, 0, h->stream>>>(a, nullptr, Tout, ep);
  if (prof) cudaEventRecord(e1, h->stream);
  h->stats.kernel_launches++;
  if (timed) h->stats.spmm_launches++;
}

// fused upward step of a stencil-form level (kernels.cuh k_stencil_prolong_jacobi):
//   Yout = (X0 + P Yc) + omega D^-1 (B - A (X0 + P Yc))   [+ dot(B, Yout) on the finest level]
template <typename T, int KT, int MODE>
void launch_prolong_jacobi(cs_b200_handle* h, DevLevel& L, const T* Yc, const T* X0, T* Yout, const T* B, bool timed) {
  const DevCsr& m = L.A;
  const DiaDev<T> a{(const T*)m.dia, m.dia_ld, m.nrows, m.dia_nr};
  const CsrP<T> p{L.P.rowptr, L.P.colidx, (const T*)L.P.vals, L.P.ell_col, (const T*)L.P.ell_val, L.P.ell_ld};
  const SpmmEpi<T> ep{B, (const T*)L.dinv, (T)L.omega, h->d_ctl, h->d_partials};
  constexpr int V16 = 16 / (int)sizeof(T);
  constexpr int CGn = KT / (KT < V16 ? KT : V16);
  constexpr int RPP = NT / CGn;
  constexpr int SMEM = (RPP + 2) * (PJ_TC + 2) * KT * (int)sizeof(T);
  static_assert(SMEM <= 48 * 1024, "tile fits the default dynamic shared memory");
  const long long ntiles = (long long)((m.dia_nr + RPP - 1) / RPP) *
                           ((((long long)m.nrows + m.dia_nr - 1) / m.dia_nr + PJ_TC - 1) / PJ_TC);
  const int grid = (int)std::max<long long>(1, std::min<long long>(h->grid_spmm, ntiles));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool prof = h->profile && timed;
  if (prof) {
    if (h->prof_used + 2 > h->prof_ev.size())
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e); }
    e0 = h->prof_ev[h->prof_used++];
    e1 = h->prof_ev[h->prof_used++];
    // the two launches it replaces: SP_ADD on P (nnz_P (s+4) + (n+1) 4 + Yc + X read + X write) and the
    // Jacobi sweep on A (nnz (s+4) + (n+1) 4 + X + Y + B + 1/diag)
    const double fb = (double)m.nnz * (sizeof(T) + 4) + (double)(m.nrows + 1) * 4 + 3.0 * (double)m.nrows * KT * sizeof(T) +
                      (double)m.nrows * sizeof(T) + (double)L.P.nnz * (sizeof(T) + 4) + (double)(m.nrows + 1) * 4 +
                      2.0 * (double)m.nrows * KT * sizeof(T);
    h->prof_bytes += fb;
    h->prof_slot.push_back(2 * 7 + (sizeof(T) == 4 ? 1 : 0));
    h->prof_pair_bytes.push_back(fb);
    cudaEventRecord(e0, h->stream);
  }
  constexpr int MINB = sizeof(T) == 4 ? 4 : 3;
  k_stencil_prolong_jacobi<T, KT, MODE, MINB><<<grid, NT, SMEM, h->stream>>>(a, p, Yc, X0, Yout, ep);
  if (prof) cudaEventRecord(e1, h->stream);
  h->stats.kernel_launches++;
  if (timed) h->stats.spmm_launches++;
}

// z = M^-1 r : one V(1,1) cycle, damped Jacobi, on panels of width KT.
//   in : h->R (residual, read-only)      out: h->Z ; rho_new = r.z folded into the last kernel
// Level buffers: b = right-hand side, x = running correction, t = residual scratch,
// y = post-smoothed correction.  Finest level: b = R, x = stage, t = AP, y = Z.
struct VcBufs { void *b0, *x0, *t0, *y0; };   // finest-level panels of the cycle

template <typename T, int KT>
void launch_vcycle_on(cs_b200_handle* h, std::vector<DevLevel>& lv, const VcBufs& vb, bool level0_presmoothed) {
  const int nl = (int)lv.size();
  auto B = [&](int l) { return l == 0 ? (T*)vb.b0 : (T*)lv[l].b; };
  auto X = [&](int l) { return l == 0 ? (T*)vb.x0 : (T*)lv[l].x; };
  auto Tm = [&](int l) { return l == 0 ? (T*)vb.t0 : (T*)lv[l].t; };
  auto Y = [&](int l) { return l == 0 ? (T*)vb.y0 : (T*)lv[l].y; };
  for (int l = 0; l < nl - 1; ++l) {
    DevLevel& L = lv[l];
    const size_t nelem = (size_t)L.n_pad * KT;
    if (implicit_x0(L)) {
      launch_stencil_res0<T, KT>(h, L, B(l), Tm(l), l == 0);
    } else {
      if (!(l == 0 && level0_presmoothed)) {
        k_jacobi0<T, KT><<<ew_grid_n<T, KT>(h, L.n_pad), NT, 0, h->stream>>>(
            nelem, B(l), (const T*)L.dinv, (T)L.omega, X(l));
        h->stats.kernel_launches++;
      }
      launch_spmm_on<T, KT, SP_RES>(h, L.A, X(l), Tm(l), B(l), nullptr, 0.0, l == 0);
    }
    launch_spmm_on<T, KT, SP_PLAIN>(h, L.R, Tm(l), B(l + 1), nullptr, nullptr, 0.0, false);
  }
  {
    DevLevel& C = lv[nl - 1];
    if (h->d_pinv) {
      k_coarse_dense<T, KT><<<((int)C.n * KT + NT - 1) / NT, NT, 0, h->stream>>>((int)C.n, h->d_pinv, (const T*)B(nl - 1), Y(nl - 1));
      h->stats.kernel_launches++;
    } else {  // coarsening stalled above the dense limit: 4 damped-Jacobi sweeps (symmetric)
      const int l = nl - 1;
      k_jacobi0<T, KT><<<ew_grid_n<T, KT>(h, C.n_pad), NT, 0, h->stream>>>(
          (size_t)C.n_pad * KT, B(l), (const T*)C.dinv, (T)C.omega, X(l));
      h->stats.kernel_launches++;
      launch_spmm_on<T, KT, SP_JACOBI>(h, C.A, X(l), Y(l), B(l), (const T*)C.dinv, C.omega, false);
      launch_spmm_on<T, KT, SP_JACOBI>(h, C.A, Y(l), X(l), B(l), (const T*)C.dinv, C.omega, false);
      launch_spmm_on<T, KT, SP_JACOBI>(h, C.A, X(l), Y(l), B(l), (const T*)C.dinv, C.omega, false);
    }
  }
  static const bool fuse_off = std::getenv("CS_B200_NO_FUSED_PROLONG") != nullptr;
  for (int l = nl - 2; l >= 0; --l) {
    DevLevel& L = lv[l];
    if (L.A.dia && !fuse_off) {
      // stencil-form level: prolongate + correct + post-smooth in one kernel (x1 stays in shared memory)
      const T* x0 = implicit_x0(L) ? nullptr : X(l);
      if (l == 0) launch_prolong_jacobi<T, KT, SP_JACOBI_DOT>(h, L, Y(l + 1), x0, Y(l), B(l), true);
      else launch_prolong_jacobi<T, KT, SP_JACOBI>(h, L, Y(l + 1), x0, Y(l), B(l), false);
      continue;
    }
    launch_spmm_on<T, KT, SP_ADD>(h, L.P, Y(l + 1), X(l), X(l) /* staged as B */, nullptr, 0.0, false);
    if (l == 0)
      launch_spmm_on<T, KT, SP_JACOBI_DOT>(h, L.A, X(l), Y(l), B(l), (const T*)L.dinv, L.omega, true);
    else
      launch_spmm_on<T, KT, SP_JACOBI>(h, L.A, X(l), Y(l), B(l), (const T*)L.dinv, L.omega, false);
  }
}

// the cycle of this handle: fp32 copies when `mixed`, else the handle's own type
template <typename T, int KT>
void launch_vcycle(cs_b200_handle* h, bool level0_presmoothed) {
  if (h->mixed) {
    const VcBufs vb{h->R32, h->X32, h->T32, h->Z32};
    launch_vcycle_on<float, KT>(h, h->lv32, vb, level0_presmoothed);
  } else {
    const VcBufs vb{h->R, h->stage, h->AP, h->Z};
    launch_vcycle_on<T, KT>(h, h->lv, vb, level0_presmoothed);
  }
}

template <typename T, int KT>
void launch_iteration(cs_b200_handle* h) {
  const size_t nelem = (size_t)h->n_pad * KT;
  const int g = ew_grid<T, KT>(h);
  launch_spmm<T, KT, SP_CG>(h, (const T*)h->P, (T*)h->AP, nullptr);
  if (!h->amg) {
    k_cg_update_r<T, KT><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->AP, (const T*)h->d_dinv,
                                                  (T*)h->R, h->d_ctl, h->d_partials);
    k_cg_update_xp<T, KT><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->R, (const T*)h->d_dinv,
                                                   (T*)h->X, (T*)h->P, h->d_ctl);
    h->stats.kernel_launches += 2;
  } else {
    // r -= alpha Ap with the finest pre-smoothing folded in; V-cycle; then the deferred
    // x += alpha p together with p = z + beta p  (9 instead of 11 panel passes)
    if (h->mixed) {
      k_cg_update_r0<T, KT, float><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->AP, (const T*)h->d_dinv,
                                                            (T)h->lv[0].omega, (T*)h->R,
                                                            implicit_x0(h->lv32[0]) ? nullptr : (float*)h->X32,
                                                            (float*)h->R32, h->d_ctl);
      launch_vcycle<T, KT>(h, true);
      k_cg_update_xp2<T, KT, float><<<g, NT, 0, h->stream>>>(nelem, (const float*)h->Z32, (T*)h->X, (T*)h->P,
                                                             h->d_ctl);
    } else {
      k_cg_update_r0<T, KT, T><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->AP, (const T*)h->d_dinv,
                                                        (T)h->lv[0].omega, (T*)h->R,
                                                        implicit_x0(h->lv[0]) ? nullptr : (T*)h->stage, nullptr,
                                                        h->d_ctl);
      launch_vcycle<T, KT>(h, true);
      k_cg_update_xp2<T, KT, T><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->Z, (T*)h->X, (T*)h->P, h->d_ctl);
    }
    h->stats.kernel_launches += 2;
  }
}

template <typename T, int KT>
int run_chunk(cs_b200_handle* h, int chunk) {
  GraphSlot& gs = h->graphs[kt_index(KT)];
  if (h->opts.use_graph > 0 && !h->profile) {   // use_graph == 2: host-polled chunks
    if (!gs.exec || gs.chunk != chunk) {
      if (gs.exec) cudaGraphExecDestroy(gs.exec);
      gs.exec = nullptr;
      cudaGraph_t graph;
      const int64_t kl = h->stats.kernel_launches, sl = h->stats.spmm_launches;
      CK(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      for (int i = 0; i < chunk; ++i) launch_iteration<T, KT>(h);
      CK(h, cudaStreamEndCapture(h->stream, &graph));
      gs.kernels = h->stats.kernel_launches - kl;
      gs.spmms = h->stats.spmm_launches - sl;
      h->stats.kernel_launches = kl;
      h->stats.spmm_launches = sl;
      CK(h, cudaGraphInstantiate(&gs.exec, graph, 0));
      cudaGraphDestroy(graph);
      gs.chunk = chunk;
    }
    CK(h, cudaGraphLaunch(gs.exec, h->stream));
    h->stats.kernel_launches += gs.kernels;
    h->stats.spmm_launches += gs.spmms;
  } else {
    for (int i = 0; i < chunk; ++i) launch_iteration<T, KT>(h);
    CK(h, cudaGetLastError());
  }
  return CS_B200_OK;
}

// The whole PCG loop of a panel as ONE graph launch: a kernel node that evaluates the loop
// condition, then a WHILE conditional node whose body is one captured iteration followed by
// the condition kernel.  The device decides when to stop (cg_after_precond / k_cg_update_r
// clear ctl->nactive; itmax bounds the loop), the host neither polls nor re-launches.
template <typename T, int KT>
int run_loop(cs_b200_handle* h) {
  GraphSlot& gs = h->graphs[kt_index(KT)];
  if (!gs.loop_exec) {
    cudaGraph_t graph;
    CK(h, cudaGraphCreate(&graph, 0));
    cudaGraphConditionalHandle cond;
    CK(h, cudaGraphConditionalHandleCreate(&cond, graph, 0, cudaGraphCondAssignDefault));
    cudaGraphNode_t n_pre, n_while;
    PanelCtl* ctl = h->d_ctl;
    void* args[] = {&cond, &ctl};
    cudaKernelNodeParams kp = {};
    kp.func = (void*)k_loop_cond;
    kp.gridDim = dim3(1);
    kp.blockDim = dim3(1);
    kp.kernelParams = args;
    CK(h, cudaGraphAddKernelNode(&n_pre, graph, nullptr, 0, &kp));
    cudaGraphNodeParams cp = {cudaGraphNodeTypeConditional};
    cp.conditional.handle = cond;
    cp.conditional.type = cudaGraphCondTypeWhile;
    cp.conditional.size = 1;
    CK(h, cudaGraphAddNode(&n_while, graph, &n_pre, 1, &cp));
    cudaGraph_t body = cp.conditional.phGraph_out[0];
    const int64_t kl = h->stats.kernel_launches, sl = h->stats.spmm_launches;
    CK(h, cudaStreamBeginCaptureToGraph(h->stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
    launch_iteration<T, KT>(h);
    k_loop_cond<<<1, 1, 0, h->stream>>>(cond, h->d_ctl);
    CK(h, cudaStreamEndCapture(h->stream, nullptr));
    gs.loop_kernels = h->stats.kernel_launches - kl + 1;
    gs.loop_spmms = h->stats.spmm_launches - sl;
    h->stats.kernel_launches = kl;
    h->stats.spmm_launches = sl;
    CK(h, cudaGraphInstantiate(&gs.loop_exec, graph, 0));
    cudaGraphDestroy(graph);
  }
  CK(h, cudaGraphLaunch(gs.loop_exec, h->stream));
  return CS_B200_OK;
}

// Solve A X = B for the panel whose B is already staged and whose ctl (src/dst/weight)
// has been uploaded.  Leaves X = solution, AP = B - A X, ctl (host copy) updated.
template <typename T, int KT>
int solve_panel(cs_b200_handle* h, double rtol, int64_t itmax) {
  const size_t nelem = (size_t)h->n_pad * KT;
  // Krylov.jl's default is sqrt(eps(T)); for T = Float32 that (3.5e-4) sits ABOVE the
  // reference's own 1e-4 residual gate, so the fp32 path keeps the fp64 value.
  const double atol = h->opts.atol > 0 ? h->opts.atol
                      : h->opts.atol < 0 ? 0.0
                      : std::sqrt(std::numeric_limits<double>::epsilon());
  const int g = ew_grid<T, KT>(h);
  const int imax = (int)std::min<int64_t>(itmax, std::numeric_limits<int>::max() - 1);
  CK(h, cudaEventRecord(h->ev2, h->stream));
  if (!h->amg) {
    k_set_stall<<<1, 1, 0, h->stream>>>(h->d_ctl, 2000);
    k_cg_init<T, KT><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->B, (const T*)h->d_dinv, (T*)h->X,
                                              (T*)h->R, (T*)h->P, h->d_ctl, h->d_partials, rtol, atol,
                                              imax);
    h->stats.kernel_launches++;
  } else {
    // x = 0, p = 0, r = b ; z = M^-1 r (V-cycle; its last kernel sets rho0, tolerances,
    // activity because ctl->init = 1) ; p = z + 0*p
    CK(h, cudaMemsetAsync(h->X, 0, nelem * sizeof(T), h->stream));
    CK(h, cudaMemsetAsync(h->P, 0, nelem * sizeof(T), h->stream));
    CK(h, cudaMemcpyAsync(h->R, h->B, nelem * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
    k_set_ctl<<<1, 1, 0, h->stream>>>(h->d_ctl, rtol, atol, imax, 40);
    if (h->mixed) {
      k_convert<T, float><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->R, (float*)h->R32);
      launch_vcycle<T, KT>(h, false);
      k_cg_update_xp2<T, KT, float><<<g, NT, 0, h->stream>>>(nelem, (const float*)h->Z32, (T*)h->X, (T*)h->P,
                                                             h->d_ctl);
      h->stats.kernel_launches++;
    } else {
      launch_vcycle<T, KT>(h, false);
      k_cg_update_xp2<T, KT, T><<<g, NT, 0, h->stream>>>(nelem, (const T*)h->Z, (T*)h->X, (T*)h->P, h->d_ctl);
    }
    h->stats.kernel_launches += 2;
  }
  CK(h, cudaGetLastError());
  const int chunk = h->amg ? std::min(h->opts.check_every, 4) : h->opts.check_every;
  const bool device_loop = h->opts.use_graph == 1 && !h->profile;
  if (device_loop) {
    int rc = run_loop<T, KT>(h);
    if (rc) return rc;
  }
  for (;;) {
    CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(PanelCtl), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->profile) harvest_profile(h);
    if (device_loop) {
      GraphSlot& gs = h->graphs[kt_index(KT)];
      h->stats.kernel_launches += 1 + gs.loop_kernels * h->h_ctl->iter;
      h->stats.spmm_launches += gs.loop_spmms * h->h_ctl->iter;
      break;
    }
    if (h->h_ctl->nactive == 0) break;
    int rc = run_chunk<T, KT>(h, chunk);
    if (rc) return rc;
  }
  // true residual  AP = B - A X  (core.jl:640, 648-651)
  launch_spmm<T, KT, 2>(h, (const T*)h->X, (T*)h->AP, (const T*)h->B);
  CK(h, cudaGetLastError());
  CK(h, cudaEventRecord(h->ev3, h->stream));
  CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(PanelCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (h->profile) harvest_profile(h);
  float ms = 0;
  CK(h, cudaEventElapsedTime(&ms, h->ev2, h->ev3));
  h->stats.kernel_ms += ms;
  return CS_B200_OK;
}

int gather_panel_status(cs_b200_handle* h, int kt, int64_t c0, int64_t* iters, double* relres,
                        int64_t itmax, bool* any_fail, bool* any_maxit, std::string* msg) {
  for (int c = 0; c < kt; ++c) {
    const PanelCtl& ct = *h->h_ctl;
    const double bn = ct.bnorm[c];
    const double rr = bn > 0 ? std::sqrt(ct.resid[c] / bn) : 0.0;
    if (iters) iters[c0 + c] = ct.iters[c];
    if (relres) relres[c0 + c] = rr;
    h->stats.iterations += ct.iters[c];
    if (!(rr < h->opts.resid_gate)) {
      if (!*any_fail) {
        char buf[256];
        snprintf(buf, sizeof buf,
                 "CUDA PCG solver residual %g exceeds tolerance %g for column %lld (%d iterations)",
                 rr, h->opts.resid_gate, (long long)(c0 + c + 1), ct.iters[c]);
        *msg = buf;
      }
      *any_fail = true;
    }
    // a column frozen by the stagnation guard above its tolerance is reported like one that ran into
    // itmax: results written, CS_B200_ERR_MAXITER, the true-residual gate decides (core.jl:639-641)
    if ((ct.iters[c] >= itmax || ct.stalled[c]) && std::sqrt(ct.rho[c]) > ct.tol[c]) *any_maxit = true;
  }
  return 0;
}

// node currents of the panel in X (src/out.jl:178-290): branch-current maxima, then max(inflow, outflow)
// per node with the 1e-8 zeroing, accumulated into the cumulative / max vectors (src/out.jl:100-107)
template <typename T, int KT>
void launch_currents(cs_b200_handle* h, bool want_curr, int accumulate) {
  const int grid = (int)std::min<int64_t>(h->grid_spmm, (h->n + (NT / KT) - 1) / (NT / KT));
  if (h->A0.dia) {
    const DiaDev<T> a{(const T*)h->A0.dia, h->A0.dia_ld, (int)h->n, h->A0.dia_nr};
    k_cur_max_dia<T, KT><<<grid, NT, 0, h->stream>>>(a, (const T*)h->X, h->d_ctl, h->d_partials);
    k_cur_acc_dia<T, KT><<<grid, NT, 0, h->stream>>>(a, (const T*)h->X, h->d_ctl, want_curr ? (T*)h->AP : nullptr,
                                                     (T*)h->d_cum, (T*)h->d_max, accumulate, h->opts.log_transform, KT);
  } else {
    k_cur_max<T, KT><<<grid, NT, 0, h->stream>>>((int)h->n, h->d_rowptr, h->d_colidx, (const T*)h->d_vals,
                                                 (const T*)h->X, h->d_ctl, h->d_partials);
    k_cur_acc<T, KT><<<grid, NT, 0, h->stream>>>((int)h->n, h->d_rowptr, h->d_colidx, (const T*)h->d_vals,
                                                 (const T*)h->X, h->d_ctl, want_curr ? (T*)h->AP : nullptr,
                                                 (T*)h->d_cum, (T*)h->d_max, accumulate, h->opts.log_transform, KT);
  }
  h->stats.kernel_launches += 2;
}

int next_kt(int64_t remaining, int ktmax) {
  int kt = ktmax;
  while (kt > remaining) kt >>= 1;
  return kt < 1 ? 1 : kt;
}

template <typename T, int KT>
int pairs_panel(cs_b200_handle* h, int64_t c0, const int64_t* src, const int64_t* dst,
                const double* weight, double rtol, int64_t itmax, T* R, T* volt, T* curr,
                int accumulate, int64_t* iters, double* relres, bool* any_fail, bool* any_maxit,
                std::string* msg) {
  const size_t nelem = (size_t)h->n_pad * KT;
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  for (int c = 0; c < KT; ++c) {
    hc->src[c] = src[c0 + c];
    hc->dst[c] = dst[c0 + c];
    hc->weight[c] = weight ? weight[c0 + c] : 1.0;
  }
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  h->stats.h2d_bytes += sizeof(PanelCtl);
  CK(h, cudaMemsetAsync(h->B, 0, nelem * sizeof(T), h->stream));
  k_pair_rhs<T, KT><<<1, 32, 0, h->stream>>>((T*)h->B, h->d_ctl);
  h->stats.kernel_launches++;
  int rc = solve_panel<T, KT>(h, rtol, itmax);
  if (rc) return rc;
  k_pair_extract<T, KT><<<1, 32, 0, h->stream>>>((const T*)h->X, h->d_ctl);
  h->stats.kernel_launches++;
  if (accumulate || curr) {
    launch_currents<T, KT>(h, curr != nullptr, accumulate);
  }
  CK(h, cudaGetLastError());
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  if (curr) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->AP,
                                                    (T*)h->stage, h->d_ctl, 0);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(curr + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  if (volt) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->X,
                                                    (T*)h->stage, h->d_ctl, 1);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(volt + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  // status gathered from the host copy taken inside solve_panel; xsrc/xdst need a re-read
  gather_panel_status(h, KT, c0, iters, relres, itmax, any_fail, any_maxit, msg);
  CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(PanelCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  h->stats.d2h_bytes += sizeof(PanelCtl);
  for (int c = 0; c < KT; ++c) R[c0 + c] = (T)(h->h_ctl->xdst[c] - h->h_ctl->xsrc[c]);
  return CS_B200_OK;
}

// panel of cs_b200_solve_sources: like pairs_panel, with the right-hand sides scattered from
// the caller's sparse columns and the shifted voltages of the probe rows as the small result
template <typename T, int KT>
int sources_panel(cs_b200_handle* h, int64_t c0, const int64_t* colptr, const int64_t* rows,
                  const double* vals, const int64_t* ref, const double* weight, double rtol,
                  int64_t itmax, int64_t nprobe, T* probe_volt, T* volt, T* curr, int accumulate,
                  int64_t* iters, double* relres, bool* any_fail, bool* any_maxit, std::string* msg) {
  const size_t nelem = (size_t)h->n_pad * KT;
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  int ent_ptr[MAXKT + 1];
  const int64_t e0 = colptr[c0];
  for (int c = 0; c < KT; ++c) {
    hc->src[c] = ref[c0 + c];
    hc->dst[c] = -1;
    hc->weight[c] = weight ? weight[c0 + c] : 1.0;
    ent_ptr[c] = (int)(colptr[c0 + c] - e0);
  }
  ent_ptr[KT] = (int)(colptr[c0 + KT] - e0);
  const size_t nent = (size_t)ent_ptr[KT];
  if (nent > h->sp_cap) {
    cudaFree(h->d_sp_rows); cudaFree(h->d_sp_vals);
    h->d_sp_rows = nullptr; h->d_sp_vals = nullptr;
    h->sp_cap = std::max<size_t>(nent, 1024);
    CK(h, cudaMalloc(&h->d_sp_rows, h->sp_cap * sizeof(long long)));
    CK(h, cudaMalloc(&h->d_sp_vals, h->sp_cap * sizeof(double)));
  }
  if (!h->d_sp_ptr) CK(h, cudaMalloc(&h->d_sp_ptr, (MAXKT + 1) * sizeof(int)));
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  CK(h, h2d(h, h->d_sp_ptr, ent_ptr, (KT + 1) * sizeof(int)));
  if (nent) {
    CK(h, h2d(h, h->d_sp_rows, rows + e0, nent * sizeof(long long)));
    CK(h, h2d(h, h->d_sp_vals, vals + e0, nent * sizeof(double)));
  }
  h->stats.h2d_bytes += sizeof(PanelCtl) + nent * 16.0;
  CK(h, cudaMemsetAsync(h->B, 0, nelem * sizeof(T), h->stream));
  k_sparse_rhs<T, KT><<<1, 32, 0, h->stream>>>((T*)h->B, h->d_sp_ptr, h->d_sp_rows, h->d_sp_vals);
  h->stats.kernel_launches++;
  int rc = solve_panel<T, KT>(h, rtol, itmax);
  if (rc) return rc;
  gather_panel_status(h, KT, c0, iters, relres, itmax, any_fail, any_maxit, msg);
  k_pair_extract<T, KT><<<1, 32, 0, h->stream>>>((const T*)h->X, h->d_ctl);
  h->stats.kernel_launches++;
  if (nprobe > 0 && probe_volt) {
    k_probe<T, KT><<<(int)std::min<int64_t>(64, (nprobe * KT + 255) / 256), 256, 0, h->stream>>>(
        (const T*)h->X, h->d_ctl, h->d_probe, (int)nprobe, (T*)h->d_probe_out);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(probe_volt + (size_t)c0 * nprobe, h->d_probe_out, (size_t)nprobe * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)nprobe * KT * sizeof(T);
  }
  if (accumulate || curr) {
    launch_currents<T, KT>(h, curr != nullptr, accumulate);
  }
  CK(h, cudaGetLastError());
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  if (curr) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->AP,
                                                    (T*)h->stage, h->d_ctl, 0);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(curr + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  if (volt) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->X,
                                                    (T*)h->stage, h->d_ctl, 1);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(volt + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  CK(h, cudaStreamSynchronize(h->stream));
  return CS_B200_OK;
}

template <typename T>
int solve_sources_t(cs_b200_handle* h, int64_t k, const int64_t* colptr, const int64_t* rows,
                    const double* vals, const int64_t* ref, const double* weight, double rtol,
                    int64_t itmax, int64_t nprobe, const int64_t* probe, T* probe_volt, T* volt,
                    T* curr, int accumulate, int64_t* iters, double* relres);

// ---- superposition driver (cs_b200_solve_pairs_superposed) ----------------------------------
// panel of point solves  A u_x = e_{nodes[x]} - e_{nodes[0]}  for x = x0 .. x0+KT-1 (1-based among
// the focal nodes); the shifted solutions land in columns x0-1 .. of U (column-major, ld = n_pad)
template <typename T, int KT>
int point_panel(cs_b200_handle* h, int64_t x0, const int64_t* nodes, double rtol, int64_t itmax, T* U,
                int64_t* point_iters, bool* any_fail, bool* any_maxit, std::string* msg) {
  const size_t nelem = (size_t)h->n_pad * KT;
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  for (int c = 0; c < KT; ++c) {
    hc->src[c] = nodes[0];
    hc->dst[c] = nodes[x0 + c];
    hc->weight[c] = 1.0;
  }
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  h->stats.h2d_bytes += sizeof(PanelCtl);
  CK(h, cudaMemsetAsync(h->B, 0, nelem * sizeof(T), h->stream));
  k_pair_rhs<T, KT><<<1, 32, 0, h->stream>>>((T*)h->B, h->d_ctl);
  h->stats.kernel_launches++;
  int rc = solve_panel<T, KT>(h, rtol, itmax);
  if (rc) return rc;
  gather_panel_status(h, KT, 0, nullptr, nullptr, itmax, any_fail, any_maxit, msg);
  if (point_iters)
    for (int c = 0; c < KT; ++c) point_iters[x0 - 1 + c] = h->h_ctl->iters[c];
  k_pair_extract<T, KT><<<1, 32, 0, h->stream>>>((const T*)h->X, h->d_ctl);
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n_pad, (const T*)h->X,
                                                  U + (size_t)(x0 - 1) * h->n_pad, h->d_ctl, 1);
  h->stats.kernel_launches += 2;
  CK(h, cudaGetLastError());
  CK(h, cudaStreamSynchronize(h->stream));
  return CS_B200_OK;
}

// panel of pairs c0 .. c0+KT-1 formed from U; same outputs as pairs_panel
template <typename T, int KT>
int combine_panel(cs_b200_handle* h, int64_t c0, const int64_t* nodes, const int64_t* pi, const int64_t* pj,
                  const double* weight, const T* U, int* d_ci, int* d_cj, T* R, T* volt, T* curr,
                  int accumulate, double* relres, int64_t itmax, bool* any_fail, bool* any_maxit,
                  std::string* msg) {
  const size_t nelem = (size_t)h->n_pad * KT;
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  int ci[MAXKT], cj[MAXKT];
  for (int c = 0; c < KT; ++c) {
    hc->src[c] = nodes[pi[c0 + c]];
    hc->dst[c] = nodes[pj[c0 + c]];
    hc->weight[c] = weight ? weight[c0 + c] : 1.0;
    ci[c] = (int)pi[c0 + c] - 1;      // point 0 is the reference: its solution is identically 0
    cj[c] = (int)pj[c0 + c] - 1;
  }
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  CK(h, h2d(h, d_ci, ci, KT * sizeof(int)));
  CK(h, h2d(h, d_cj, cj, KT * sizeof(int)));
  h->stats.h2d_bytes += sizeof(PanelCtl) + 2.0 * KT * sizeof(int);
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  k_combine<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n_pad, U, d_ci, d_cj, (T*)h->X);
  CK(h, cudaMemsetAsync(h->B, 0, nelem * sizeof(T), h->stream));
  k_pair_rhs<T, KT><<<1, 32, 0, h->stream>>>((T*)h->B, h->d_ctl);
  // the reference's gate on the combined voltage: AP = B - A X, ||AP|| / ||B||  (core.jl:640-641)
  launch_spmm<T, KT, SP_RESNORM>(h, (const T*)h->X, (T*)h->AP, (const T*)h->B);
  h->stats.kernel_launches += 2;
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(PanelCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  gather_panel_status(h, KT, c0, nullptr, relres, itmax, any_fail, any_maxit, msg);
  k_pair_extract<T, KT><<<1, 32, 0, h->stream>>>((const T*)h->X, h->d_ctl);
  h->stats.kernel_launches++;
  if (accumulate || curr) {
    launch_currents<T, KT>(h, curr != nullptr, accumulate);
  }
  CK(h, cudaGetLastError());
  if (curr) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->AP,
                                                    (T*)h->stage, h->d_ctl, 0);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(curr + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  if (volt) {
    k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->X,
                                                    (T*)h->stage, h->d_ctl, 1);
    h->stats.kernel_launches++;
    CK(h, cudaMemcpyAsync(volt + (size_t)c0 * h->n, h->stage, (size_t)h->n * KT * sizeof(T),
                          cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  }
  CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(PanelCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  h->stats.d2h_bytes += sizeof(PanelCtl);
  for (int c = 0; c < KT; ++c) R[c0 + c] = (T)(h->h_ctl->xdst[c] - h->h_ctl->xsrc[c]);
  return CS_B200_OK;
}

template <typename T>
int solve_pairs_superposed_t(cs_b200_handle* h, int64_t np, const int64_t* nodes, int64_t k,
                             const int64_t* pi, const int64_t* pj, const double* weight, double rtol,
                             int64_t itmax, T* R, T* volt, T* curr, int accumulate,
                             int64_t* point_iters, double* relres);

int ensure_io_pipeline(cs_b200_handle* h) {
  if (h->s_in) return CS_B200_OK;
  CK(h, cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
  CK(h, cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
  const size_t bytes = (size_t)h->n * h->ktmax * h->esize();
  for (int i = 0; i < 2; ++i) {
    CK(h, cudaMalloc(&h->io_in[i], bytes));
    CK(h, cudaMalloc(&h->io_out[i], bytes));
    CK(h, cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
    CK(h, cudaEventCreateWithFlags(&h->ev_used[i], cudaEventDisableTiming));
    CK(h, cudaEventCreateWithFlags(&h->ev_ready[i], cudaEventDisableTiming));
    CK(h, cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
  }
  return CS_B200_OK;
}

// upload of panel `ip` (columns c0 .. c0+kt) into its staging slot, on the upload stream;
// waits until the panel that used the slot two panels ago has been transposed out of it
template <typename T>
int rhs_upload(cs_b200_handle* h, int ip, int64_t c0, int kt, const T* rhs) {
  const int s = ip & 1;
  if (ip >= 2) CK(h, cudaStreamWaitEvent(h->s_in, h->ev_used[s], 0));
  CK(h, cudaMemcpyAsync(h->io_in[s], rhs + (size_t)c0 * h->n, (size_t)h->n * kt * sizeof(T),
                        cudaMemcpyHostToDevice, h->s_in));
  CK(h, cudaEventRecord(h->ev_in[s], h->s_in));
  h->stats.h2d_bytes += (double)h->n * kt * sizeof(T);
  return CS_B200_OK;
}

template <typename T, int KT>
int rhs_panel(cs_b200_handle* h, int ip, int64_t c0, T* lhs, double rtol, int64_t itmax,
              int64_t* iters, double* relres, bool* any_fail, bool* any_maxit, std::string* msg) {
  const size_t nelem = (size_t)h->n_pad * KT;
  const int s = ip & 1;
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  for (int c = 0; c < KT; ++c) hc->src[c] = hc->dst[c] = -1;
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemsetAsync(h->B, 0, nelem * sizeof(T), h->stream));
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  CK(h, cudaStreamWaitEvent(h->stream, h->ev_in[s], 0));
  k_cm_to_panel<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->io_in[s],
                                                  (T*)h->B, KT);
  CK(h, cudaEventRecord(h->ev_used[s], h->stream));
  h->stats.kernel_launches++;
  int rc = solve_panel<T, KT>(h, rtol, itmax);
  if (rc) return rc;
  gather_panel_status(h, KT, c0, iters, relres, itmax, any_fail, any_maxit, msg);
  if (ip >= 2) CK(h, cudaStreamWaitEvent(h->stream, h->ev_out[s], 0));   // slot's last download done
  k_panel_to_cm<T, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const T*)h->X,
                                                  (T*)h->io_out[s], h->d_ctl, 0);
  h->stats.kernel_launches++;
  CK(h, cudaEventRecord(h->ev_ready[s], h->stream));
  CK(h, cudaStreamWaitEvent(h->s_out, h->ev_ready[s], 0));
  CK(h, cudaMemcpyAsync(lhs + (size_t)c0 * h->n, h->io_out[s], (size_t)h->n * KT * sizeof(T),
                        cudaMemcpyDeviceToHost, h->s_out));
  CK(h, cudaEventRecord(h->ev_out[s], h->s_out));
  h->stats.d2h_bytes += (double)h->n * KT * sizeof(T);
  return CS_B200_OK;
}

#define DISPATCH_KT(kt, CALL)                    \
  switch (kt) {                                  \
    case 1: { constexpr int KT = 1; CALL; } break; \
    case 2: { constexpr int KT = 2; CALL; } break; \
    case 4: { constexpr int KT = 4; CALL; } break; \
    default: { constexpr int KT = 8; CALL; } break; \
  }

template <typename T>
int solve_pairs_t(cs_b200_handle* h, int64_t k, const int64_t* src, const int64_t* dst,
                  const double* weight, double rtol, int64_t itmax, T* R, T* volt, T* curr,
                  int accumulate, int64_t* iters, double* relres) {
  bool any_fail = false, any_maxit = false;
  std::string msg;
  int64_t c0 = 0;
  while (c0 < k) {
    const int kt = next_kt(k - c0, h->ktmax);
    int rc = 0;
    DISPATCH_KT(kt, (rc = pairs_panel<T, KT>(h, c0, src, dst, weight, rtol, itmax, R, volt, curr,
                                             accumulate, iters, relres, &any_fail, &any_maxit,
                                             &msg)));
    if (rc) return rc;
    c0 += kt;
  }
  if (any_fail) return set_err(h, CS_B200_ERR_RESIDUAL, "%s", msg.c_str());
  if (any_maxit) return set_err(h, CS_B200_ERR_MAXITER, "itmax reached (or the recurrence stagnated) before rtol");
  return CS_B200_OK;
}

template <typename T>
int solve_sources_t(cs_b200_handle* h, int64_t k, const int64_t* colptr, const int64_t* rows,
                    const double* vals, const int64_t* ref, const double* weight, double rtol,
                    int64_t itmax, int64_t nprobe, const int64_t* probe, T* probe_volt, T* volt,
                    T* curr, int accumulate, int64_t* iters, double* relres) {
  bool any_fail = false, any_maxit = false;
  std::string msg;
  if (nprobe > 0 && probe_volt) {
    const size_t need = (size_t)nprobe;
    if (need > h->probe_cap) {
      cudaFree(h->d_probe); cudaFree(h->d_probe_out);
      h->d_probe = nullptr; h->d_probe_out = nullptr;
      h->probe_cap = need;
      CK(h, cudaMalloc(&h->d_probe, need * sizeof(long long)));
      CK(h, cudaMalloc(&h->d_probe_out, need * MAXKT * sizeof(double)));
    }
    CK(h, h2d(h, h->d_probe, probe, need * sizeof(long long)));
  }
  int64_t c0 = 0;
  while (c0 < k) {
    const int kt = next_kt(k - c0, h->ktmax);
    int rc = 0;
    DISPATCH_KT(kt, (rc = sources_panel<T, KT>(h, c0, colptr, rows, vals, ref, weight, rtol, itmax,
                                               nprobe, probe_volt, volt, curr, accumulate, iters,
                                               relres, &any_fail, &any_maxit, &msg)));
    if (rc) return rc;
    c0 += kt;
  }
  if (any_fail) return set_err(h, CS_B200_ERR_RESIDUAL, "%s", msg.c_str());
  if (any_maxit) return set_err(h, CS_B200_ERR_MAXITER, "itmax reached (or the recurrence stagnated) before rtol");
  return CS_B200_OK;
}

template <typename T>
int solve_pairs_superposed_t(cs_b200_handle* h, int64_t np, const int64_t* nodes, int64_t k,
                             const int64_t* pi, const int64_t* pj, const double* weight, double rtol,
                             int64_t itmax, T* R, T* volt, T* curr, int accumulate,
                             int64_t* point_iters, double* relres) {
  bool any_fail = false, any_maxit = false;
  std::string msg;
  T* U = nullptr;
  int *d_ci = nullptr, *d_cj = nullptr;
  const size_t ubytes = (size_t)h->n_pad * (size_t)(np - 1) * sizeof(T);
  auto cleanup = [&]() { cudaFree(U); cudaFree(d_ci); cudaFree(d_cj); };
  cudaError_t e = cudaMalloc(&U, ubytes);
  if (e == cudaSuccess) e = cudaMalloc(&d_ci, MAXKT * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&d_cj, MAXKT * sizeof(int));
  if (e == cudaSuccess) e = cudaMemsetAsync(U, 0, ubytes, h->stream);
  if (e != cudaSuccess) {
    cleanup();
    return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s allocating %zu bytes for the point solutions",
                   cudaGetErrorString(e), ubytes);
  }
  int rc = 0;
  int64_t x0 = 1;
  while (!rc && x0 < np) {
    const int kt = next_kt(np - x0, h->ktmax);
    DISPATCH_KT(kt, (rc = point_panel<T, KT>(h, x0, nodes, rtol, itmax, U, point_iters, &any_fail,
                                             &any_maxit, &msg)));
    x0 += kt;
  }
  int64_t c0 = 0;
  while (!rc && c0 < k) {
    const int kt = next_kt(k - c0, h->ktmax);
    DISPATCH_KT(kt, (rc = combine_panel<T, KT>(h, c0, nodes, pi, pj, weight, U, d_ci, d_cj, R, volt, curr,
                                               accumulate, relres, itmax, &any_fail, &any_maxit, &msg)));
    c0 += kt;
  }
  cudaStreamSynchronize(h->stream);
  cleanup();
  if (rc) return rc;
  if (any_fail) return set_err(h, CS_B200_ERR_RESIDUAL, "%s", msg.c_str());
  if (any_maxit) return set_err(h, CS_B200_ERR_MAXITER, "itmax reached (or the recurrence stagnated) before rtol");
  return CS_B200_OK;
}

template <typename T>
int solve_rhs_t(cs_b200_handle* h, int64_t k, const T* rhs, T* lhs, double rtol, int64_t itmax,
                int64_t* iters, double* relres) {
  bool any_fail = false, any_maxit = false;
  std::string msg;
  int rc = ensure_io_pipeline(h);
  if (rc) return rc;
  // the upload stream must not overtake work of an earlier call that still reads the slots
  CK(h, cudaEventRecord(h->ev_used[0], h->stream));
  CK(h, cudaStreamWaitEvent(h->s_in, h->ev_used[0], 0));
  int64_t c0 = 0;
  int ip = 0;
  rc = rhs_upload<T>(h, 0, 0, next_kt(k, h->ktmax), rhs);
  while (!rc && c0 < k) {
    const int kt = next_kt(k - c0, h->ktmax);
    const int64_t c1 = c0 + kt;
    if (c1 < k) {   // next panel's upload overlaps this panel's solve
      rc = rhs_upload<T>(h, ip + 1, c1, next_kt(k - c1, h->ktmax), rhs);
      if (rc) break;
    }
    DISPATCH_KT(kt, (rc = rhs_panel<T, KT>(h, ip, c0, lhs, rtol, itmax, iters, relres, &any_fail,
                                           &any_maxit, &msg)));
    c0 = c1;
    ++ip;
  }
  // drain both copy streams whatever happened: the caller owns rhs/lhs again on return
  cudaStreamSynchronize(h->s_in);
  cudaStreamSynchronize(h->s_out);
  cudaStreamSynchronize(h->stream);
  if (rc) return rc;
  if (any_fail) return set_err(h, CS_B200_ERR_RESIDUAL, "%s", msg.c_str());
  if (any_maxit) return set_err(h, CS_B200_ERR_MAXITER, "itmax reached (or the recurrence stagnated) before rtol");
  return CS_B200_OK;
}

void begin_call(cs_b200_handle* h) {
  cudaSetDevice(h->device);
  h->err.clear();
  const double setup = h->stats.setup_ms;
  h->stats = cs_b200_stats{};
  h->stats.setup_ms = setup;
  cudaEventRecord(h->ev0, h->stream);
}
void end_call(cs_b200_handle* h) {
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.solve_ms = ms;
}

int ensure_flush(cs_b200_handle* h) {
  if (h->d_flush) return 0;
  h->flush_elems = (size_t)64 << 20;  // 256 MB of floats > 126 MB L2
  CK(h, cudaMalloc(&h->d_flush, h->flush_elems * sizeof(float)));
  CK(h, cudaMemsetAsync(h->d_flush, 0, h->flush_elems * sizeof(float), h->stream));
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
namespace {
template <typename T>
int assemble_raster(cs_b200_handle* h, int64_t nrows, int64_t ncols, const T* g_host,
                           int four, int avg_res, std::vector<int>& rp_host) {
  const int64_t ncell = nrows * ncols;
  T* d_g = nullptr;
  int *d_valid = nullptr, *d_nodeid = nullptr, *d_rowcnt = nullptr;
  auto cleanup = [&]() { cudaFree(d_g); cudaFree(d_valid); cudaFree(d_nodeid); cudaFree(d_rowcnt); };
#define CKR(call)                                                                          \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      cleanup();                                                                           \
      return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s at %s:%d (%s)",                   \
                     cudaGetErrorString(_e), __FILE__, __LINE__, #call);                   \
    }                                                                                      \
  } while (0)
  CKR(cudaMalloc(&d_g, (size_t)ncell * sizeof(T)));
  CKR(cudaMalloc(&d_valid, (size_t)ncell * sizeof(int)));
  CKR(cudaMalloc(&d_nodeid, (size_t)ncell * sizeof(int)));
  CKR(h2d(h, d_g, g_host, (size_t)ncell * sizeof(T)));
  const int grid = (int)std::min<int64_t>((ncell + 255) / 256, (int64_t)h->num_sms * 32);
  ras::k_valid<T><<<grid, 256, 0, h->stream>>>(ncell, d_g, d_valid);
  CKR(cudaGetLastError());
  CKR(ras::exclusive_scan(d_valid, d_nodeid, ncell, h->stream));
  int last_id = 0, last_valid = 0;
  CKR(cudaMemcpy(&last_id, d_nodeid + (ncell - 1), sizeof(int), cudaMemcpyDeviceToHost));
  CKR(cudaMemcpy(&last_valid, d_valid + (ncell - 1), sizeof(int), cudaMemcpyDeviceToHost));
  const int64_t n = (int64_t)last_id + last_valid;
  if (n <= 0) { cleanup(); return set_err(h, CS_B200_ERR_ARG, "raster has no cell with conductance > 0"); }
  CKR(cudaMalloc(&d_rowcnt, (size_t)(n + 1) * sizeof(int)));
  CKR(cudaMemsetAsync(d_rowcnt, 0, (size_t)(n + 1) * sizeof(int), h->stream));
  ras::k_count<<<grid, 256, 0, h->stream>>>((int)nrows, (int)ncols, four, d_valid, d_nodeid, d_rowcnt);
  CKR(cudaGetLastError());
  CKR(cudaMalloc(&h->d_rowptr, (size_t)(n + 1) * sizeof(int)));
  CKR(ras::exclusive_scan(d_rowcnt, h->d_rowptr, n + 1, h->stream));
  rp_host.resize((size_t)n + 1);
  CKR(cudaMemcpy(rp_host.data(), h->d_rowptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost));
  const int64_t nnz = rp_host[(size_t)n];
  if (nnz <= 0) { cleanup(); return set_err(h, CS_B200_ERR_ARG, "assembled matrix is empty"); }
  CKR(cudaMalloc(&h->d_colidx, (size_t)nnz * sizeof(int)));
  CKR(cudaMalloc(&h->d_vals, (size_t)nnz * sizeof(T)));
  ras::k_fill<T><<<grid, 256, 0, h->stream>>>((int)nrows, (int)ncols, four, avg_res, d_g, d_valid, d_nodeid,
                                              h->d_rowptr, h->d_colidx, (T*)h->d_vals);
  CKR(cudaGetLastError());
  CKR(cudaStreamSynchronize(h->stream));
#undef CKR
  cleanup();
  h->n = n;
  h->nnz = nnz;
  h->n_pad = (n + 3) / 4 * 4;
  return CS_B200_OK;
}

}  // namespace

namespace {
template <typename T>
__global__ void k_apply_grounds(int n, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                T* __restrict__ vals, const T* __restrict__ g, const unsigned char* __restrict__ mask) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const bool mi = mask && mask[i];
    for (int j = rowptr[i]; j < rowptr[i + 1]; ++j) {
      const int c = colidx[j];
      if (mi) vals[j] = c == i ? T(1) : T(0);
      else if (mask && mask[c]) vals[j] = T(0);
      else if (c == i && g) vals[j] += g[i];
    }
  }
}
}  // namespace

// everything derived from the operator's VALUES: captured graphs (they hold level pointers), the
// finest operator's stencil / window records, the multigrid levels.  The CSR, the plain row blocks
// and the panels stay.
static void teardown_operators(cs_b200_handle* h) {
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto& g : h->graphs) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.loop_exec) cudaGraphExecDestroy(g.loop_exec);
    g = GraphSlot{};
  }
  free_win(h->A0);
  h->A0.has_dinv = 0; h->A0.win_blocks = 0; h->A0.win_nblocks = 0; h->A0.dia_nr = 0; h->A0.dia_ld = 0;
  for (size_t l = 0; l < h->lv.size(); ++l) {
    DevLevel& L = h->lv[l];
    if (l > 0) {
      free_csr(L.A);
      cudaFree(L.dinv); cudaFree(L.x); cudaFree(L.b); cudaFree(L.t); cudaFree(L.y);
    }
    free_csr(L.P);
    free_csr(L.R);
  }
  for (size_t l = 0; l < h->lv32.size(); ++l) {
    DevLevel& L = h->lv32[l];
    free_csr(L.A);
    cudaFree(L.dinv); cudaFree(L.x); cudaFree(L.b); cudaFree(L.t); cudaFree(L.y);
    free_csr(L.P);
    free_csr(L.R);
  }
  h->lv.clear();
  h->lv32.clear();
  cudaFree(h->R32); cudaFree(h->X32); cudaFree(h->T32); cudaFree(h->Z32);
  h->R32 = h->X32 = h->T32 = h->Z32 = nullptr;
  cudaFree(h->Z); h->Z = nullptr;
  cudaFree(h->d_pinv); h->d_pinv = nullptr;
  h->amg = false;
  h->mixed = false;
}


extern "C" {

int cs_b200_version(void) { return 1002; }

const char* cs_b200_last_error(const cs_b200_handle* h) {
  return h ? h->err.c_str() : g_create_error.c_str();
}

int cs_b200_create(int64_t n, int64_t nnz, const void* rowptr, const void* colidx,
                   const void* vals, int index_bits, int index_base, int dtype, int device,
                   const cs_b200_opts* opts, cs_b200_handle** out) {
  if (!out) return set_err(nullptr, CS_B200_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (n <= 0 || nnz < 0 || !rowptr || (nnz > 0 && (!colidx || !vals)))
    return set_err(nullptr, CS_B200_ERR_ARG, "bad matrix arguments (n=%lld nnz=%lld)",
                   (long long)n, (long long)nnz);
  if ((index_bits != 32 && index_bits != 64) || (index_base != 0 && index_base != 1) ||
      (dtype != CS_B200_F32 && dtype != CS_B200_F64))
    return set_err(nullptr, CS_B200_ERR_ARG, "bad index_bits/index_base/dtype");
  if (nnz >= (int64_t)1 << 31 || n >= (int64_t)1 << 31)
    return set_err(nullptr, CS_B200_ERR_UNSUPPORTED,
                   "n and nnz must be < 2^31 (device indices are int32)");
  cs_b200_handle* h = new cs_b200_handle();
  h->n = n; h->nnz = nnz; h->dtype = dtype; h->device = device;
  int rc = common_create(h, opts);
  if (rc) { g_create_error = h->err; cs_b200_destroy(h); return rc; }
  auto fail = [&](int code) { g_create_error = h->err; cs_b200_destroy(h); return code; };
  cudaEventRecord(h->ev0, h->stream);
  const size_t es = h->esize();
#define CKC(call)                                                                              \
  do {                                                                                         \
    cudaError_t _e = (call);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (%s)", cudaGetErrorString(_e), #call);       \
      return fail(CS_B200_ERR_CUDA);                                                           \
    }                                                                                          \
  } while (0)
  if (h->opts.setup != 1) {
    // ---- device-side setup: raw index arrays go up as they are and are narrowed on the GPU; the
    // ordered aggregation seed pass starts right away on a helper thread (it only reads the
    // caller's arrays) and overlaps the upload
    const int64_t first = index_bits == 64 ? ((const int64_t*)rowptr)[0] : (int64_t)((const int32_t*)rowptr)[0];
    const int64_t last = index_bits == 64 ? ((const int64_t*)rowptr)[n] : (int64_t)((const int32_t*)rowptr)[n];
    if (first - index_base != 0 || last - index_base != nnz) {
      set_err(h, CS_B200_ERR_ARG, "rowptr does not span [0, nnz] (got %lld..%lld)", (long long)(first - index_base),
              (long long)(last - index_base));
      return fail(CS_B200_ERR_ARG);
    }
    const csb_dev::HostPattern hp{rowptr, colidx, index_bits, index_base};
    csb_dev::SeedJob* job = nullptr;
    Tick up_tick;
    if (h->opts.precond == CS_B200_PRECOND_AMG && n > 200) job = csb_dev::seed_start(n, hp);
    auto fail_job = [&](int code) { csb_dev::seed_discard(job); job = nullptr; return fail(code); };
#define CKJ(call)                                                                              \
  do {                                                                                         \
    cudaError_t _e = (call);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (%s)", cudaGetErrorString(_e), #call);       \
      return fail_job(CS_B200_ERR_CUDA);                                                       \
    }                                                                                          \
  } while (0)
    CKJ(cudaMalloc(&h->d_rowptr, (size_t)(n + 1) * sizeof(int)));
    CKJ(cudaMalloc(&h->d_colidx, std::max<size_t>(1, (size_t)nnz) * sizeof(int)));
    CKJ(cudaMalloc(&h->d_vals, std::max<size_t>(1, (size_t)nnz) * es));
    if (index_bits == 32 && index_base == 0) {
      CKJ(cudaMemcpyAsync(h->d_rowptr, rowptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
      CKJ(cudaMemcpyAsync(h->d_colidx, colidx, (size_t)nnz * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    } else {
      const size_t ib = index_bits / 8;
      void* raw = nullptr;
      CKJ(cudaMalloc(&raw, std::max<size_t>((size_t)(n + 1), (size_t)nnz) * ib));
      cudaError_t e = cudaMemcpyAsync(raw, rowptr, (size_t)(n + 1) * ib, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = (cudaError_t)csb_dev::narrow_indices(h->stream, raw, index_bits, index_base, n + 1, h->d_rowptr);
      if (e == cudaSuccess) e = cudaMemcpyAsync(raw, colidx, (size_t)nnz * ib, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = (cudaError_t)csb_dev::narrow_indices(h->stream, raw, index_bits, index_base, nnz, h->d_colidx);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      cudaFree(raw);
      CKJ(e);
    }
    CKJ(cudaMemcpyAsync(h->d_vals, vals, (size_t)nnz * es, cudaMemcpyHostToDevice, h->stream));
#undef CKJ
    if (up_tick.on) { cudaStreamSynchronize(h->stream); up_tick("upload (narrowed on device)"); }
    rc = dtype == CS_B200_F64 ? finish_setup_device<double>(h, hp, job) : finish_setup_device<float>(h, hp, job);
    if (rc) return fail(rc);
  } else {
  std::vector<int> rp, ci;
  if (index_bits == 64) {
    narrow_indices((const int64_t*)rowptr, n + 1, index_base, rp);
    narrow_indices((const int64_t*)colidx, nnz, index_base, ci);
  } else {
    narrow_indices((const int32_t*)rowptr, n + 1, index_base, rp);
    narrow_indices((const int32_t*)colidx, nnz, index_base, ci);
  }
  if (rp[0] != 0 || rp[n] != nnz) {
    set_err(h, CS_B200_ERR_ARG, "rowptr does not span [0, nnz] (got %d..%d)", rp[0], rp[n]);
    return fail(CS_B200_ERR_ARG);
  }
  CKC(cudaMalloc(&h->d_rowptr, (size_t)(n + 1) * sizeof(int)));
  CKC(cudaMalloc(&h->d_colidx, std::max<size_t>(1, (size_t)nnz) * sizeof(int)));
  CKC(cudaMalloc(&h->d_vals, std::max<size_t>(1, (size_t)nnz) * es));
  CKC(cudaMemcpyAsync(h->d_rowptr, rp.data(), (size_t)(n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CKC(cudaMemcpyAsync(h->d_colidx, ci.data(), (size_t)nnz * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CKC(cudaMemcpyAsync(h->d_vals, vals, (size_t)nnz * es, cudaMemcpyHostToDevice, h->stream));
  rc = dtype == CS_B200_F64 ? finish_setup<double>(h, rp, &ci, (const double*)vals)
                            : finish_setup<float>(h, rp, &ci, (const float*)vals);
  if (rc) return fail(rc);
  }
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  *out = h;
  return CS_B200_OK;
}

int cs_b200_create_from_device(int64_t n, int64_t nnz, const int32_t* d_rowptr,
                               const int32_t* d_colidx, const void* d_vals, int dtype, int device,
                               const cs_b200_opts* opts, cs_b200_handle** out) {
  if (!out) return set_err(nullptr, CS_B200_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (n <= 0 || nnz <= 0 || !d_rowptr || !d_colidx || !d_vals ||
      (dtype != CS_B200_F32 && dtype != CS_B200_F64) || nnz >= (int64_t)1 << 31)
    return set_err(nullptr, CS_B200_ERR_ARG, "bad arguments");
  cs_b200_handle* h = new cs_b200_handle();
  h->n = n; h->nnz = nnz; h->dtype = dtype; h->device = device;
  h->owns_matrix = false;
  int rc = common_create(h, opts);
  if (rc) { g_create_error = h->err; cs_b200_destroy(h); return rc; }
  cudaEventRecord(h->ev0, h->stream);
  h->d_rowptr = const_cast<int*>(d_rowptr);
  h->d_colidx = const_cast<int*>(d_colidx);
  h->d_vals = const_cast<void*>(d_vals);
  if (h->opts.setup != 1) {
    const csb_dev::HostPattern hp{};
    rc = dtype == CS_B200_F64 ? finish_setup_device<double>(h, hp, nullptr) : finish_setup_device<float>(h, hp, nullptr);
  } else {
    std::vector<int> rp(n + 1);
    cudaError_t e = cudaMemcpy(rp.data(), d_rowptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      set_err(h, CS_B200_ERR_CUDA, "CUDA error %s reading rowptr", cudaGetErrorString(e));
      g_create_error = h->err; cs_b200_destroy(h); return CS_B200_ERR_CUDA;
    }
    rc = dtype == CS_B200_F64 ? finish_setup<double>(h, rp, nullptr, (const double*)nullptr)
                              : finish_setup<float>(h, rp, nullptr, (const float*)nullptr);
  }
  if (rc) { g_create_error = h->err; cs_b200_destroy(h); return rc; }
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  *out = h;
  return CS_B200_OK;
}

int cs_b200_create_from_raster(int64_t nrows, int64_t ncols, const void* g, int dtype,
                               int four_neighbors, int avg_res, int device,
                               const cs_b200_opts* opts, cs_b200_handle** out,
                               int64_t* n_out, int64_t* nnz_out) {
  if (!out) return set_err(nullptr, CS_B200_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (nrows <= 0 || ncols <= 0 || !g || (dtype != CS_B200_F32 && dtype != CS_B200_F64) ||
      nrows > (int64_t)1 << 30 || ncols > (int64_t)1 << 30)
    return set_err(nullptr, CS_B200_ERR_ARG, "bad arguments");
  if (nrows * ncols * 9 >= (int64_t)1 << 31)
    return set_err(nullptr, CS_B200_ERR_UNSUPPORTED, "raster too large: 9 * cells must be < 2^31 (device indices are int32)");
  cs_b200_handle* h = new cs_b200_handle();
  h->n = 0; h->nnz = 0; h->dtype = dtype; h->device = device;
  h->owns_matrix = true;
  int rc = common_create(h, opts);
  if (rc) { g_create_error = h->err; cs_b200_destroy(h); return rc; }
  cudaEventRecord(h->ev0, h->stream);
  std::vector<int> rp;
  rc = dtype == CS_B200_F64
           ? assemble_raster<double>(h, nrows, ncols, (const double*)g, four_neighbors ? 1 : 0, avg_res ? 1 : 0, rp)
           : assemble_raster<float>(h, nrows, ncols, (const float*)g, four_neighbors ? 1 : 0, avg_res ? 1 : 0, rp);
  if (!rc) {
    if (h->opts.setup != 1) {
      const csb_dev::HostPattern hp{};
      rc = dtype == CS_B200_F64 ? finish_setup_device<double>(h, hp, nullptr) : finish_setup_device<float>(h, hp, nullptr);
    } else {
      rc = dtype == CS_B200_F64 ? finish_setup<double>(h, rp, nullptr, (const double*)nullptr)
                                : finish_setup<float>(h, rp, nullptr, (const float*)nullptr);
    }
  }
  if (rc) { g_create_error = h->err; cs_b200_destroy(h); return rc; }
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  if (n_out) *n_out = h->n;
  if (nnz_out) *nnz_out = h->nnz;
  *out = h;
  return CS_B200_OK;
}

int cs_b200_create_from_raster_poly(int64_t nrows, int64_t ncols, const void* g, const int32_t* polymap,
                                    int dtype, int four_neighbors, int avg_res, int device,
                                    const cs_b200_opts* opts, cs_b200_handle** out, int64_t* n_out,
                                    int64_t* nnz_out, int32_t* nodemap_out) {
  if (!out) return set_err(nullptr, CS_B200_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (nrows <= 0 || ncols <= 0 || !g || (dtype != CS_B200_F32 && dtype != CS_B200_F64) ||
      nrows > (int64_t)1 << 30 || ncols > (int64_t)1 << 30)
    return set_err(nullptr, CS_B200_ERR_ARG, "bad arguments");
  if (nrows * ncols * 17 >= (int64_t)1 << 31)
    return set_err(nullptr, CS_B200_ERR_UNSUPPORTED, "raster too large: 17 * cells must be < 2^31 (device indices are int32)");
  const int64_t ncell = nrows * ncols;
  int max_poly = 0;
  if (polymap) {
    for (int64_t i = 0; i < ncell; ++i) {
      if (polymap[i] < 0) return set_err(nullptr, CS_B200_ERR_ARG, "polygon ids must be >= 0 (cell %lld holds %d)", (long long)i, polymap[i]);
      max_poly = std::max(max_poly, (int)polymap[i]);
    }
    if (max_poly > (1 << 27)) return set_err(nullptr, CS_B200_ERR_UNSUPPORTED, "polygon ids above 2^27 are not supported");
  }
  cs_b200_handle* h = new cs_b200_handle();
  h->n = 0; h->nnz = 0; h->dtype = dtype; h->device = device;
  h->owns_matrix = true;
  int rc = common_create(h, opts);
  auto fail = [&](int code) { g_create_error = h->err; cs_b200_destroy(h); return code; };
  if (rc) return fail(rc);
  cudaEventRecord(h->ev0, h->stream);
  double* d_g = nullptr;
  int* d_poly = nullptr;
  int* d_node = nullptr;
  void* d_raw = nullptr;
  csb_dev::DCsr L;
  auto cleanup = [&]() { cudaFree(d_g); cudaFree(d_poly); cudaFree(d_node); cudaFree(d_raw); };
  cudaError_t e = cudaMalloc(&d_g, (size_t)ncell * sizeof(double));
  if (e == cudaSuccess && dtype == CS_B200_F64) e = h2d(h, d_g, g, (size_t)ncell * sizeof(double));
  if (e == cudaSuccess && dtype == CS_B200_F32) {
    e = cudaMalloc(&d_raw, (size_t)ncell * sizeof(float));
    if (e == cudaSuccess) e = h2d(h, d_raw, g, (size_t)ncell * sizeof(float));
    if (e == cudaSuccess) e = (cudaError_t)csb_dev::convert_values(h->stream, (const float*)d_raw, d_g, ncell);
  }
  if (e == cudaSuccess && polymap) {
    e = cudaMalloc(&d_poly, (size_t)ncell * sizeof(int));
    if (e == cudaSuccess) e = h2d(h, d_poly, polymap, (size_t)ncell * sizeof(int));
  }
  if (e != cudaSuccess) { cleanup(); set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (raster upload)", cudaGetErrorString(e)); return fail(CS_B200_ERR_CUDA); }
  rc = csb_dev::assemble_raster_polygons(h->stream, nrows, ncols, d_g, d_poly, max_poly, four_neighbors ? 1 : 0,
                                         avg_res ? 1 : 0, L, &d_node, h->err);
  if (rc) { cleanup(); return fail(rc == -1 ? CS_B200_ERR_ARG : rc_dev(h, rc)); }
  h->n = L.nrows;
  h->nnz = L.nnz;
  h->n_pad = (h->n + 3) / 4 * 4;
  h->d_rowptr = L.ptr;
  h->d_colidx = L.idx;
  if (dtype == CS_B200_F64) {
    h->d_vals = L.val;
  } else {
    e = cudaMalloc(&h->d_vals, std::max<size_t>(1, (size_t)L.nnz) * sizeof(float));
    if (e == cudaSuccess) e = (cudaError_t)csb_dev::convert_values(h->stream, L.val, (float*)h->d_vals, L.nnz);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(L.val);
    if (e != cudaSuccess) { cleanup(); set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (value conversion)", cudaGetErrorString(e)); return fail(CS_B200_ERR_CUDA); }
  }
  if (nodemap_out) {
    e = cudaMemcpyAsync(nodemap_out, d_node, (size_t)ncell * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { cleanup(); set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (node map download)", cudaGetErrorString(e)); return fail(CS_B200_ERR_CUDA); }
  }
  cleanup();
  if (h->opts.setup != 1) {
    const csb_dev::HostPattern hp{};
    rc = dtype == CS_B200_F64 ? finish_setup_device<double>(h, hp, nullptr) : finish_setup_device<float>(h, hp, nullptr);
  } else {
    std::vector<int> rp((size_t)h->n + 1);
    e = cudaMemcpy(rp.data(), h->d_rowptr, rp.size() * sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { set_err(h, CS_B200_ERR_CUDA, "CUDA error %s reading rowptr", cudaGetErrorString(e)); return fail(CS_B200_ERR_CUDA); }
    rc = dtype == CS_B200_F64 ? finish_setup<double>(h, rp, nullptr, (const double*)nullptr)
                              : finish_setup<float>(h, rp, nullptr, (const float*)nullptr);
  }
  if (rc) return fail(rc);
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  if (n_out) *n_out = h->n;
  if (nnz_out) *nnz_out = h->nnz;
  *out = h;
  return CS_B200_OK;
}

int cs_b200_get_csr(cs_b200_handle* h, int32_t* rowptr, int32_t* colidx, void* vals) {
  if (!h) return CS_B200_ERR_ARG;
  cudaSetDevice(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  if (rowptr) CK(h, cudaMemcpy(rowptr, h->d_rowptr, (size_t)(h->n + 1) * sizeof(int), cudaMemcpyDeviceToHost));
  if (colidx) CK(h, cudaMemcpy(colidx, h->d_colidx, (size_t)h->nnz * sizeof(int), cudaMemcpyDeviceToHost));
  if (vals) CK(h, cudaMemcpy(vals, h->d_vals, (size_t)h->nnz * h->esize(), cudaMemcpyDeviceToHost));
  return CS_B200_OK;
}

static const DevCsr* pick_level(cs_b200_handle* h, int level, int which, bool* is_f32, double* omega,
                                int64_t* ncols) {
  if (!h || level < 0 || which < 0 || which > 2) return nullptr;
  std::vector<DevLevel>& lv = h->mixed ? h->lv32 : h->lv;
  if (lv.empty() && level == 0 && which == 0) {   // no hierarchy (Jacobi): the handle's own operator
    *is_f32 = h->dtype == CS_B200_F32;
    *omega = 0.0;
    *ncols = h->n;
    return &h->A0;
  }
  if (level >= (int)lv.size()) return nullptr;
  if (which > 0 && level + 1 >= (int)lv.size()) return nullptr;
  *is_f32 = h->mixed || h->dtype == CS_B200_F32;
  *omega = lv[level].omega;
  const DevCsr* m = which == 0 ? &lv[level].A : which == 1 ? &lv[level].P : &lv[level].R;
  *ncols = which == 0 ? lv[level].n : which == 1 ? lv[level + 1].n : lv[level].n;
  if (which == 2) *ncols = lv[level].n;
  return m;
}

int cs_b200_level_info(cs_b200_handle* h, int level, int which, int64_t* nrows, int64_t* ncols,
                       int64_t* nnz, double* omega, int* windowed) {
  bool f32 = false;
  double om = 0.0;
  int64_t nc = 0;
  const DevCsr* m = pick_level(h, level, which, &f32, &om, &nc);
  if (!m) return CS_B200_ERR_ARG;
  if (nrows) *nrows = m->nrows;
  if (ncols) *ncols = nc;
  if (nnz) *nnz = m->nnz;
  if (omega) *omega = om;
  if (windowed) *windowed = m->dia ? 2 : (m->win_meta ? 1 : 0);   // 2 = stencil (DIA) form
  return CS_B200_OK;
}

int cs_b200_level_csr(cs_b200_handle* h, int level, int which, int32_t* rowptr, int32_t* colidx,
                      double* vals) {
  bool f32 = false;
  double om = 0.0;
  int64_t nc = 0;
  const DevCsr* m = pick_level(h, level, which, &f32, &om, &nc);
  if (!m) return CS_B200_ERR_ARG;
  cudaSetDevice(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  if (rowptr) CK(h, cudaMemcpy(rowptr, m->rowptr, (size_t)(m->nrows + 1) * sizeof(int), cudaMemcpyDeviceToHost));
  if (colidx) CK(h, cudaMemcpy(colidx, m->colidx, (size_t)m->nnz * sizeof(int), cudaMemcpyDeviceToHost));
  if (vals) {
    if (f32) {
      std::vector<float> tmp((size_t)m->nnz);
      CK(h, cudaMemcpy(tmp.data(), m->vals, (size_t)m->nnz * sizeof(float), cudaMemcpyDeviceToHost));
      for (int64_t i = 0; i < m->nnz; ++i) vals[i] = (double)tmp[i];
    } else {
      CK(h, cudaMemcpy(vals, m->vals, (size_t)m->nnz * sizeof(double), cudaMemcpyDeviceToHost));
    }
  }
  return CS_B200_OK;
}

int cs_b200_set_grounds(cs_b200_handle* h, const void* finite_g, const uint8_t* dirichlet) {
  if (!h) return CS_B200_ERR_ARG;
  if (h->opts.setup == 1)
    return set_err(h, CS_B200_ERR_UNSUPPORTED, "cs_b200_set_grounds needs the device-side setup (opts.setup != 1)");
  if (!h->owns_matrix)
    return set_err(h, CS_B200_ERR_UNSUPPORTED, "cs_b200_set_grounds: the handle borrows its matrix (create_from_device)");
  cudaSetDevice(h->device);
  h->err.clear();
  const size_t es = h->esize();
  const size_t vb = std::max<size_t>(1, (size_t)h->nnz) * es;
  cudaEventRecord(h->ev0, h->stream);
  if (!h->d_vals0) {
    CK(h, cudaMalloc(&h->d_vals0, vb));
    CK(h, cudaMemcpyAsync(h->d_vals0, h->d_vals, vb, cudaMemcpyDeviceToDevice, h->stream));
  } else {
    CK(h, cudaMemcpyAsync(h->d_vals, h->d_vals0, vb, cudaMemcpyDeviceToDevice, h->stream));
  }
  void* d_g = nullptr;
  unsigned char* d_m = nullptr;
  auto cleanup = [&]() { cudaFree(d_g); cudaFree(d_m); };
  if (finite_g) {
    cudaError_t e = cudaMalloc(&d_g, (size_t)h->n * es);
    if (e == cudaSuccess) e = h2d(h, d_g, finite_g, (size_t)h->n * es);
    if (e != cudaSuccess) { cleanup(); return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (finite grounds)", cudaGetErrorString(e)); }
  }
  if (dirichlet) {
    cudaError_t e = cudaMalloc(&d_m, (size_t)h->n);
    if (e == cudaSuccess) e = h2d(h, d_m, dirichlet, (size_t)h->n);
    if (e != cudaSuccess) { cleanup(); return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (Dirichlet mask)", cudaGetErrorString(e)); }
  }
  if (finite_g || dirichlet) {
    const int g = (int)std::min<int64_t>((h->n + 255) / 256, (int64_t)h->num_sms * 32);
    if (h->dtype == CS_B200_F64)
      k_apply_grounds<double><<<g, 256, 0, h->stream>>>((int)h->n, h->d_rowptr, h->d_colidx, (double*)h->d_vals,
                                                        (const double*)d_g, d_m);
    else
      k_apply_grounds<float><<<g, 256, 0, h->stream>>>((int)h->n, h->d_rowptr, h->d_colidx, (float*)h->d_vals,
                                                       (const float*)d_g, d_m);
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cleanup();
  if (e != cudaSuccess) return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s applying the grounds", cudaGetErrorString(e));
  h->grounds_applied = finite_g || dirichlet;
  teardown_operators(h);
  const csb_dev::HostPattern none{};
  int rc = h->dtype == CS_B200_F64 ? build_operators<double>(h, none, nullptr, nullptr)
                                   : build_operators<float>(h, none, nullptr, nullptr);
  if (rc) return rc;
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  return CS_B200_OK;
}

int cs_b200_components(cs_b200_handle* h, int32_t* label, int64_t* ncomp) {
  if (!h) return CS_B200_ERR_ARG;
  if (!label) return set_err(h, CS_B200_ERR_ARG, "label is NULL");
  if (h->grounds_applied)
    return set_err(h, CS_B200_ERR_UNSUPPORTED, "cs_b200_components: grounds are applied (cs_b200_set_grounds)");
  cudaSetDevice(h->device);
  h->err.clear();
  const int n = (int)h->n;
  int *d_parent = nullptr, *d_flag = nullptr, *d_ord = nullptr;
  auto cleanup = [&]() { cudaFree(d_parent); cudaFree(d_flag); cudaFree(d_ord); };
#define CKC_(call)                                                                         \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      cleanup();                                                                           \
      return set_err(h, CS_B200_ERR_CUDA, "CUDA error %s at %s:%d (%s)",                   \
                     cudaGetErrorString(_e), __FILE__, __LINE__, #call);                   \
    }                                                                                      \
  } while (0)
  CKC_(cudaMalloc(&d_parent, (size_t)n * sizeof(int)));
  CKC_(cudaMalloc(&d_flag, (size_t)(n + 1) * sizeof(int)));
  CKC_(cudaMalloc(&d_ord, (size_t)(n + 1) * sizeof(int)));
  CKC_(cudaMemsetAsync(d_flag + n, 0, sizeof(int), h->stream));   // ordinal[n] = number of components
  const int grid = (int)std::min<int64_t>((h->n + 255) / 256, (int64_t)h->num_sms * 32);
  if (h->dtype == CS_B200_F64) {
    ccl::k_cc_init<double><<<grid, 256, 0, h->stream>>>(n, h->d_rowptr, h->d_colidx, (const double*)h->d_vals, d_parent);
    ccl::k_cc_hook<double><<<grid, 256, 0, h->stream>>>(n, h->d_rowptr, h->d_colidx, (const double*)h->d_vals, d_parent);
  } else {
    ccl::k_cc_init<float><<<grid, 256, 0, h->stream>>>(n, h->d_rowptr, h->d_colidx, (const float*)h->d_vals, d_parent);
    ccl::k_cc_hook<float><<<grid, 256, 0, h->stream>>>(n, h->d_rowptr, h->d_colidx, (const float*)h->d_vals, d_parent);
  }
  ccl::k_cc_flatten<<<grid, 256, 0, h->stream>>>(n, d_parent, d_flag);
  CKC_(cudaGetLastError());
  CKC_(ras::exclusive_scan(d_flag, d_ord, (int64_t)n + 1, h->stream));
  ccl::k_cc_label<<<grid, 256, 0, h->stream>>>(n, d_parent, d_ord, d_flag);
  CKC_(cudaGetLastError());
  CKC_(cudaMemcpyAsync(label, d_flag, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  int total = 0;
  CKC_(cudaMemcpyAsync(&total, d_ord + n, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CKC_(cudaStreamSynchronize(h->stream));
#undef CKC_
  cleanup();
  if (ncomp) *ncomp = total;
  return CS_B200_OK;
}

int cs_b200_get_dims(const cs_b200_handle* h, int64_t* n, int64_t* nnz) {
  if (!h) return CS_B200_ERR_ARG;
  if (n) *n = h->n;
  if (nnz) *nnz = h->nnz;
  return CS_B200_OK;
}

void cs_b200_destroy(cs_b200_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  teardown_operators(h);
  if (h->owns_matrix) { cudaFree(h->d_rowptr); cudaFree(h->d_colidx); cudaFree(h->d_vals); }
  cudaFree(h->d_vals0);
  void* bufs[] = {h->d_dinv, h->d_bstart, h->X, h->R, h->P, h->AP, h->B, h->stage,
                  h->d_cum, h->d_max, h->d_ctl, h->d_partials, h->d_flush};
  for (void* b : bufs) if (b) cudaFree(b);
  if (h->h_ctl) cudaFreeHost(h->h_ctl);
  cudaFree(h->d_sp_rows); cudaFree(h->d_sp_vals); cudaFree(h->d_sp_ptr);
  cudaFree(h->d_probe); cudaFree(h->d_probe_out);
  for (int i = 0; i < 2; ++i) {
    cudaFree(h->io_in[i]); cudaFree(h->io_out[i]);
    cudaEvent_t evs[] = {h->ev_in[i], h->ev_used[i], h->ev_ready[i], h->ev_out[i]};
    for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
  }
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev2) cudaEventDestroy(h->ev2);
  if (h->ev3) cudaEventDestroy(h->ev3);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int cs_b200_reset_currents(cs_b200_handle* h) {
  if (!h) return CS_B200_ERR_ARG;
  cudaSetDevice(h->device);
  CK(h, cudaMemsetAsync(h->d_cum, 0, (size_t)h->n_pad * h->esize(), h->stream));
  const int g = (int)std::min<int64_t>(4096, (h->n_pad + 255) / 256);
  if (h->dtype == CS_B200_F64)
    k_fill<double><<<g, 256, 0, h->stream>>>((double*)h->d_max, (size_t)h->n_pad, -9999.0);
  else
    k_fill<float><<<g, 256, 0, h->stream>>>((float*)h->d_max, (size_t)h->n_pad, -9999.0f);
  CK(h, cudaGetLastError());
  CK(h, cudaStreamSynchronize(h->stream));
  return CS_B200_OK;
}

int cs_b200_read_currents(cs_b200_handle* h, void* cum, void* max) {
  if (!h) return CS_B200_ERR_ARG;
  cudaSetDevice(h->device);
  if (cum) CK(h, cudaMemcpyAsync(cum, h->d_cum, (size_t)h->n * h->esize(), cudaMemcpyDeviceToHost, h->stream));
  if (max) CK(h, cudaMemcpyAsync(max, h->d_max, (size_t)h->n * h->esize(), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return CS_B200_OK;
}

int cs_b200_currents_device_ptrs(cs_b200_handle* h, void** d_cum, void** d_max) {
  if (!h) return CS_B200_ERR_ARG;
  if (d_cum) *d_cum = h->d_cum;
  if (d_max) *d_max = h->d_max;
  return CS_B200_OK;
}

int cs_b200_stream(cs_b200_handle* h, void** stream) {
  if (!h || !stream) return CS_B200_ERR_ARG;
  *stream = (void*)h->stream;
  return CS_B200_OK;
}

int cs_b200_profile_spmm(cs_b200_handle* h, int enable, double* total_ms, int64_t* launches) {
  if (!h) return CS_B200_ERR_ARG;
  if (total_ms) *total_ms = h->prof_ms;
  if (launches) *launches = h->prof_launches;
  if (enable >= 0) {
    h->profile = enable ? 1 : 0;
    h->prof_ms = 0.0;
    h->prof_launches = 0;
    h->prof_used = 0;
    h->prof_bytes = 0.0;
    h->prof_slot.clear();
    h->prof_pair_bytes.clear();
    for (int i = 0; i < 16; ++i) { h->prof_slot_ms[i] = 0.0; h->prof_slot_bytes[i] = 0.0; h->prof_slot_launches[i] = 0; }
  }
  return CS_B200_OK;
}

int cs_b200_profile_classes(cs_b200_handle* h, double* ms16, double* bytes16, int64_t* launches16) {
  if (!h) return CS_B200_ERR_ARG;
  for (int i = 0; i < 16; ++i) {
    if (ms16) ms16[i] = h->prof_slot_ms[i];
    if (bytes16) bytes16[i] = h->prof_slot_bytes[i];
    if (launches16) launches16[i] = h->prof_slot_launches[i];
  }
  return CS_B200_OK;
}

int cs_b200_profile_bytes(cs_b200_handle* h, double* algorithmic_bytes) {
  if (!h || !algorithmic_bytes) return CS_B200_ERR_ARG;
  *algorithmic_bytes = h->prof_bytes;
  return CS_B200_OK;
}

int cs_b200_get_stats(const cs_b200_handle* h, cs_b200_stats* out) {
  if (!h || !out) return CS_B200_ERR_ARG;
  *out = h->stats;
  return CS_B200_OK;
}

int cs_b200_spmv(cs_b200_handle* h, const void* x, void* y, int reps, double* ms_per_rep) {
  if (!h || !x || !y || reps < 1) return set_err(h, CS_B200_ERR_ARG, "bad spmv arguments");
  begin_call(h);
  const size_t bytes = (size_t)h->n * h->esize();
  CK(h, cudaMemcpyAsync(h->X, x, bytes, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaEventRecord(h->ev2, h->stream));
  for (int r = 0; r < reps; ++r) {
    if (h->dtype == CS_B200_F64)
      launch_spmm<double, 1, 0>(h, (const double*)h->X, (double*)h->AP, nullptr);
    else
      launch_spmm<float, 1, 0>(h, (const float*)h->X, (float*)h->AP, nullptr);
  }
  CK(h, cudaGetLastError());
  CK(h, cudaEventRecord(h->ev3, h->stream));
  CK(h, cudaMemcpyAsync(y, h->AP, bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  float ms = 0;
  CK(h, cudaEventElapsedTime(&ms, h->ev2, h->ev3));
  if (ms_per_rep) *ms_per_rep = ms / reps;
  h->stats.kernel_ms = ms;
  h->stats.h2d_bytes = h->stats.d2h_bytes = (double)bytes;
  end_call(h);
  return CS_B200_OK;
}

int cs_b200_spmm(cs_b200_handle* h, int k, const void* x, void* y) {
  const bool add = getenv("CS_B200_SPMM_ADD") != nullptr;   // debug: Y = X + A X through SP_ADD
  if (!h || !x || !y || (k != 1 && k != 2 && k != 4 && k != 8) || k > h->ktmax)
    return set_err(h, CS_B200_ERR_ARG, "bad spmm arguments");
  begin_call(h);
  const size_t bytes = (size_t)h->n * k * h->esize();
  const size_t nelem = (size_t)h->n_pad * k;
  const int tg = (int)std::min<size_t>(4096, (nelem + 255) / 256);
  CK(h, cudaMemcpyAsync(h->stage, x, bytes, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemsetAsync(h->X, 0, nelem * h->esize(), h->stream));
  const bool f64 = h->dtype == CS_B200_F64;
  if (f64) { DISPATCH_KT(k, (k_cm_to_panel<double, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const double*)h->stage, (double*)h->X, KT))); }
  else { DISPATCH_KT(k, (k_cm_to_panel<float, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const float*)h->stage, (float*)h->X, KT))); }
  if (add) {
    CK(h, cudaMemcpyAsync(h->AP, h->X, nelem * h->esize(), cudaMemcpyDeviceToDevice, h->stream));
    if (f64) { DISPATCH_KT(k, (launch_spmm<double, KT, SP_ADD>(h, (const double*)h->X, (double*)h->AP, (const double*)h->AP))); }
    else { DISPATCH_KT(k, (launch_spmm<float, KT, SP_ADD>(h, (const float*)h->X, (float*)h->AP, (const float*)h->AP))); }
  } else {
  if (f64) { DISPATCH_KT(k, (launch_spmm<double, KT, SP_PLAIN>(h, (const double*)h->X, (double*)h->AP, nullptr))); }
  else { DISPATCH_KT(k, (launch_spmm<float, KT, SP_PLAIN>(h, (const float*)h->X, (float*)h->AP, nullptr))); }
  }
  if (f64) { DISPATCH_KT(k, (k_panel_to_cm<double, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const double*)h->AP, (double*)h->stage, h->d_ctl, 0))); }
  else { DISPATCH_KT(k, (k_panel_to_cm<float, KT><<<tg, 256, 0, h->stream>>>((int)h->n, (size_t)h->n, (const float*)h->AP, (float*)h->stage, h->d_ctl, 0))); }
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(y, h->stage, bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  end_call(h);
  return CS_B200_OK;
}

int cs_b200_bench_spmm(cs_b200_handle* h, int k, int reps, int flush_l2, double* ms_per_rep) {
  if (!h || reps < 1 || (k != 1 && k != 2 && k != 4 && k != 8) || k > h->ktmax)
    return set_err(h, CS_B200_ERR_ARG, "bad bench_spmm arguments");
  begin_call(h);
  if (flush_l2) { int rc = ensure_flush(h); if (rc) return rc; }
  const size_t pe = (size_t)h->n_pad * k;
  const int g = (int)std::min<size_t>(4096, (pe + 255) / 256);
  if (h->dtype == CS_B200_F64) k_fill<double><<<g, 256, 0, h->stream>>>((double*)h->X, pe, 1.0);
  else k_fill<float><<<g, 256, 0, h->stream>>>((float*)h->X, pe, 1.0f);
  double total = 0;
  auto one = [&]() {
    if (h->dtype == CS_B200_F64) { DISPATCH_KT(k, (launch_spmm<double, KT, 0>(h, (const double*)h->X, (double*)h->AP, nullptr))); }
    else { DISPATCH_KT(k, (launch_spmm<float, KT, 0>(h, (const float*)h->X, (float*)h->AP, nullptr))); }
  };
  one();  // warm-up
  if (flush_l2) {
    for (int r = 0; r < reps; ++r) {
      k_flush<<<h->num_sms * 8, 256, 0, h->stream>>>(h->d_flush, h->flush_elems);
      CK(h, cudaEventRecord(h->ev2, h->stream));
      one();
      CK(h, cudaEventRecord(h->ev3, h->stream));
      CK(h, cudaEventSynchronize(h->ev3));
      float ms = 0;
      CK(h, cudaEventElapsedTime(&ms, h->ev2, h->ev3));
      total += ms;
    }
  } else {
    CK(h, cudaEventRecord(h->ev2, h->stream));
    for (int r = 0; r < reps; ++r) one();
    CK(h, cudaEventRecord(h->ev3, h->stream));
    CK(h, cudaEventSynchronize(h->ev3));
    float ms = 0;
    CK(h, cudaEventElapsedTime(&ms, h->ev2, h->ev3));
    total = ms;
  }
  CK(h, cudaGetLastError());
  if (ms_per_rep) *ms_per_rep = total / reps;
  h->stats.kernel_ms = total;
  end_call(h);
  return CS_B200_OK;
}

int cs_b200_bench_cg_iter(cs_b200_handle* h, int k, int reps, double* ms_per_rep) {
  if (!h || reps < 1 || (k != 1 && k != 2 && k != 4 && k != 8) || k > h->ktmax)
    return set_err(h, CS_B200_ERR_ARG, "bad bench_cg_iter arguments");
  begin_call(h);
  PanelCtl* hc = h->h_ctl;
  std::memset(hc, 0, sizeof(PanelCtl));
  for (int c = 0; c < k; ++c) {
    hc->src[c] = (c * 7919) % h->n;
    hc->dst[c] = h->n - 1 - (c * 104729) % (h->n / 2 + 1);
    if (hc->dst[c] == hc->src[c]) hc->dst[c] = (hc->src[c] + 1) % h->n;
    hc->weight[c] = 1.0;
  }
  CK(h, cudaMemcpyAsync(h->d_ctl, hc, sizeof(PanelCtl), cudaMemcpyHostToDevice, h->stream));
  const size_t nelem = (size_t)h->n_pad * k;
  CK(h, cudaMemsetAsync(h->B, 0, nelem * h->esize(), h->stream));
  const bool f64 = h->dtype == CS_B200_F64;
#define BOTH(CALLD, CALLF) do { if (f64) { DISPATCH_KT(k, CALLD); } else { DISPATCH_KT(k, CALLF); } } while (0)
  BOTH((k_pair_rhs<double, KT><<<1, 32, 0, h->stream>>>((double*)h->B, h->d_ctl)),
       (k_pair_rhs<float, KT><<<1, 32, 0, h->stream>>>((float*)h->B, h->d_ctl)));
  BOTH((k_cg_init<double, KT><<<ew_grid<double, KT>(h), NT, 0, h->stream>>>(nelem, (const double*)h->B, (const double*)h->d_dinv, (double*)h->X, (double*)h->R, (double*)h->P, h->d_ctl, h->d_partials, 0.0, 0.0, 1 << 30)),
       (k_cg_init<float, KT><<<ew_grid<float, KT>(h), NT, 0, h->stream>>>(nelem, (const float*)h->B, (const float*)h->d_dinv, (float*)h->X, (float*)h->R, (float*)h->P, h->d_ctl, h->d_partials, 0.0, 0.0, 1 << 30)));
  for (int w = 0; w < 3; ++w) BOTH((launch_iteration<double, KT>(h)), (launch_iteration<float, KT>(h)));
  CK(h, cudaEventRecord(h->ev2, h->stream));
  for (int r = 0; r < reps; ++r) BOTH((launch_iteration<double, KT>(h)), (launch_iteration<float, KT>(h)));
  CK(h, cudaEventRecord(h->ev3, h->stream));
  CK(h, cudaEventSynchronize(h->ev3));
  CK(h, cudaGetLastError());
  float ms = 0;
  CK(h, cudaEventElapsedTime(&ms, h->ev2, h->ev3));
  if (ms_per_rep) *ms_per_rep = ms / reps;
  h->stats.kernel_ms = ms;
  end_call(h);
  return CS_B200_OK;
}

int cs_b200_solve_rhs(cs_b200_handle* h, int64_t k, const void* rhs, void* lhs, double rtol,
                      int64_t itmax, int64_t* iters, double* relres) {
  if (!h || k < 1 || !rhs || !lhs || !(rtol >= 0) || itmax < 0)
    return set_err(h, CS_B200_ERR_ARG, "bad solve_rhs arguments");
  begin_call(h);
  int rc = h->dtype == CS_B200_F64
               ? solve_rhs_t<double>(h, k, (const double*)rhs, (double*)lhs, rtol, itmax, iters, relres)
               : solve_rhs_t<float>(h, k, (const float*)rhs, (float*)lhs, rtol, itmax, iters, relres);
  end_call(h);
  return rc;
}

int cs_b200_solve_pairs(cs_b200_handle* h, int64_t k, const int64_t* src, const int64_t* dst,
                        const double* weight, double rtol, int64_t itmax, void* R, void* volt,
                        void* curr, int accumulate, int64_t* iters, double* relres) {
  if (!h || k < 1 || !src || !dst || !R || !(rtol >= 0) || itmax < 0)
    return set_err(h, CS_B200_ERR_ARG, "bad solve_pairs arguments");
  for (int64_t c = 0; c < k; ++c)
    if (src[c] < 0 || src[c] >= h->n || dst[c] < 0 || dst[c] >= h->n || src[c] == dst[c])
      return set_err(h, CS_B200_ERR_ARG, "pair %lld: src/dst out of range or equal (%lld, %lld)",
                     (long long)c, (long long)src[c], (long long)dst[c]);
  begin_call(h);
  int rc = h->dtype == CS_B200_F64
               ? solve_pairs_t<double>(h, k, src, dst, weight, rtol, itmax, (double*)R,
                                       (double*)volt, (double*)curr, accumulate, iters, relres)
               : solve_pairs_t<float>(h, k, src, dst, weight, rtol, itmax, (float*)R, (float*)volt,
                                      (float*)curr, accumulate, iters, relres);
  end_call(h);
  return rc;
}

int cs_b200_solve_sources(cs_b200_handle* h, int64_t k, const int64_t* colptr, const int64_t* rows,
                          const double* vals, const int64_t* ref, const double* weight,
                          double rtol, int64_t itmax, int64_t nprobe, const int64_t* probe,
                          void* probe_volt, void* volt, void* curr, int accumulate,
                          int64_t* iters, double* relres) {
  if (!h || k < 1 || !colptr || !ref || !(rtol >= 0) || itmax < 0 || nprobe < 0 ||
      (nprobe > 0 && !probe) || colptr[0] != 0)
    return set_err(h, CS_B200_ERR_ARG, "bad solve_sources arguments");
  for (int64_t c = 0; c < k; ++c) {
    if (colptr[c + 1] < colptr[c] || ref[c] < 0 || ref[c] >= h->n)
      return set_err(h, CS_B200_ERR_ARG, "column %lld: bad colptr or reference row", (long long)c);
  }
  if (colptr[k] > 0 && (!rows || !vals)) return set_err(h, CS_B200_ERR_ARG, "rows/vals missing");
  for (int64_t e = 0; e < colptr[k]; ++e)
    if (rows[e] < 0 || rows[e] >= h->n)
      return set_err(h, CS_B200_ERR_ARG, "entry %lld: row %lld out of range", (long long)e, (long long)rows[e]);
  for (int64_t i = 0; i < nprobe; ++i)
    if (probe[i] < 0 || probe[i] >= h->n) return set_err(h, CS_B200_ERR_ARG, "probe row out of range");
  begin_call(h);
  int rc = h->dtype == CS_B200_F64
               ? solve_sources_t<double>(h, k, colptr, rows, vals, ref, weight, rtol, itmax, nprobe, probe,
                                         (double*)probe_volt, (double*)volt, (double*)curr, accumulate,
                                         iters, relres)
               : solve_sources_t<float>(h, k, colptr, rows, vals, ref, weight, rtol, itmax, nprobe, probe,
                                        (float*)probe_volt, (float*)volt, (float*)curr, accumulate, iters,
                                        relres);
  end_call(h);
  return rc;
}

int cs_b200_solve_pairs_superposed(cs_b200_handle* h, int64_t np, const int64_t* nodes, int64_t k,
                                   const int64_t* pi, const int64_t* pj, const double* weight,
                                   double rtol, int64_t itmax, void* R, void* volt, void* curr,
                                   int accumulate, int64_t* point_iters, double* relres) {
  if (!h || np < 2 || !nodes || k < 1 || !pi || !pj || !R || !(rtol >= 0) || itmax < 0)
    return set_err(h, CS_B200_ERR_ARG, "bad solve_pairs_superposed arguments");
  for (int64_t x = 0; x < np; ++x) {
    if (nodes[x] < 0 || nodes[x] >= h->n)
      return set_err(h, CS_B200_ERR_ARG, "focal node %lld out of range", (long long)x);
    if (x > 0 && nodes[x] == nodes[0])
      return set_err(h, CS_B200_ERR_ARG, "focal node %lld repeats the reference node", (long long)x);
  }
  for (int64_t c = 0; c < k; ++c)
    if (pi[c] < 0 || pi[c] >= np || pj[c] < 0 || pj[c] >= np || nodes[pi[c]] == nodes[pj[c]])
      return set_err(h, CS_B200_ERR_ARG, "pair %lld: indices out of range or equal nodes", (long long)c);
  begin_call(h);
  int rc = h->dtype == CS_B200_F64
               ? solve_pairs_superposed_t<double>(h, np, nodes, k, pi, pj, weight, rtol, itmax, (double*)R,
                                                  (double*)volt, (double*)curr, accumulate, point_iters, relres)
               : solve_pairs_superposed_t<float>(h, np, nodes, k, pi, pj, weight, rtol, itmax, (float*)R,
                                                 (float*)volt, (float*)curr, accumulate, point_iters, relres);
  end_call(h);
  return rc;
}

}  // extern "C"
// ---------------------------------------------------------------------------------------------
// multi-GPU: NCCL behind the C ABI (loaded at run time, so a single-GPU user needs no NCCL)
// ---------------------------------------------------------------------------------------------
#include <dlfcn.h>

namespace {

struct NcclId { char internal[128]; };
typedef void* ncclComm_p;
// enums of nccl.h (stable across NCCL 2.x)
enum { NCCL_INT8 = 0, NCCL_INT32 = 2, NCCL_INT64 = 4, NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8 };
enum { NCCL_SUM = 0, NCCL_MAX = 2 };

struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(ncclComm_p*, int, NcclId, int) = nullptr;
  int (*CommDestroy)(ncclComm_p) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_p, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::string err;
};

NcclApi& nccl_api() {
  static NcclApi api;
  if (api.lib || !api.err.empty()) return api;
  const char* names[] = {std::getenv("CS_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    if (!nm) continue;
    api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) { api.err = std::string("cannot load NCCL (libnccl.so.2): ") + dlerror(); return api; }
  auto sym = [&](const char* s) { void* p = dlsym(api.lib, s); if (!p) api.err = std::string("NCCL symbol missing: ") + s; return p; };
  api.GetUniqueId = (int (*)(NcclId*))sym("ncclGetUniqueId");
  api.CommInitRank = (int (*)(ncclComm_p*, int, NcclId, int))sym("ncclCommInitRank");
  api.CommDestroy = (int (*)(ncclComm_p))sym("ncclCommDestroy");
  api.Broadcast = (int (*)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t))sym("ncclBroadcast");
  api.AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t))sym("ncclAllReduce");
  api.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_p, cudaStream_t))sym("ncclAllGather");
  api.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
  return api;
}

thread_local std::string g_comm_error;

}  // namespace

struct cs_b200_comm {
  int device = 0, rank = 0, nranks = 1;
  ncclComm_p comm = nullptr;
  cudaStream_t stream = nullptr;
  std::string err;
};

namespace {
int comm_err(cs_b200_comm* c, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_comm_error = buf;
  return code;
}
#define CKN(c, call)                                                                                  \
  do {                                                                                                \
    int _r = (call);                                                                                  \
    if (_r != 0) return comm_err(c, CS_B200_ERR_CUDA, "NCCL error %s (%s)", nccl_api().GetErrorString(_r), #call); \
  } while (0)
#define CKU(c, call)                                                                                  \
  do {                                                                                                \
    cudaError_t _e = (call);                                                                          \
    if (_e != cudaSuccess) return comm_err(c, CS_B200_ERR_CUDA, "CUDA error %s (%s)", cudaGetErrorString(_e), #call); \
  } while (0)
}  // namespace

extern "C" {

int cs_b200_comm_unique_id(void* id128) {
  if (!id128) return comm_err(nullptr, CS_B200_ERR_ARG, "id128 is NULL");
  NcclApi& api = nccl_api();
  if (!api.err.empty()) return comm_err(nullptr, CS_B200_ERR_UNSUPPORTED, "%s", api.err.c_str());
  NcclId id;
  CKN(nullptr, api.GetUniqueId(&id));
  std::memcpy(id128, &id, sizeof id);
  return CS_B200_OK;
}

int cs_b200_comm_init(int device, int rank, int nranks, const void* id128, cs_b200_comm** out) {
  if (!out || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return comm_err(nullptr, CS_B200_ERR_ARG, "bad comm_init arguments");
  *out = nullptr;
  NcclApi& api = nccl_api();
  if (!api.err.empty()) return comm_err(nullptr, CS_B200_ERR_UNSUPPORTED, "%s", api.err.c_str());
  CKU(nullptr, cudaSetDevice(device));
  cs_b200_comm* c = new cs_b200_comm();
  c->device = device; c->rank = rank; c->nranks = nranks;
  NcclId id;
  std::memcpy(&id, id128, sizeof id);
  int r = api.CommInitRank(&c->comm, nranks, id, rank);
  if (r != 0) { comm_err(nullptr, CS_B200_ERR_CUDA, "NCCL error %s (ncclCommInitRank)", api.GetErrorString(r)); delete c; return CS_B200_ERR_CUDA; }
  cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { comm_err(nullptr, CS_B200_ERR_CUDA, "CUDA error %s creating the comm stream", cudaGetErrorString(e)); api.CommDestroy(c->comm); delete c; return CS_B200_ERR_CUDA; }
  *out = c;
  return CS_B200_OK;
}

void cs_b200_comm_destroy(cs_b200_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
  if (c->comm) nccl_api().CommDestroy(c->comm);
  delete c;
}

const char* cs_b200_comm_last_error(const cs_b200_comm* c) { return c ? c->err.c_str() : g_comm_error.c_str(); }

int cs_b200_comm_barrier(cs_b200_comm* c) {
  if (!c) return CS_B200_ERR_ARG;
  cudaSetDevice(c->device);
  int* d = nullptr;
  CKU(c, cudaMalloc(&d, sizeof(int)));
  cudaMemsetAsync(d, 0, sizeof(int), c->stream);
  int r = nccl_api().AllReduce(d, d, 1, NCCL_INT32, NCCL_SUM, c->comm, c->stream);
  cudaError_t e = cudaStreamSynchronize(c->stream);
  cudaFree(d);
  if (r != 0) return comm_err(c, CS_B200_ERR_CUDA, "NCCL error %s (barrier)", nccl_api().GetErrorString(r));
  CKU(c, e);
  return CS_B200_OK;
}

int cs_b200_comm_max_double(cs_b200_comm* c, double* v, int count) {
  if (!c || !v || count < 1) return CS_B200_ERR_ARG;
  cudaSetDevice(c->device);
  double* d = nullptr;
  CKU(c, cudaMalloc(&d, (size_t)count * sizeof(double)));
  cudaMemcpyAsync(d, v, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c->stream);
  int r = nccl_api().AllReduce(d, d, (size_t)count, NCCL_FLOAT64, NCCL_MAX, c->comm, c->stream);
  cudaMemcpyAsync(v, d, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
  cudaError_t e = cudaStreamSynchronize(c->stream);
  cudaFree(d);
  if (r != 0) return comm_err(c, CS_B200_ERR_CUDA, "NCCL error %s (max_double)", nccl_api().GetErrorString(r));
  CKU(c, e);
  return CS_B200_OK;
}

int cs_b200_comm_reduce_currents(cs_b200_comm* c, cs_b200_handle* h) {
  if (!c || !h || h->device != c->device) return comm_err(c, CS_B200_ERR_ARG, "bad reduce_currents arguments");
  cudaSetDevice(c->device);
  const int dt = h->dtype == CS_B200_F64 ? NCCL_FLOAT64 : NCCL_FLOAT32;
  // on the handle's own stream: ordered right behind the last accumulation kernel, no host sync between
  CKN(c, nccl_api().AllReduce(h->d_cum, h->d_cum, (size_t)h->n, dt, NCCL_SUM, c->comm, h->stream));
  CKN(c, nccl_api().AllReduce(h->d_max, h->d_max, (size_t)h->n, dt, NCCL_MAX, c->comm, h->stream));
  CKU(c, cudaStreamSynchronize(h->stream));
  return CS_B200_OK;
}

int cs_b200_comm_gather_pairs(cs_b200_comm* c, int64_t k_total, const int64_t* my_idx, int64_t k_mine,
                              const double* my_R, double* R_all) {
  if (!c || k_total < 1 || k_mine < 0 || (k_mine > 0 && (!my_idx || !my_R)) || !R_all)
    return comm_err(c, CS_B200_ERR_ARG, "bad gather_pairs arguments");
  cudaSetDevice(c->device);
  // fixed-size slots: ceil(k_total / nranks) (index, value) pairs per rank, index -1 = empty
  const int64_t slot = (k_total + c->nranks - 1) / c->nranks;
  if (k_mine > slot) return comm_err(c, CS_B200_ERR_ARG, "rank %d holds %lld pairs, more than ceil(k_total / nranks) = %lld", c->rank, (long long)k_mine, (long long)slot);
  std::vector<double> send((size_t)2 * slot, -1.0), recv((size_t)2 * slot * c->nranks);
  for (int64_t i = 0; i < k_mine; ++i) { send[2 * i] = (double)my_idx[i]; send[2 * i + 1] = my_R[i]; }
  double *ds = nullptr, *dr = nullptr;
  CKU(c, cudaMalloc(&ds, send.size() * sizeof(double)));
  cudaError_t e = cudaMalloc(&dr, recv.size() * sizeof(double));
  if (e != cudaSuccess) { cudaFree(ds); CKU(c, e); }
  cudaMemcpyAsync(ds, send.data(), send.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream);
  int r = nccl_api().AllGather(ds, dr, send.size(), NCCL_FLOAT64, c->comm, c->stream);
  cudaMemcpyAsync(recv.data(), dr, recv.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
  e = cudaStreamSynchronize(c->stream);
  cudaFree(ds); cudaFree(dr);
  if (r != 0) return comm_err(c, CS_B200_ERR_CUDA, "NCCL error %s (gather_pairs)", nccl_api().GetErrorString(r));
  CKU(c, e);
  for (int64_t i = 0; i < k_total; ++i) R_all[i] = -1.0;
  for (size_t q = 0; q + 1 < recv.size(); q += 2) {
    const int64_t idx = (int64_t)recv[q];
    if (idx >= 0 && idx < k_total) R_all[idx] = recv[q + 1];
  }
  return CS_B200_OK;
}

int cs_b200_create_bcast(cs_b200_comm* c, int root, int64_t n, int64_t nnz, const void* rowptr,
                         const void* colidx, const void* vals, int index_bits, int index_base,
                         int dtype, const cs_b200_opts* opts, cs_b200_handle** out) {
  if (!out) return comm_err(c, CS_B200_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (!c || root < 0 || root >= c->nranks || n <= 0 || nnz <= 0 || (dtype != CS_B200_F32 && dtype != CS_B200_F64) ||
      nnz >= (int64_t)1 << 31 || n >= (int64_t)1 << 31 || (index_bits != 32 && index_bits != 64) ||
      (index_base != 0 && index_base != 1))
    return comm_err(c, CS_B200_ERR_ARG, "bad create_bcast arguments");
  const bool is_root = c->rank == root;
  if (is_root && (!rowptr || !colidx || !vals)) return comm_err(c, CS_B200_ERR_ARG, "the root rank must pass the matrix");
  cs_b200_handle* h = new cs_b200_handle();
  h->n = n; h->nnz = nnz; h->dtype = dtype; h->device = c->device;
  int rc = common_create(h, opts);
  auto fail = [&](int code) { c->err = h->err; g_create_error = h->err; cs_b200_destroy(h); return code; };
  if (rc) return fail(rc);
  cudaEventRecord(h->ev0, h->stream);
  const size_t es = h->esize();
  const bool amg = h->opts.precond == CS_B200_PRECOND_AMG && n > 200 && h->opts.setup != 1;
  csb_dev::SeedJob* job = nullptr;
  const csb_dev::HostPattern hp{rowptr, colidx, index_bits, index_base};
  if (is_root && amg) job = csb_dev::seed_start(n, hp);   // overlaps the upload and the broadcast
  auto fail_job = [&](int code) { csb_dev::seed_discard(job); job = nullptr; return fail(code); };
#define CKB(call)                                                                                  \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      set_err(h, CS_B200_ERR_CUDA, "CUDA error %s (%s)", cudaGetErrorString(_e), #call);           \
      return fail_job(CS_B200_ERR_CUDA);                                                           \
    }                                                                                              \
  } while (0)
#define CKBN(call)                                                                                 \
  do {                                                                                             \
    int _r = (call);                                                                               \
    if (_r != 0) {                                                                                 \
      set_err(h, CS_B200_ERR_CUDA, "NCCL error %s (%s)", nccl_api().GetErrorString(_r), #call);    \
      return fail_job(CS_B200_ERR_CUDA);                                                           \
    }                                                                                              \
  } while (0)
  CKB(cudaMalloc(&h->d_rowptr, (size_t)(n + 1) * sizeof(int)));
  CKB(cudaMalloc(&h->d_colidx, (size_t)nnz * sizeof(int)));
  CKB(cudaMalloc(&h->d_vals, (size_t)nnz * es));
  if (is_root) {
    if (index_bits == 32 && index_base == 0) {
      CKB(cudaMemcpyAsync(h->d_rowptr, rowptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
      CKB(cudaMemcpyAsync(h->d_colidx, colidx, (size_t)nnz * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    } else {
      const size_t ib = index_bits / 8;
      void* raw = nullptr;
      CKB(cudaMalloc(&raw, std::max<size_t>((size_t)(n + 1), (size_t)nnz) * ib));
      cudaError_t e = cudaMemcpyAsync(raw, rowptr, (size_t)(n + 1) * ib, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = (cudaError_t)csb_dev::narrow_indices(h->stream, raw, index_bits, index_base, n + 1, h->d_rowptr);
      if (e == cudaSuccess) e = cudaMemcpyAsync(raw, colidx, (size_t)nnz * ib, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = (cudaError_t)csb_dev::narrow_indices(h->stream, raw, index_bits, index_base, nnz, h->d_colidx);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      cudaFree(raw);
      CKB(e);
    }
    CKB(cudaMemcpyAsync(h->d_vals, vals, (size_t)nnz * es, cudaMemcpyHostToDevice, h->stream));
  }
  // one broadcast of the CSR (SURVEY.md 8e), on the handle's stream behind the upload
  NcclApi& api = nccl_api();
  CKBN(api.Broadcast(h->d_rowptr, h->d_rowptr, (size_t)(n + 1), NCCL_INT32, root, c->comm, h->stream));
  CKBN(api.Broadcast(h->d_colidx, h->d_colidx, (size_t)nnz, NCCL_INT32, root, c->comm, h->stream));
  CKBN(api.Broadcast(h->d_vals, h->d_vals, (size_t)nnz * es, NCCL_INT8, root, c->comm, h->stream));
  // the root's ordered aggregation seeds travel the same way (n ints) instead of every rank
  // downloading the pattern and repeating the pass
  int* d_seed = nullptr;
  csb_dev::DeviceSeed ds;
  if (amg) {
    CKB(cudaMalloc(&d_seed, (size_t)(n + 1) * sizeof(int)));
    if (is_root) {
      const int* seed = nullptr;
      int64_t cnt = 0;
      const int nagg = csb_dev::seed_wait(job, &seed, &cnt);
      cudaError_t e = cudaMemcpyAsync(d_seed, seed, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = cudaMemcpyAsync(d_seed + n, &nagg, sizeof(int), cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      csb_dev::seed_discard(job);
      job = nullptr;
      if (e != cudaSuccess) { cudaFree(d_seed); CKB(e); }
    }
    int r = api.Broadcast(d_seed, d_seed, (size_t)(n + 1), NCCL_INT32, root, c->comm, h->stream);
    int nagg = 0;
    cudaError_t e = cudaMemcpyAsync(&nagg, d_seed + n, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (r != 0 || e != cudaSuccess) {
      cudaFree(d_seed);
      set_err(h, CS_B200_ERR_CUDA, "broadcast of the aggregation seeds failed (%s)", r != 0 ? api.GetErrorString(r) : cudaGetErrorString(e));
      return fail_job(CS_B200_ERR_CUDA);
    }
    ds.d_seed = d_seed;
    ds.nagg = nagg;
  }
#undef CKB
#undef CKBN
  if (h->opts.setup != 1) {
    const csb_dev::HostPattern none{};
    rc = dtype == CS_B200_F64 ? finish_setup_device<double>(h, none, nullptr, amg ? &ds : nullptr)
                              : finish_setup_device<float>(h, none, nullptr, amg ? &ds : nullptr);
  } else {
    std::vector<int> rp(n + 1);
    cudaError_t e = cudaMemcpy(rp.data(), h->d_rowptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { cudaFree(d_seed); set_err(h, CS_B200_ERR_CUDA, "CUDA error %s reading rowptr", cudaGetErrorString(e)); return fail(CS_B200_ERR_CUDA); }
    rc = dtype == CS_B200_F64 ? finish_setup<double>(h, rp, nullptr, (const double*)nullptr)
                              : finish_setup<float>(h, rp, nullptr, (const float*)nullptr);
  }
  cudaFree(d_seed);
  if (rc) return fail(rc);
  cudaEventRecord(h->ev1, h->stream);
  cudaEventSynchronize(h->ev1);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev0, h->ev1);
  h->stats.setup_ms = ms;
  *out = h;
  return CS_B200_OK;
}

}  // extern "C"
