/*
 * cs_b200.h -- C ABI of libcsb200.so: a B200-native (sm_100a) replacement for the
 * inner Laplacian-solve loop of Circuitscape.jl (pairwise + advanced mode).
 *
 * This is the drop-in boundary.  The reference (Julia) reaches a solver through
 * three methods that package extensions overload (ext/CircuitscapePardisoExt.jl:31-45,
 * ext/CircuitscapeAppleAccelerateExt.jl:8-22):
 *
 *   construct_cholesky_factor(matrix, solver)          src/core.jl:379,519-523
 *        -> cs_b200_create            (once per connected component)
 *   solve_linear_system(factor, matrix, rhs::Matrix)   src/core.jl:463,646-653
 *        -> cs_b200_solve_rhs         (n x k column-major in, n x k out, true
 *                                      residual gate 1e-4 reported per column)
 *   multiple_solve(solver, matrix, sources::Vector)    src/raster/advanced.jl:307-333
 *        -> cs_b200_create + cs_b200_solve_rhs(k = 1)
 *
 * and the batched driver around them (src/core.jl:312-515: RHS  -1 at src, +1 at
 * dst; shift so v[src] = 0; R = v[dst] - v[src]; per-pair node currents
 * src/out.jl:178-290 accumulated into cumulative / max maps src/out.jl:100-107)
 * is offered as ONE device-resident call so n x k voltages never cross PCIe:
 *
 *        -> cs_b200_solve_pairs / cs_b200_solve_sources  + cs_b200_read_currents
 *
 * All entry points use plain pointers and sizes; every function returns 0 on
 * success or a negative cs_b200_status; cs_b200_last_error() gives the text.
 * Host buffers are copied during the call (the caller keeps ownership; Julia:
 * GC.@preserve).  A handle is NOT re-entrant: one in-flight call per handle.
 * INTEGRATION.md shows the Julia `ccall` glue that binds these symbols.
 */
#ifndef CS_B200_H
#define CS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cs_b200_handle cs_b200_handle;

enum cs_b200_status {
  CS_B200_OK = 0,
  CS_B200_ERR_ARG = -1,        /* bad argument                                    */
  CS_B200_ERR_CUDA = -2,       /* CUDA runtime error (no GPU, OOM, launch failure) */
  CS_B200_ERR_RESIDUAL = -3,   /* a column failed the true-residual gate (1e-4), the
                                  reference's `error("... exceeds tolerance 1e-4")`,
                                  src/core.jl:641,650                              */
  CS_B200_ERR_MAXITER = -4,    /* itmax reached, or a column's recurrence stagnated (reduced-precision
                                  storage), before rtol: results still written, relres[] says how far */
  CS_B200_ERR_UNSUPPORTED = -5
};

enum cs_b200_dtype { CS_B200_F32 = 0, CS_B200_F64 = 1 };

enum cs_b200_precond {
  CS_B200_PRECOND_JACOBI = 0,  /* D^-1, built on device                            */
  CS_B200_PRECOND_AMG = 1      /* aggregation multigrid V-cycle, Jacobi-smoothed
                                  (the reference's AMG role, src/core.jl:164-167)  */
};

/* Options; zero-initialise then override.  0 means "library default".             */
typedef struct cs_b200_opts {
  int32_t precond;        /* cs_b200_precond                                       */
  int32_t panel_width;    /* RHS columns solved together per panel: 1,2,4,8 (def 8) */
  int32_t check_every;    /* CG iterations between host convergence polls (def 16)  */
  int32_t use_graph;      /* 0/1: whole PCG loop as a device-side WHILE graph (def);
                             2: host-polled graph chunks of check_every iterations;
                             -1: plain launches                                       */
  double atol;            /* absolute term of the stop test; 0 => sqrt(eps(Float64)), the
                             Krylov.jl default in force at src/core.jl:639; <0 => none */
  double resid_gate;      /* true-residual gate (def 1e-4, src/core.jl:641)         */
  int32_t log_transform;  /* current maps accumulate log10(c) (src/out.jl:305-309)  */
  int32_t window;         /* TMA-staged windowed SpMM: 0 auto (operators >= 20000 rows),
                             1 always, -1 never (plain direct-gather kernel)         */
  int32_t mixed;          /* fp64 handles with AMG: run the V-cycle in fp32 (CG vectors,
                             dot products and the residual gate stay fp64): 0 auto (on),
                             -1 off                                                  */
  int32_t setup;          /* where the multigrid hierarchy and the windowed records are built:
                             0 auto (on the device), 1 on the host (amg_host.hpp / win_host.hpp,
                             the round-1 path, kept for A/B checks), 2 on the device           */
  int32_t stencil;        /* stencil (DIA) SpMM for operators whose entries all sit on the 9 raster
                             diagonals (full rasters, regular coarse grids): 0 auto (operators
                             >= 20000 rows), 1 always, -1 never                                */
  int32_t reserved[3];
} cs_b200_opts;

/* Per-call statistics (milliseconds measured with CUDA events on the solve stream). */
typedef struct cs_b200_stats {
  double setup_ms;        /* create: upload + preconditioner build                  */
  double solve_ms;        /* last solve_*: device time incl. H2D/D2H inside the call */
  double kernel_ms;       /* last solve_*: iteration kernels only                   */
  int64_t iterations;     /* last solve_*: sum over columns                         */
  int64_t spmm_launches;  /* last solve_*: SpMM kernel launches                     */
  int64_t kernel_launches;/* last solve_*: all kernel launches                      */
  double h2d_bytes, d2h_bytes;
} cs_b200_stats;

/* Build the device-resident operator for one connected component.
 * CSR of a symmetric matrix (so Julia's SparseMatrixCSC colptr/rowval/nzval can be
 * passed as-is).  index_bits in {32,64}: width of rowptr/colidx entries;
 * index_base in {0,1}; dtype: type of `vals`, of all RHS/solution buffers and of the
 * device arithmetic.  device: CUDA ordinal.  opts may be NULL.                      */
int cs_b200_create(int64_t n, int64_t nnz, const void* rowptr, const void* colidx,
                   const void* vals, int index_bits, int index_base, int dtype,
                   int device, const cs_b200_opts* opts, cs_b200_handle** out);

/* Same, but rowptr/colidx/vals already live on `device` (int32 0-based indices,
 * values of `dtype`).  Used after an NCCL broadcast of the matrix to peer GPUs.    */
int cs_b200_create_from_device(int64_t n, int64_t nnz, const int32_t* d_rowptr,
                               const int32_t* d_colidx, const void* d_vals, int dtype,
                               int device, const cs_b200_opts* opts, cs_b200_handle** out);

/* The step BEFORE the path (SURVEY.md 8f rank 2): assemble the Laplacian of a conductance raster
 * on the device and build the handle on it -- construct_node_map without polygons
 * (src/raster/pairwise.jl:271-281), construct_graph (src/raster/pairwise.jl:317-367) and
 * laplacian! (src/core.jl:608-624) as three kernels around two prefix sums; nothing of size nnz
 * is built on the host or crosses PCIe on the way in.
 * g: host, COLUMN-major nrows x ncols (a Julia Matrix as it lies in memory), element type `dtype`;
 * cells with g <= 0 (0, NODATA -9999, NaN) are not nodes.  Nodes are numbered 0.. in memory
 * order over the valid cells -- the reference's numbering minus one.  avg_res / four_neighbors:
 * connect_using_avg_resistances / connect_four_neighbors_only.  The whole raster becomes ONE
 * operator (block diagonal over its connected components; a solve's sources and ground must
 * lie in one component, as they do in the reference's per-component calls).
 * *n_out / *nnz_out (optional): nodes and stored entries of the assembled matrix.            */
int cs_b200_create_from_raster(int64_t nrows, int64_t ncols, const void* g, int dtype,
                               int four_neighbors, int avg_res, int device,
                               const cs_b200_opts* opts, cs_b200_handle** out,
                               int64_t* n_out, int64_t* nnz_out);

/* Same with SHORT-CIRCUIT POLYGONS (construct_node_map with a polygon map, src/raster/pairwise.jl:283-314):
 * polymap: host, column-major nrows x ncols int32, 0 = no polygon (NULL = none).  Every cell of a polygon,
 * NODATA cells included, takes the node of the polygon's first valid cell; node labels are compacted in
 * order; parallel cell adjacencies between merged nodes add up and adjacencies inside a node vanish
 * (sparse(I,J,V) + laplacian!, src/core.jl:608-624).  nodemap_out (optional): host, column-major
 * nrows x ncols int32, the node id of every cell (1-based like the reference's nodemap, 0 = none) --
 * what the host needs to place focal points, sources and grounds.                                   */
int cs_b200_create_from_raster_poly(int64_t nrows, int64_t ncols, const void* g, const int32_t* polymap,
                                    int dtype, int four_neighbors, int avg_res, int device,
                                    const cs_b200_opts* opts, cs_b200_handle** out, int64_t* n_out,
                                    int64_t* nnz_out, int32_t* nodemap_out);

/* Copy the handle's CSR (0-based, int32 indices, values of the handle's dtype) to host buffers
 * of n+1, nnz and nnz elements; any pointer may be NULL.  Parity / debugging hook.            */
int cs_b200_get_csr(cs_b200_handle* h, int32_t* rowptr, int32_t* colidx, void* vals);

/* Advanced mode on a RESIDENT operator (src/raster/advanced.jl:274-305): the reference rebuilds
 * `G + diag(finite grounds)` with the rows / columns of the Inf grounds deleted for every solve; here
 * the handle keeps the component's Laplacian and this call re-derives the operator on the device:
 *     finite_g  (n values of the handle's dtype, or NULL)   added to the diagonal
 *     dirichlet (n bytes, non-zero = tied to ground, or NULL) row and column replaced by the identity
 *                                                           row -- the deleted row with its 0 V kept in place
 * then 1/diag, the stencil / window records and the multigrid hierarchy are rebuilt from the device-
 * resident CSR (no matrix crosses PCIe; ~0.1 s at 10^6 nodes).  Right-hand sides passed afterwards must
 * be zero at the Dirichlet rows (the reference drops those sources).  Calling it again starts from the
 * pristine values; NULL, NULL restores the original operator.  Needs the device-side setup and a
 * handle that owns its matrix.                                                                    */
int cs_b200_set_grounds(cs_b200_handle* h, const void* finite_g, const uint8_t* dirichlet);

/* Multigrid hierarchy inspection (parity / debugging hooks; levels exist only with the AMG
 * preconditioner).  which: 0 = operator A_l, 1 = prolongator P_l (level l <- l+1), 2 = restriction
 * R_l = P_l^T.  level_info returns CS_B200_ERR_ARG past the last level (and for P / R on the
 * coarsest); omega = Jacobi damping of the level.  level_csr copies the operator as 0-based CSR
 * with fp64 values (converted when the cycle runs in fp32); any pointer may be NULL.            */
int cs_b200_level_info(cs_b200_handle* h, int level, int which, int64_t* nrows, int64_t* ncols,
                       int64_t* nnz, double* omega, int* windowed);
int cs_b200_level_csr(cs_b200_handle* h, int level, int which, int32_t* rowptr, int32_t* colidx,
                      double* vals);

/* Connected components of the handle's operator as created: an edge is a stored off-diagonal entry with
 * a non-zero value. label: host, n int32, the 0-based ordinal of each node's component. Components are
 * numbered in order of their smallest node: the order of graph.connected_components and of
 * Graphs.connected_components. Isolated nodes are components of their own. *ncomp may be NULL.
 * Returns CS_B200_ERR_UNSUPPORTED on a handle with grounds applied (cs_b200_set_grounds).
 * Union-find on the device (hooking with path halving, then one prefix sum over the root flags); with
 * the whole-raster handles of cs_b200_create_from_raster[_poly] this says which pairs a solve may
 * take (both nodes in one component) without building the graph on the host.                       */
int cs_b200_components(cs_b200_handle* h, int32_t* label, int64_t* ncomp);

/* n and nnz of the handle's operator. */
int cs_b200_get_dims(const cs_b200_handle* h, int64_t* n, int64_t* nnz);

void cs_b200_destroy(cs_b200_handle* h);

/* Text of the last error on this handle (or of the last failed create if h==NULL). */
const char* cs_b200_last_error(const cs_b200_handle* h);

/* y = A x, `reps` times back to back; *ms_per_rep = mean device time of one SpMV
 * (CUDA events).  x, y: host vectors of n values of the handle's dtype.  Benchmark
 * and parity hook for the headline kernel.                                          */
int cs_b200_spmv(cs_b200_handle* h, const void* x, void* y, int reps, double* ms_per_rep);

/* Y = A X for k in {1,2,4,8} columns through the panel SpMM kernel: x, y host,
 * column-major n x k.  Parity hook for the batched kernel at any size.             */
int cs_b200_spmm(cs_b200_handle* h, int k, const void* x, void* y);

/* Y = A X for a row-major n x k panel resident on the device (k in 1,2,4,8),
 * timing only -- no host traffic.  flush_l2 != 0 writes a >L2 buffer between reps. */
int cs_b200_bench_spmm(cs_b200_handle* h, int k, int reps, int flush_l2, double* ms_per_rep);

/* One fused PCG iteration (SpMM+dot, residual update+dot, direction update) on a
 * device-resident panel of width k, `reps` times; timing only.                      */
int cs_b200_bench_cg_iter(cs_b200_handle* h, int k, int reps, double* ms_per_rep);

/* solve_linear_system(factor, matrix, rhs): A X = B for k right-hand sides.
 * rhs, lhs: host, column-major n x k (Julia Matrix / Vector when k = 1).
 * iters[k], relres[k] (true relative residual ||A x - b|| / ||b||) may be NULL.
 * Returns CS_B200_ERR_RESIDUAL if any column fails the gate (lhs still written).    */
int cs_b200_solve_rhs(cs_b200_handle* h, int64_t k, const void* rhs, void* lhs,
                      double rtol, int64_t itmax, int64_t* iters, double* relres);

/* Batched focal-pair solve, device-resident:
 *   for c in 0..k-1:  A v = e_dst[c] - e_src[c];  v -= v[src[c]];  R[c] = v[dst[c]]
 * src/dst: 0-based rows of this component.  R: k values of dtype.
 * volt: NULL or host column-major n x k (shifted voltages).
 * If accumulate != 0 the node-current vector of every pair (src/out.jl:178-207:
 * max(inflow, outflow) per node with the 1e-8 relative zeroing of src/out.jl:281-287)
 * is added weight[c] times into the handle's cumulative vector and max-ed into its
 * max vector (src/out.jl:100-107); weight == NULL means 1 each.
 * curr: NULL or host column-major n x k of the per-pair node currents.              */
int cs_b200_solve_pairs(cs_b200_handle* h, int64_t k, const int64_t* src, const int64_t* dst,
                        const double* weight, double rtol, int64_t itmax, void* R,
                        void* volt, void* curr, int accumulate, int64_t* iters,
                        double* relres);

/* Pairwise driver by SUPERPOSITION -- the reference's Shortcut (src/core.jl:685-739), extended
 * to voltage / current maps.  All pairs among `np` focal nodes of ONE connected component share
 * the operator and are linear in the right-hand side, so np-1 solves
 *     A u_x = e_{nodes[x]} - e_{nodes[0]} ,  u_x -= u_x[nodes[0]]        (x = 1 .. np-1, u_0 = 0)
 * give every pair:  v(i,j) = u_j - u_i , shifted so that v[src] = 0 , R = v[dst].
 * pi / pj: the k pairs as indices into `nodes` (src = nodes[pi[c]], dst = nodes[pj[c]]).
 * R, volt, curr, accumulate, weight: exactly as cs_b200_solve_pairs.  Each combined voltage is
 * put through the true-residual gate against its own right-hand side (relres[k]); point_iters
 * (np-1 values, may be NULL) are the iterations of the point solves.  Needs np-1 device vectors.  */
int cs_b200_solve_pairs_superposed(cs_b200_handle* h, int64_t np, const int64_t* nodes, int64_t k,
                                   const int64_t* pi, const int64_t* pj, const double* weight,
                                   double rtol, int64_t itmax, void* R, void* volt, void* curr,
                                   int accumulate, int64_t* point_iters, double* relres);

/* Batched solve with SPARSE right-hand sides, device-resident -- the advanced-mode kernel
 * (src/raster/advanced.jl:274-305) for source/ground sets without finite grounds, and
 * the all-to-one loop built on it (src/raster/onetoall.jl:110-118,146-151):
 *   column c:  b = sum_e vals[e] * e_rows[e]   for e in colptr[c] .. colptr[c+1]-1
 *              A v = b ;  v -= v[ref[c]]
 * A Dirichlet ground at ref[c] with the other entries as current sources is expressed on
 * the singular Laplacian by giving ref[c] the entry  -(sum of the sources)  (current
 * conservation), exactly as the pairwise driver does with  -1 / +1 ; duplicates of a row
 * within a column add.  Nothing of size n crosses PCIe unless volt / curr are requested.
 * probe: nprobe rows whose shifted voltages are returned in probe_volt (host, k x nprobe,
 * row-major, dtype); may be NULL / 0.  volt, curr, accumulate, weight: as in solve_pairs.  */
int cs_b200_solve_sources(cs_b200_handle* h, int64_t k, const int64_t* colptr, const int64_t* rows,
                          const double* vals, const int64_t* ref, const double* weight,
                          double rtol, int64_t itmax, int64_t nprobe, const int64_t* probe,
                          void* probe_volt, void* volt, void* curr, int accumulate,
                          int64_t* iters, double* relres);

/* Cumulative / max node-current vectors (n values of dtype each; either may be
 * NULL).  max is initialised to -9999 like src/utils.jl:124.                        */
int cs_b200_read_currents(cs_b200_handle* h, void* cum, void* max);
int cs_b200_reset_currents(cs_b200_handle* h);
/* Device pointers of the same vectors (for an NCCL reduce across ranks).            */
int cs_b200_currents_device_ptrs(cs_b200_handle* h, void** d_cum, void** d_max);

int cs_b200_get_stats(const cs_b200_handle* h, cs_b200_stats* out);

/* The CUDA stream (cudaStream_t) every kernel of this handle is launched on, so a
 * caller can bracket calls with its own CUDA events.                                */
int cs_b200_stream(cs_b200_handle* h, void** stream);

/* Per-launch timing of the dominant kernel.  enable = 1/0 switches event pairs around
 * every SpMM launch on/off (the CUDA-graph path is bypassed while on) and clears the
 * totals; enable < 0 only reads.  *total_ms / *launches: totals since last enable.  */
int cs_b200_profile_spmm(cs_b200_handle* h, int enable, double* total_ms, int64_t* launches);

/* Algorithmic bytes (nnz (s_v+4) + (n+1) 4 + panel passes, DESIGN.md section 4) summed over
 * the launches timed since profiling was last enabled; read BEFORE disabling.          */
int cs_b200_profile_bytes(cs_b200_handle* h, double* algorithmic_bytes);

/* ---- multi-GPU: pair sharding behind the C ABI (SURVEY.md 8e) -----------------------------
 * One process (or thread) per GPU.  The path shards over independent focal pairs against ONE
 * replicated read-only operator -- the axis the reference threads over (src/core.jl:262-272) --
 * so the only collectives are: the broadcast of the matrix from the root, and at the END of a job
 * the gather of the per-pair resistances and the SUM / MAX reduction of the cumulative / max
 * current vectors (src/out.jl:100-107).  NCCL is loaded at run time (dlopen "libnccl.so.2"); the
 * host language only has to move the 128-byte unique id from rank 0 to the other ranks (MPI
 * broadcast, a socket, a file) -- nothing else crosses the host.                              */
typedef struct cs_b200_comm cs_b200_comm;

/* rank 0: fill id128 (128 bytes) with a fresh NCCL unique id                                 */
int cs_b200_comm_unique_id(void* id128);
/* every rank: join the communicator on `device`                                              */
int cs_b200_comm_init(int device, int rank, int nranks, const void* id128, cs_b200_comm** out);
void cs_b200_comm_destroy(cs_b200_comm* c);
const char* cs_b200_comm_last_error(const cs_b200_comm* c);

/* cs_b200_create on every rank from the matrix held by `root` (arguments as cs_b200_create;
 * rowptr / colidx / vals may be NULL on the other ranks, n / nnz / dtype / index_* must agree):
 * the root uploads and narrows the CSR, one ncclBroadcast replicates it (and the root's
 * aggregation seeds), every rank builds its own preconditioner from the device copy.          */
int cs_b200_create_bcast(cs_b200_comm* c, int root, int64_t n, int64_t nnz, const void* rowptr,
                         const void* colidx, const void* vals, int index_bits, int index_base,
                         int dtype, const cs_b200_opts* opts, cs_b200_handle** out);

/* end of job: cum <- SUM over ranks, max <- MAX over ranks, in place in every rank's handle
 * (ncclAllReduce on the handle's solve stream, right behind the last accumulation kernel)     */
int cs_b200_comm_reduce_currents(cs_b200_comm* c, cs_b200_handle* h);

/* end of job: every rank contributes the resistances of its own pairs (global pair indices
 * my_idx[k_mine], values my_R[k_mine], fp64) and receives all k_total of them in R_all
 * (entries no rank contributed stay -1, the reference's "not solved" marker).                 */
int cs_b200_comm_gather_pairs(cs_b200_comm* c, int64_t k_total, const int64_t* my_idx,
                              int64_t k_mine, const double* my_R, double* R_all);

/* max over ranks of a host double (timings) / sum of int64 counters                           */
int cs_b200_comm_max_double(cs_b200_comm* c, double* v, int count);
int cs_b200_comm_barrier(cs_b200_comm* c);

/* The same totals per kernel class (read before disabling): 16 slots, slot = 2 * epilogue + (fp32 ? 1 : 0)
 * with epilogue 0 plain, 1 CG (p.Ap), 2 residual + norms (gate), 3 residual, 4 Jacobi sweep, 5 Jacobi
 * sweep + r.z, 6 prolong-add, 7 fused prolongation + sweep.                                          */
int cs_b200_profile_classes(cs_b200_handle* h, double* ms16, double* bytes16, int64_t* launches16);

/* Library/ABI version: major*1000 + minor.                                          */
int cs_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CS_B200_H */
