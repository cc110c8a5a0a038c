/*
 * dfe.h — C ABI of libdfe_b200.so: the B200 (sm_100a) differentiable P1-FEM Poisson hot path.
 *
 * This is the drop-in boundary for the ONE path of danieleschmidt/DiffFE-Physics-Lab that this
 * repository accelerates: DifferentiableFESolver.forward and its autograd backward
 * (reference diffhe/solver.py:49-183).  The reference has no FFI of its own (it is pure Python);
 * each entry point below names the reference code region it replaces.  INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types; every function returns a dfe_status
 *     (0 = ok) and never throws; dfe_last_error() returns a thread-local message.
 *   - all arithmetic is IEEE float64; indices crossing the ABI are int64 (host side) — the
 *     library keeps int32 copies on the device.
 *   - pointers named *_host are host memory; all others are DEVICE memory on the device the
 *     mesh was created for, owned by the caller (torch).  Work is enqueued on `stream`
 *     (a cudaStream_t passed as void*); nothing synchronises unless stated.
 *   - a dfe_mesh is immutable after creation; concurrent calls on different streams are
 *     safe when each call has its own workspace.
 *   - there is NO CPU compute path: compute entry points fail with DFE_ERR_CUDA without a GPU.
 */
#ifndef DFE_H_
#define DFE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFE_ABI_VERSION 1

typedef enum dfe_status {
  DFE_OK = 0,
  DFE_ERR_INVALID = 1,       /* bad argument (shape, index out of range, null pointer)      */
  DFE_ERR_CUDA = 2,          /* CUDA runtime error, or no device                             */
  DFE_ERR_UNSUPPORTED = 3,   /* valid input outside what this build implements               */
  DFE_ERR_NOT_CONVERGED = 4, /* PCG hit maxit before the recursive residual reached tol      */
  DFE_ERR_BREAKDOWN = 5,     /* PCG breakdown: p^T A p <= 0 or non-finite (K_free not SPD,    */
                             /* e.g. no Dirichlet node — the reference returns garbage there) */
  DFE_ERR_WORKSPACE = 6      /* workspace too small                                          */
} dfe_status;

/* kappa layouts (SURVEY §8b).  The reference accepts only SCALAR (solver.py:32-43). */
typedef enum dfe_kappa_mode {
  DFE_KAPPA_SCALAR = 0,          /* kappa[1]            one value shared by every sample/element */
  DFE_KAPPA_PER_SAMPLE = 1,      /* kappa[B]            one value per sample (1-D batched path)   */
  DFE_KAPPA_PER_ELEMENT = 2,     /* kappa[n_el]         field shared by every sample              */
  DFE_KAPPA_PER_SAMPLE_ELEMENT = 3 /* kappa[B*n_el]     row-major (B, n_el)                       */
} dfe_kappa_mode;

typedef struct dfe_mesh dfe_mesh;

typedef struct dfe_mesh_info {
  int32_t dim;          /* 1 or 2                                              */
  int32_t device;       /* CUDA device ordinal, or -1 for a host-only handle   */
  int64_t n_nodes, n_elements, n_dirichlet, n_free;
  int64_t nnz_full;     /* structural nnz of K      (all nodes)                */
  int64_t nnz_free;     /* structural nnz of K_free (free rows/cols)           */
  int64_t sell_nnz;     /* padded length of the SELL-32 copy of K_free         */
  int32_t max_row_nnz;  /* widest row of K_free                                */
  int32_t chain1d;      /* 1: elements are (e,e+1) and Dirichlet ⊆ {first,last} — fused 1-D path usable */
} dfe_mesh_info;

const char* dfe_last_error(void);
int dfe_abi_version(void);
/* number of CUDA devices visible to the library (0 on a CPU-only host; never fails) */
int dfe_device_count(void);

/* ---------------------------------------------------------------- mesh (reference diffhe/mesh.py:14-52,127-129)
 * Replaces: the FEMesh container as consumed by solver.py:82-85,112-117,160-171.
 * nodes_host   (n_nodes, dim) row-major f64      = FEMesh.nodes
 * elems_host   (n_el, dim+1) row-major int64     = FEMesh.elements
 * dir_idx_host/dir_val_host (n_dir)              = FEMesh.dirichlet_nodes items IN DICT ORDER
 * device >= 0: build symbolic data on the host and upload to that device; device == -1: host-only
 * handle (pattern queries work, compute calls return DFE_ERR_CUDA) — used by CPU tests.
 * Builds: int32 connectivity, free map / rank (free_nodes(), mesh.py:127-129), the structural CSR
 * pattern of K and K_free (rows and columns ascending; {(p,q): some element holds p and q} — the
 * positions solver.py:89-92,137-140 write), node->element adjacency in ascending element order
 * (the reference's accumulation order), Dirichlet lifting lists in dict order (solver.py:166-169),
 * and a SELL-32 layout of K_free for SpMV.
 */
int dfe_mesh_create(int dim, int64_t n_nodes, int64_t n_el, const double* nodes_host,
                    const int64_t* elems_host, int64_t n_dir, const int64_t* dir_idx_host,
                    const double* dir_val_host, int device, dfe_mesh** out);
/* Same, with an explicit number of nodes per element: dim + 1 (P1, what dfe_mesh_create passes) or (dim + 1)(dim + 2) / 2
 * (P2: 1-D [left, right, mid], 2-D [v0, v1, v2, m01, m12, m20]; geometry is read from the vertices).  P2 elements are an
 * item of the reference's roadmap (reference README.md:139-143), not of its code: there is no upstream arithmetic to match,
 * the load is F = M f with the consistent mass matrix, and the mesh takes the general CSR + PCG route only (the fused 1-D,
 * banded, shared-memory-batch and multigrid routes report "unsupported"). */
int dfe_mesh_create_p(int dim, int nodes_per_element, int64_t n_nodes, int64_t n_el, const double* nodes_host,
                      const int64_t* elems_host, int64_t n_dir, const int64_t* dir_idx_host,
                      const double* dir_val_host, int device, dfe_mesh** out);
void dfe_mesh_destroy(dfe_mesh* m);
int dfe_mesh_get_info(const dfe_mesh* m, dfe_mesh_info* info);
/* Host copies of the patterns (int64, owned by the handle).  which = 0: K (n_nodes rows),
 * which = 1: K_free (n_free rows, columns renumbered by rank in free_nodes()). */
int dfe_mesh_csr_host(const dfe_mesh* m, int which, const int64_t** rowptr, const int64_t** col,
                      int64_t* n_rows, int64_t* nnz);
/* free_nodes() (mesh.py:127-129), ascending, int64, owned by the handle. */
int dfe_mesh_free_nodes_host(const dfe_mesh* m, const int64_t** free_nodes, int64_t* n_free);

/* ---------------------------------------------------------------- fused 1-D path (chain meshes)
 * Replaces solver.py:73-98 (_solve_1d) + :153-183 (_apply_bc_and_solve) for B independent samples
 * on one mesh, and their autograd backward (LinalgSolveExBackward0 + the CopySlices chain).
 * One persistent kernel per call: per-sample HBM traffic is read f + write u (forward),
 * read gbar + read u (+ write gf) (backward).  K is never materialised.
 *   f, u, gbar, gf : (B, n_nodes) f64 with row strides ld* (elements)
 *   kappa          : SCALAR -> [1], PER_SAMPLE -> [B], PER_ELEMENT -> [n_el], PER_SAMPLE_ELEMENT -> (B, n_el)
 *                    (the per-element layouts run with one Neumann sweep only, i.e. up to 2e5 nodes)
 *   n_refine       : Neumann/refinement sweeps after the structured solve (1 meets 1e-12 up to
 *                    ~2e5 nodes; pass 2 beyond; <0 selects automatically)
 *   gkappa         : PER_SAMPLE -> [B];  SCALAR -> [1] (sum over the batch, fixed order);
 *                    PER_ELEMENT -> [n_el] (sum over the batch);  PER_SAMPLE_ELEMENT -> (B, n_el)
 *   gf may be NULL (f does not require grad).
 * Workspace: dfe_solve1d_workspace_bytes(m, B) bytes of device memory, contents undefined.
 *
 * dfe_solve1d_supported   1 if the fused path takes this mesh in BOTH directions for (kappa_mode, n_refine); the
 *                         host layer asks once, in forward, and routes the call to the general path otherwise.
 * dfe_solve1d_bwd_misfit  the adjoint of a data-misfit loss in ONE pass (BASELINE config 5, reference
 *                         examples/poisson_1d_demo.py:104-110: loss = mean((u - u_data)^2); loss.backward()):
 *                         reads u_data and u, forms gbar = scale * (u - u_data) on the fly (Dirichlet entries dropped),
 *                         and returns  loss = (scale / 2) * sum_i (u_i - u_data_i)^2  next to dL/dkappa —
 *                         SCALAR: gkappa[1], loss[1] summed over the batch (pass adjacent words of one buffer and
 *                         all-reduce it); PER_SAMPLE: gkappa[B], loss[B].  Pipelined kernel only (chain mesh up to
 *                         163840 nodes, 16-byte aligned rows), else DFE_ERR_UNSUPPORTED.
 * dfe_mesh_fault          sticky fault word of the handle (0 = healthy): set when a wait inside a fused 1-D kernel
 *                         exceeded its bound; the outputs of that call are overwritten with NaN and every later
 *                         dfe_solve1d_* call on the handle fails.  Read it after synchronising the stream.
 */
size_t dfe_solve1d_workspace_bytes(const dfe_mesh* m, int64_t B);
int dfe_solve1d_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* kappa,
                    int kappa_mode, int n_refine, double* u, int64_t ldu, void* ws, size_t ws_bytes,
                    void* stream);
int dfe_solve1d_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u,
                    int64_t ldu, const double* kappa, int kappa_mode, int n_refine, double* gf,
                    int64_t ldgf, double* gkappa, void* ws, size_t ws_bytes, void* stream);
int dfe_solve1d_bwd_misfit(const dfe_mesh* m, int64_t B, const double* u_data, int64_t ldd, const double* u,
                           int64_t ldu, const double* kappa, int kappa_mode, int n_refine, double scale, double* gf,
                           int64_t ldgf, double* gkappa, double* loss, void* ws, size_t ws_bytes, void* stream);
int dfe_solve1d_supported(const dfe_mesh* m, int kappa_mode, int n_refine);
int dfe_mesh_fault(const dfe_mesh* m);

/* ---------------------------------------------------------------- general path (2-D triangles, and 1-D meshes that are not chains)
 * dfe_assemble   replaces solver.py:82-96 / :112-145: K on the structural CSR of all nodes and F,
 *                accumulated per row in ascending element order without atomics — values are
 *                bit-identical to the reference's dense K at pattern positions.
 *                kappa_mode SCALAR or PER_ELEMENT.  vals_full[nnz_full], F[n_nodes].
 * dfe_eliminate  replaces solver.py:162-171: F_free = F[free] - K[free,D] g (dict order),
 *                K_free = K[free][:,free] (CSR order into vals_free if non-NULL, and SELL-32 into
 *                sell_vals if non-NULL), dinv = 1/diag(K_free).
 * dfe_pcg        replaces solver.py:174 (torch.linalg.solve) and, called on gbar_free, the adjoint
 *                solve of LinalgSolveExBackward0 (K symmetric): Jacobi-PCG in one cooperative
 *                kernel, deterministic dot products, stops when the recursive ||r||/||rhs|| <= tol.
 *                Synchronises the stream before returning and reports iterations / residual through
 *                iters_host / relres_host (may be NULL).  Returns DFE_ERR_NOT_CONVERGED / _BREAKDOWN.
 * dfe_scatter    replaces solver.py:177-181: u = 0; u[d] = g (or 0 when zero_bc); u[free] = x.
 * dfe_gather_free v_free = v[free]   (gbar -> gbar_free; Dirichlet entries dropped, SURVEY A7)
 * dfe_grad       replaces autograd of solver.py:88-96,139-145,169 (SURVEY A8): lam_full is lambda
 *                scattered with zeros on Dirichlet nodes, u the full solution.
 *                gkappa: SCALAR -> [1], PER_ELEMENT -> [n_el];  gf[n_nodes] or NULL.
 *                ws: dfe_grad_workspace_bytes(m) bytes.
 */
int dfe_assemble(const dfe_mesh* m, const double* kappa, int kappa_mode, const double* f,
                 double* vals_full, double* F, void* stream);
int dfe_eliminate(const dfe_mesh* m, const double* vals_full, const double* F, double* vals_free,
                  double* sell_vals, double* F_free, double* dinv, void* stream);
size_t dfe_pcg_workspace_bytes(const dfe_mesh* m);
int dfe_pcg(const dfe_mesh* m, const double* sell_vals, const double* dinv, const double* rhs,
            double* x, double tol, int64_t maxit, int64_t* iters_host, double* relres_host, void* ws,
            size_t ws_bytes, void* stream);
int dfe_scatter(const dfe_mesh* m, const double* x_free, int zero_bc, double* u, void* stream);
int dfe_gather_free(const dfe_mesh* m, const double* v_full, double* v_free, void* stream);
size_t dfe_grad_workspace_bytes(const dfe_mesh* m);
int dfe_grad(const dfe_mesh* m, const double* lam_full, const double* u, const double* kappa,
             int kappa_mode, double* gkappa, double* gf, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- structured 2-D meshes: multigrid-preconditioned CG
 * For meshes with the topology of FEMesh.rectangle() (reference mesh.py:79-121: node id = row*(nx+1)+col, triangles
 * [a,b,d], [b,c,d] per quad, every boundary node Dirichlet) K_free is numerically a 5-point operator on the grid of
 * interior nodes, and Jacobi-PCG (dfe_pcg) needs O(nx) iterations (7435 at 1024 x 1024 with a 1e3 contrast).  These
 * entry points replace solver.py:174 / the adjoint solve by CG preconditioned with a V(nu, nu) multigrid cycle
 * (damped Jacobi, operator-dependent interpolation, Galerkin coarse operators): ~50 iterations, same stopping rule.
 *   dfe_mg_supported   1 if the mesh has that structure (and >= 1024 unknowns)
 *   dfe_mg_setup       vals_full from dfe_assemble -> hierarchy (dfe_mg_hierarchy_bytes(m) bytes of device memory;
 *                      keep it for the adjoint solve).  Synchronises the stream.  DFE_ERR_UNSUPPORTED if the assembled
 *                      matrix is not numerically 5-point (node coordinates moved off the grid): use dfe_pcg.
 *   dfe_mg_pcg         like dfe_pcg (rhs / x on the free numbering, recursive ||r|| <= tol ||rhs||, synchronises,
 *                      DFE_ERR_NOT_CONVERGED / _BREAKDOWN); nu = smoothing sweeps before and after each coarse-grid
 *                      correction (1..4; 2 is the default of the host layer); ws: dfe_mg_workspace_bytes(m) bytes.
 */
int dfe_mg_supported(const dfe_mesh* m);
size_t dfe_mg_hierarchy_bytes(const dfe_mesh* m);
size_t dfe_mg_workspace_bytes(const dfe_mesh* m);
int dfe_mg_setup(const dfe_mesh* m, const double* vals_full, void* hier, size_t hier_bytes, void* stream);
int dfe_mg_pcg(const dfe_mesh* m, const void* hier, const double* rhs, double* x, double tol, int64_t maxit, int nu,
               int64_t* iters_host, double* relres_host, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- batched small systems sharing one matrix
 * (BASELINE config 5b: many forcing samples, shared kappa, small 2-D mesh).  Replaces, for every sample b of the
 * batch, solver.py:143-145 (load), :165-169 (lifting), :174 (solve), :177-181 (scatter) and their autograd
 * backward — the per-sample sequence dfe_assemble/dfe_eliminate/dfe_pcg/dfe_scatter/dfe_grad above, which is
 * latency-bound for meshes of ~1e3 unknowns.  ONE CTA owns a sample: K_free (SELL-32, from dfe_eliminate) and the
 * search direction live in shared memory, Jacobi-PCG to the recursive tolerance, fixed-order reductions.
 *   dfe_batch_supported  1 if the mesh fits (n_free <= 2048 and matrix + vectors <= 200 KB of shared memory)
 *   dfe_batch_fwd        f, u: (B, n_nodes) with row strides ldf / ldu; vals_full: K on the full pattern
 *                        (dfe_assemble, any f), sell_vals / dinv from dfe_eliminate
 *   dfe_batch_bwd        gbar, u, gf: (B, n_nodes); gkappa: SCALAR -> (B) per-sample sums (the caller adds them up
 *                        for the shared parameter), PER_ELEMENT -> (B, n_el); gf may be NULL
 *   iters / relres / status: device arrays of length B (status 0 ok, 4 not converged, 5 breakdown); the calls are
 *                        asynchronous on `stream`.
 */
int dfe_batch_supported(const dfe_mesh* m);
int dfe_batch_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* vals_full,
                  const double* sell_vals, const double* dinv, double* u, int64_t ldu, double tol, int64_t maxit,
                  int32_t* iters, double* relres, int32_t* status, void* stream);
int dfe_batch_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                  const double* sell_vals, const double* dinv, int kappa_mode, double* gf, int64_t ldgf,
                  double* gkappa, double tol, int64_t maxit, int32_t* iters, double* relres, int32_t* status,
                  void* stream);

/* ---------------------------------------------------------------- the same batch, banded direct solver
 * When the half bandwidth of K_free is <= 32 (dfe_band_supported; e.g. FEMesh.rectangle(nx, ny) with nx <= 32 in the
 * reference's node numbering) the shared matrix is factored ONCE per call, K_free = L L^T, and every sample costs two
 * banded triangular solves (a warp owns 16 samples) — ~13x fewer flops than Jacobi-PCG at 961 unknowns and no
 * reductions.  This is the closest replacement of solver.py:174 (dense LU) for config 5b.
 *   dfe_band_factor   vals_full from dfe_assemble; factor: dfe_band_factor_bytes(m) bytes of device memory;
 *                     status_dev (optional, device int32): 0 ok, 5 = pivot <= 0 (K_free not SPD)
 *   dfe_band_fwd/bwd  like dfe_batch_fwd/bwd with `factor` instead of the SELL matrix;
 *                     ws: dfe_band_workspace_bytes(m, B) bytes.  All calls are asynchronous on `stream`.
 *                     Row strides ldf / ldu / ldg / ldgf are >= n_nodes (else DFE_ERR_INVALID); the rows of f, u, gbar
 *                     and gf need only the 8-byte alignment of a double (odd strides and offsets are fine).
 *   dfe_band_npad     leading dimension of a block of right-hand sides in free numbering (n_free rounded up to 32)
 *   dfe_band_solve    X <- A_free^{-1} X for B right-hand sides, X (B, npad) row-major in FREE numbering (row r of a sample
 *                     = free node dfe_mesh_free_nodes_host()[r]; entries r >= n_free must be 0 and stay 0), in place, with
 *                     a factor from dfe_band_factor.  `vals_full` given to dfe_band_factor may be ANY symmetric positive
 *                     definite matrix on the pattern of K (e.g. M + dt K): this is the operator-reuse entry point for
 *                     time stepping (reference README.md:139-143 roadmap: heat equation; examples/heat_2d.py).  Block TRSM
 *                     on the FP64 tensor cores (mma.sync m8n8k4.f64).
 */
int dfe_band_supported(const dfe_mesh* m);
size_t dfe_band_factor_bytes(const dfe_mesh* m);
size_t dfe_band_workspace_bytes(const dfe_mesh* m, int64_t B);
int dfe_band_factor(const dfe_mesh* m, const double* vals_full, void* factor, int32_t* status_dev, void* stream);
int dfe_band_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* vals_full,
                 const void* factor, double* u, int64_t ldu, void* ws, size_t ws_bytes, void* stream);
int dfe_band_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                 const void* factor, int kappa_mode, double* gf, int64_t ldgf, double* gkappa, void* ws,
                 size_t ws_bytes, void* stream);
int64_t dfe_band_npad(const dfe_mesh* m);
int dfe_band_solve(const dfe_mesh* m, int64_t B, double* X, const void* factor, void* stream);

/* ---------------------------------------------------------------- banded direct solver, one matrix per sample
 * The same banded solve when every sample has its own conductivity: kappa[B] (DFE_KAPPA_PER_SAMPLE) or kappa[B * n_el]
 * row-major (DFE_KAPPA_PER_SAMPLE_ELEMENT); any other mode gives DFE_ERR_INVALID.  Per sample: assembly of K(kappa_b)
 * (bit-identical to dfe_assemble in the matching SCALAR / PER_ELEMENT mode), blocked banded Cholesky of K_free(kappa_b)
 * (bit-identical to dfe_band_factor on that matrix), the lifted load, and two banded triangular solves.
 *   dfe_band_ps_supported        1 for a 2-D P1 mesh with dfe_band_supported (the gradient kernels then fit)
 *   dfe_band_ps_factor_bytes     (12 * n_el + B * npad * 33) * 8 bytes, npad = dfe_band_npad(m); 262 KB per sample at
 *                                FEMesh.rectangle(32, 32) (npad 992), about 1.07 GB at B = 4096.  Layout, in doubles:
 *                                  geom[8 * n_el] | geom2[4 * n_el]   per-element constants of the load / gradient kernels
 *                                  then per sample b: invd[npad] | Lr[npad * 32]   (invd[i] = 1 / L_ii,
 *                                  Lr[i * 32 + d - 1] = L[i][i - d]: the first npad * 33 doubles of a dfe_band_factor buffer)
 *   dfe_band_ps_workspace_bytes  ws of both calls: B * (nnz_full + npad) doubles + npad * 33 int32
 *   dfe_band_ps_fwd   fills `factors` and u (B, ldu); status[B] (device int32): 0 ok, 5 = a pivot failed the SPD test
 *                     (pivot <= 1e-12 x its diagonal entry: K_free(kappa_b) is not SPD), sample by sample
 *   dfe_band_ps_bwd   lambda_b = K_free(kappa_b)^{-1} gbar_b[free] with the factors of dfe_band_ps_fwd, then
 *                     gkappa (same layout as kappa: -lambda_b^T K0_e u_b, per element or summed per sample) and
 *                     gf = dL/df (B, ldgf; may be NULL)
 *   Row strides ldf / ldu / ldg / ldgf are >= n_nodes (else DFE_ERR_INVALID); rows need only 8-byte alignment.  Both
 *   calls are asynchronous on `stream`.
 */
int dfe_band_ps_supported(const dfe_mesh* m);
size_t dfe_band_ps_factor_bytes(const dfe_mesh* m, int64_t B);
size_t dfe_band_ps_workspace_bytes(const dfe_mesh* m, int64_t B);
int dfe_band_ps_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* kappa, int kappa_mode,
                    void* factors, double* u, int64_t ldu, int32_t* status, void* ws, size_t ws_bytes, void* stream);
int dfe_band_ps_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                    const void* factors, int kappa_mode, double* gf, int64_t ldgf, double* gkappa,
                    void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- differentiable heat-equation rollouts
 * Backward Euler with the lumped mass, (M_L + dt K) u^{n+1} = M_L u^n + dt F, Dirichlet nodes held at the mesh's values,
 * for B states sharing one factor of A = M_L + dt K (dfe_band_factor), and its discrete adjoint.  In free numbering,
 *   forward   A_ff x_{n+1} = m * x_n + c                     m = M_L[free], c = dt F_free - (A g)_free
 *   adjoint   A_ff lambda_n = gbar_n + m * lambda_{n+1}        lambda_{N+1} = 0
 *   dL/du0[free] = m * lambda_1,   dL/dkappa_e = -dt sum_n sum_b lam~_n^T K0_e u_n,   dL/df = W^T (dt sum_n sum_b lam~_n)
 * (lam~: lambda with zeros on the Dirichlet nodes; W: the load operator, dfe_grad's gf).  Each rollout call is ONE launch
 * of a block-TRSM kernel (FP64 tensor cores) with the time loop inside; results do not depend on `warps`.
 *   dfe_heat_supported   1 for 2-D P1 meshes with dfe_band_supported and a gradient kernel that fits shared memory
 *   dfe_heat_warps       warps per CTA (16 states each) the rollout kernels choose for B states (0 if unsupported)
 *   dfe_heat_fwd         n_steps steps.  u0 (B, .) node layout with row stride ldu0, or NULL: X already holds x_0.
 *                        X (B, npad) free-layout carry (dfe_band_npad), holds x_{n_steps} on return; the state after step
 *                        j (0-based) is written to traj + b * ld_b + j * ld_t in node layout, Dirichlet values included.
 *                        m_free / c_free: (npad), zero beyond n_free.
 *   dfe_heat_adj         steps n0 + n_steps down to n0 + 1.  X (B, npad) carries lambda_{n+1} in and lambda_{n0+1} out
 *                        (zero it before step N); gbar (B, R, n_nodes)-like with strides ldg_b / ldg_t holds dL/du_n for
 *                        n % g_every == 0 at slot n / g_every - 1 (NULL: no loss term in this range); lam (n_steps, B, npad)
 *                        receives lambda_{n0+1+j} at slot j; lam_sum (B, npad) += lambda_n in step order.
 *   dfe_heat_grad        per-step partial sums of lam~^T K0_e u for steps n0+1 .. n0+n_seg (u: state of step n0+1+j of
 *                        sample b at u + b * ld_b + j * ld_t; lam as written by dfe_heat_adj) into ws, which holds
 *                        dfe_heat_grad_bytes(m, B, n_total) bytes for the whole rollout of n_total steps.
 *   dfe_heat_grad_sum    dL/dkappa from the partials of all n_total steps, added in a fixed step order (independent of how
 *                        the rollout was split): PER_ELEMENT -> gkappa[n_el], SCALAR -> gkappa[1].
 *   fault (device int32): set to 1 if a bounded wait inside a rollout kernel expired; the outputs are then invalid.
 * X, m_free, c_free, lam and lam_sum must be 16-byte aligned.  All calls are asynchronous on `stream`.
 */
int dfe_heat_supported(const dfe_mesh* m);
int dfe_heat_warps(const dfe_mesh* m, int64_t B);
size_t dfe_heat_grad_bytes(const dfe_mesh* m, int64_t B, int64_t n_total);
int dfe_heat_fwd(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0, const void* factor,
                 const double* m_free, const double* c_free, double* X, double* traj, int64_t ld_b, int64_t ld_t,
                 int warps, int32_t* fault, void* stream);
int dfe_heat_adj(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_steps, const double* gbar, int64_t ldg_b,
                 int64_t ldg_t, int64_t g_every, const void* factor, const double* m_free, double* X, double* lam,
                 double* lam_sum, int warps, int32_t* fault, void* stream);
int dfe_heat_grad(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_seg, int64_t n_total, const double* u, int64_t ld_b,
                  int64_t ld_t, const double* lam, void* ws, size_t ws_bytes, void* stream);
int dfe_heat_grad_sum(const dfe_mesh* m, int64_t B, int64_t n_total, double dt, int kappa_mode, double* gkappa, void* ws,
                      size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- heat-equation rollouts, one conductivity per sample
 * The rollouts above when every sample has its own conductivity: kappa[B] (DFE_KAPPA_PER_SAMPLE) or kappa[B * n_el]
 * row-major (DFE_KAPPA_PER_SAMPLE_ELEMENT); any other mode gives DFE_ERR_INVALID.  Per sample b, in free numbering,
 *   A_b = M_L + dt K(kappa_b),   c_b = dt F_free - (A_b g)_free
 *   forward   A_b,ff x_{n+1} = m * x_n + c_b ;   adjoint   A_b,ff lambda_n = gbar_n + m * lambda_{n+1}
 *   dL/dkappa_{b,e} = -dt sum_n lam~_{n,b}^T K0_e u_{n,b}   (PER_SAMPLE: summed over e in a fixed order)
 * One warp per sample runs both banded sweeps of its own factor (no tensor cores: there is no shared B operand).
 * Meshes: dfe_band_ps_supported (else DFE_ERR_UNSUPPORTED).
 *   dfe_heat_ps_factor_bytes     (10 * n_el + B * npad * 33) * 8 bytes, npad = dfe_band_npad(m): 262 KB per sample at
 *                                FEMesh.rectangle(32, 32), about 1.07 GB at B = 4096.  Layout, in doubles:
 *                                  K0[6 * n_el] | element node / free-rank table[4 * n_el]   (per-element gradient tables)
 *                                  then per sample b: invd[npad] | Lr[npad * 32]   (the layout of dfe_band_ps_factor_bytes)
 *   dfe_heat_ps_workspace_bytes  ws of dfe_heat_ps_setup: B * nnz_full doubles (A_b on the pattern of K, left there on
 *                                return) + npad * 33 int32
 *   dfe_heat_ps_setup   mass / load (n_nodes): the lumped mass and the load vector F of the source (load may be NULL: no
 *                       source), shared by the batch.  Assembles and factors every A_b (bit-identical to dfe_assemble,
 *                       dt * K + mass on the diagonal with two roundings, and dfe_band_factor), fills `factors` (16-byte
 *                       aligned) and c_free (B, npad), zero beyond n_free; status[B] (device int32): 0 ok, 5 = A_b not SPD.
 *   dfe_heat_ps_fwd     as dfe_heat_fwd, with the factors and c_free (B, npad) of dfe_heat_ps_setup; m_free (npad).
 *   dfe_heat_ps_adj     as dfe_heat_adj, with the factors of dfe_heat_ps_setup.
 *   dfe_heat_ps_grad    gacc (B, n_el) += lam~_n^T K0_e u_n for the steps of one segment (u and lam as for dfe_heat_grad),
 *                       added one step at a time from the last step down: call it for the segments in descending order
 *                       on a zeroed gacc and the sums are bit-identical however the rollout was split, and independent of B.
 *   dfe_heat_ps_grad_sum  gkappa = -dt gacc: (B, n_el) for PER_SAMPLE_ELEMENT, (B) summed per sample for PER_SAMPLE.
 * Offsets into the factors, trajectory and lambda buffers are 64-bit.  The kernels never wait on each other's warps (no
 * fault word).  All calls are asynchronous on `stream`.
 */
size_t dfe_heat_ps_factor_bytes(const dfe_mesh* m, int64_t B);
size_t dfe_heat_ps_workspace_bytes(const dfe_mesh* m, int64_t B);
int dfe_heat_ps_setup(const dfe_mesh* m, int64_t B, const double* kappa, int kappa_mode, double dt, const double* mass,
                      const double* load, void* factors, double* c_free, int32_t* status, void* ws, size_t ws_bytes,
                      void* stream);
int dfe_heat_ps_fwd(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0, const void* factors,
                    const double* m_free, const double* c_free, double* X, double* traj, int64_t ld_b, int64_t ld_t,
                    void* stream);
int dfe_heat_ps_adj(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_steps, const double* gbar, int64_t ldg_b,
                    int64_t ldg_t, int64_t g_every, const void* factors, const double* m_free, double* X, double* lam,
                    double* lam_sum, void* stream);
int dfe_heat_ps_grad(const dfe_mesh* m, int64_t B, int64_t n_seg, const void* factors, const double* u, int64_t ld_b,
                     int64_t ld_t, const double* lam, double* gacc, void* stream);
int dfe_heat_ps_grad_sum(const dfe_mesh* m, int64_t B, double dt, int kappa_mode, const double* gacc, double* gkappa,
                         void* stream);

/* ---------------------------------------------------------------- heat-equation rollouts with sources in time and per sample
 * The rollouts above with a constant term per step and per sample.  Step j of a launch (u^n -> u^{n+1}) for sample b, in
 * free numbering:
 *   A_ff x_{n+1} = m * x_n + c_{j,b},   c_{j,b} = fl(c_base_b + fl(dt * F_free(q_{j,b})))
 * F_free: the reference's load vector (per element fl(fl(area / 3) * fl(((q_i + q_j) + q_k) / 3)), added in ascending
 * element order: the bits of dfe_assemble's F).  c_base is the route's constant without this source (c_free of
 * _HeatOperator / dfe_heat_ps_setup, or a per-sample c_b formed by dfe_heat_src_load itself).  Meshes: dfe_band_ps_supported,
 * and the element terms plus four input rows in 200 KB of shared memory (else DFE_ERR_UNSUPPORTED).
 *   dfe_heat_src_workspace_bytes  ws of the two source kernels: 48 bytes per element (their per-element tables, rebuilt by
 *                                 every call)
 *   dfe_heat_src_load   c (n_steps, nb, npad), zero beyond n_free: row (j, b) from q at q + j * ldq_t + b * ldq_b (node
 *                       layout, n_nodes) and c_base + b * ldbase (npad; ldbase 0: one base for every row).  c may equal
 *                       c_base when n_steps = 1 and ldbase = npad (in place).
 *   dfe_heat_fwd_src    dfe_heat_fwd, with step j of sample b reading c at c + j * ldc_t + b * ldc_b (npad; strides even
 *                       and >= 0, c 16-byte aligned).  ldc_b = 0: one row for the batch; ldc_t = 0: constant in time.
 *   dfe_heat_ps_fwd_src dfe_heat_ps_fwd, with c read as for dfe_heat_fwd_src.
 *   dfe_heat_src_grad   g row (j, b) at g + j * ldg_t + b * ldg_b (node layout, n_nodes) = W^T (dt * lam~), lam~ the row at
 *                       lam + j * ldl_t + b * ldl_b (free layout, npad) scattered with zeros on the Dirichlet nodes:
 *                       g_p = sum_{e∋p} area_e / 9 * ((l_i + l_j) + l_k), l = dt * lam~ (dfe_grad's gf).  With lam slot
 *                       j of dfe_heat_adj (lambda_{n0+1+j}) this is dL/dq at step n0 + j; with lam_sum it is dL/df_b of a
 *                       per-sample constant source.  Non-zero on Dirichlet nodes in general.
 * The Dirichlet and source-free behaviour is that of the calls above.  Offsets are 64-bit.  All calls are asynchronous on
 * `stream`; a host-only handle gives DFE_ERR_CUDA and a null handle DFE_ERR_INVALID.
 */
size_t dfe_heat_src_workspace_bytes(const dfe_mesh* m);
int dfe_heat_src_load(const dfe_mesh* m, int64_t n_steps, int64_t nb, double dt, const double* q, int64_t ldq_t,
                      int64_t ldq_b, const double* c_base, int64_t ldbase, double* c, void* ws, size_t ws_bytes,
                      void* stream);
int dfe_heat_fwd_src(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0, const void* factor,
                     const double* m_free, const double* c, int64_t ldc_t, int64_t ldc_b, double* X, double* traj,
                     int64_t ld_b, int64_t ld_t, int warps, int32_t* fault, void* stream);
int dfe_heat_ps_fwd_src(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0, const void* factors,
                        const double* m_free, const double* c, int64_t ldc_t, int64_t ldc_b, double* X, double* traj,
                        int64_t ld_b, int64_t ld_t, void* stream);
int dfe_heat_src_grad(const dfe_mesh* m, int64_t n_steps, int64_t nb, double dt, const double* lam, int64_t ldl_t,
                      int64_t ldl_b, double* g, int64_t ldg_t, int64_t ldg_b, void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DFE_H_ */
