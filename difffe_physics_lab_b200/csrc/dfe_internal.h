// Internal definitions shared by the translation units of libdfe_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "dfe.h"

namespace dfe {

void set_error(const char* fmt, ...);

#define DFE_CUDA_OK(expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      ::dfe::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                       __LINE__);                                                      \
      return DFE_ERR_CUDA;                                                             \
    }                                                                                  \
  } while (0)

#define DFE_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::dfe::set_error(__VA_ARGS__);    \
      return DFE_ERR_INVALID;           \
    }                                   \
  } while (0)

// Device-side view of a mesh (plain pointers; passed by value to kernels).
struct MeshDev {
  int dim, npe;
  int n_nodes, n_el, n_dir, n_free;
  int nnz_full, nnz_free, sell_nnz, n_slices;
  const double* nodes;       // (n_nodes, dim)
  const int* elems;          // (n_el, npe)
  const int* adj_ptr;        // (n_nodes+1) node -> adjacent elements, ascending element id
  const int* adj_elem;       // (nadj)
  const int* adj_loc;        // (nadj) local index of the node inside the element
  const int* adj_slot;       // (nadj*npe) index into vals_full of (node, elem[q])
  const int* rowptr;         // (n_nodes+1) full CSR
  const int* col;            // (nnz_full)
  const int* free_nodes;     // (n_free) node id of free row r
  const int* free_rank;      // (n_nodes) rank or -1
  const int* dir_idx;        // (n_dir) dict order
  const double* dir_val;     // (n_dir)
  const int* rowptr_f;       // (n_free+1) K_free CSR
  const int* col_f;          // (nnz_free)
  const int* src_f;          // (nnz_free) index into vals_full
  const int* diag_src;       // (n_free) index into vals_full of the diagonal
  const int* lift_ptr;       // (n_free+1)
  const int* lift_src;       // index into vals_full of K[free row, dirichlet col], dict order
  const double* lift_g;      // Dirichlet value for that entry
  const int* slice_ptr;      // (n_slices+1) SELL-32 offsets (elements)
  const int* sell_col;       // (sell_nnz) column (free numbering); padding points at the row itself
  const int* sell_src;       // (sell_nnz) index into vals_full, -1 for padding
};

// misfit adjoint of the fused 1-D path: gbar = scale * (u - u_data), loss = (scale / 2) * sum (u - u_data)^2
struct Misfit1D {
  double scale;
  double* loss;   // device: [1] (shared kappa: summed over the batch) or [B] (per-sample kappa)
};

// after a fused 1-D launch: if the handle's device fault word is set, overwrite the outputs with NaN and raise the
// host-visible word (one tiny CTA when healthy)
int poison1d_launch(const dfe_mesh* m, double* out, long long ldo, long long B, int nn, double* gk, long long ngk,
                    double* loss, long long nloss, cudaStream_t st);

// banded factor of dfe_band_factor (dfe_batch.cu): the DMMA B-operand fragments of the block TRSM, BAND_FRAGD doubles per
// block row — Ff (forward: H_k, then -S_k) and Bf (backward: H_k^T, then -S_{k+1}^T), both 16-byte aligned
constexpr int BAND_FRAGD = 2048;
void band_frags(const dfe_mesh* m, const void* factor, const double** Ff, const double** Bf);

// pieces of the banded route (dfe_batch.cu) that the per-sample-kappa route (dfe_band_ps.cu) reuses, all asynchronous:
//   band_tables  geom (8 * n_el) and geom2 (4 * n_el) per-element constants of a 2-D P1 mesh (k_band_geom, k_band_tables)
//   band_rhs     X (B, npad) = lifted load of f in free numbering (k_band_rhs_fwd); sample b's matrix at
//                vals_full + b * vstride
//   band_grad    dL/dkappa (per element, or summed per sample) and dL/df (gf may be null) from lambda = X (k_band_grad2,
//                else k_band_grad); DFE_ERR_UNSUPPORTED if neither fits
void band_tables(const dfe_mesh* m, double* geom, double* geom2, cudaStream_t st);
void band_rhs(const dfe_mesh* m, long long B, const double* f, long long ldf, const double* vals_full, long long vstride,
              const double* geom, double* X, cudaStream_t st);
int band_grad(const dfe_mesh* m, long long B, const double* X, const double* u, long long ldu, const double* geom,
              const double* geom2, int gk_per_elem, double* gk, double* gf, long long ldgf, cudaStream_t st);

// pieces of the per-sample-kappa route (dfe_band_ps.cu) that the per-sample heat rollouts (dfe_heat.cu) reuse, asynchronous:
//   band_ps_assemble  vals (B, nnz_full) = K(kappa_b) of every sample (k_bps_assemble); kappa[B] or kappa[B * n_el]
//   band_ps_factor    fac (B, npad * 33) = the banded Cholesky factor of the matrix at vals + b * vstride, sample by
//                     sample, and status[B] (k_bps_bidx into bidx (npad * 33 int32), k_bps_factor)
void band_ps_assemble(const dfe_mesh* m, long long B, const double* kappa, int per_elem, double* vals, cudaStream_t st);
void band_ps_factor(const dfe_mesh* m, long long B, const double* vals, long long vstride, int* bidx, double* fac,
                    int* status, cudaStream_t st);

}  // namespace dfe

struct dfe_mesh {
  dfe_mesh_info info{};
  // ---- host-side symbolic data (int64 copies exposed through the ABI)
  std::vector<int64_t> h_rowptr, h_col, h_rowptr_f, h_col_f, h_free;
  // ---- structured 2-D mesh (topology of FEMesh.rectangle(gx, gy) with every boundary node Dirichlet): quads per side,
  // 0 when the mesh is anything else.  Enables the multigrid-preconditioned solver (dfe_mg_*).
  int grid_nx = 0, grid_ny = 0;
  // element pattern of FEMesh.rectangle(topo_nx, topo_ny) alone (any Dirichlet set): enables the structured assembly kernel
  int topo_nx = 0, topo_ny = 0;
  // rectangle() pattern only: every coordinate difference of every triangle is 0 or in [2^-120, 2^120] and every area in
  // [2^-250, 2^250] — the geometric part of an element-matrix numerator then is 0 or in [2^-293, 2^241], and the structured
  // assembly kernel checks only kappa and the load sum per call before it uses division-free quotients (dfe_exact.cuh)
  bool topo_geo_mid = false;
  // ---- 1-D chain description
  bool chain = false;
  bool bc_left = false, bc_right = false, lift_left_first = true;
  double g_left = 0.0, g_right = 0.0;
  const double* d_hs = nullptr;  // chain: h_e/2 (h_e = x_{e+1}-x_e as the reference computes it), device, n_el
  const double* d_rh = nullptr;  // chain: correctly rounded 1/(h_e/2), device, n_el
  const double* d_X = nullptr;   // chain: X_i = sum_{e<i} h_e/2, device, n_nodes
  double x_total = 0.0;          // chain: X_{n_nodes-1}
  // sticky fault word of the fused 1-D kernels (pinned, device-mapped): a wait that exceeds its bound sets it to 1,
  // every later dfe_solve1d_* call on this handle fails with DFE_ERR_CUDA
  int* h_fault = nullptr;
  int* d_fault = nullptr;
  // device-resident copy of the fault word: the kernels raise THIS one (a read of mapped host memory from a kernel
  // costs ~150 us on B200); the poison kernel that follows every fused launch copies it into the host-visible word
  int* d_fault_dev = nullptr;
  // ---- device
  dfe::MeshDev dev{};
  int n_lift = 0;             // entries of the lifting lists (lift_src / lift_g)
  int n_adj = 0;              // entries of the node -> element adjacency (adj_elem)
  int max_adj = 0;            // most elements around one node
  std::vector<void*> allocs;  // every cudaMalloc owned by the handle
  int sm_count = 0;
};
