/*
 * lcao_b200.h — C ABI of the B200-native LCAONet hot path (liblcao_b200.so, sm_100a).
 *
 * The reference (nmdl-mizo/lcaonet v0.0.3) is pure Python: it has no FFI.  The boundary a maintainer
 * would bind is therefore the set of tensor operations its forward pass delegates to ATen /
 * torch_scatter / torch_sparse; every entry point below names the reference lines it replaces.
 * INTEGRATION.md shows the ctypes stub that binds them from the reference's own modules.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (LCAO_E_*); `lcao_last_error()` returns a
 *     thread-local message.  Nothing throws, nothing allocates device memory, no global state
 *     besides lazily-set kernel attributes: the CALLER owns every buffer (inputs, outputs, scratch).
 *   - all pointers are device pointers unless marked "host"; all calls are asynchronous on
 *     `stream` (a cudaStream_t passed as void*), re-entrant across streams.
 *   - float = IEEE fp32, row-major, innermost dimension contiguous; `ld*` = row stride in elements.
 *   - graph indices: the public edge list is int64 (2,E) like PyG's; every derived index is int32.
 *   - "source" s = edge_index[0] (aggregation centre), "target" t = edge_index[1].
 *   - in-CSR  : edges grouped by TARGET node, inside a node ordered by (source asc, edge id asc)
 *     out-CSR : edges grouped by SOURCE node, inside a node ordered by edge id asc
 */
#ifndef LCAO_B200_H
#define LCAO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCAO_OK 0
#define LCAO_E_ARG (-1)      /* bad argument (null pointer, unsupported size) */
#define LCAO_E_CUDA (-2)     /* CUDA runtime error, see lcao_last_error() */
#define LCAO_E_UNSUPPORTED (-3)

#define LCAO_MAX_UNIQUE_ORB 18
#define LCAO_MAX_POLY 8
#define LCAO_MAX_ORB 64

enum { LCAO_CUT_POLYNOMIAL = 0, LCAO_CUT_ENVELOPE = 1, LCAO_CUT_COSINE = 2 };
enum { LCAO_RBF_HYDROGEN = 0, LCAO_RBF_SPHERICAL_BESSEL = 1 };
/* Activations fused into the kernels: the parameter-free ones `activation_resolver` can return (utils/resolve.py:
 * nn/activation.py ShiftedSoftplus, torch.nn SiLU / Softplus / ReLU / Tanh / Sigmoid / GELU / ELU / LeakyReLU with their
 * default hyper-parameters).  Swish with a trainable beta is not fused (the constructor raises). */
enum {
  LCAO_ACT_NONE = 0, LCAO_ACT_SILU = 1, LCAO_ACT_SSP = 2 /* softplus(x) - ln 2 */, LCAO_ACT_SOFTPLUS = 3,
  LCAO_ACT_RELU = 4, LCAO_ACT_TANH = 5, LCAO_ACT_SIGMOID = 6, LCAO_ACT_GELU = 7 /* erf form */, LCAO_ACT_ELU = 8,
  LCAO_ACT_LEAKY_RELU = 9 /* slope 0.01 */, LCAO_ACT_LAST = 9
};
enum { LCAO_GEMM_FP32 = 0, LCAO_GEMM_TF32X3 = 1, LCAO_GEMM_TF32 = 2 };

/* Radial-basis description (host struct, passed by value to the kernel).
 * orbital o (0 <= o < n_unique*n_rep) uses unique entry o / n_rep  (reference: info.py:124-127). */
typedef struct {
  int32_t n_unique, n_rep, cutoff_kind, rbf_kind;
  double rc, a0;
  int32_t n[LCAO_MAX_UNIQUE_ORB], l[LCAO_MAX_UNIQUE_ORB], deg[LCAO_MAX_UNIQUE_ORB];
  double norm[LCAO_MAX_UNIQUE_ORB];               /* s_nl, rbf.py:92-94 */
  double poly[LCAO_MAX_UNIQUE_ORB][LCAO_MAX_POLY]; /* ascending coefficients of -(n+l)! L_{n-l-1}^{2l+1}, rbf.py:82-87 */
} lcao_basis_spec;

int lcao_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py: gpu_launches) */
int64_t lcao_launch_count(void);
const char* lcao_last_error(void);

/* ---- index construction -------------------------------------------------------------------- */
/* Bucket sort: perm lists item ids grouped by key; ptr has nb+1 entries; scratch: (nb + n) int32
 * (stable=2: nb + n + nb * ceil(n / 1024)).
 * stable=1: inside a bucket items are ordered by (sec asc, id asc) (sec may be NULL) — deterministic,
 *           cost sum_b |b|^2, meant for small buckets (edges per node, atoms per graph).
 * stable=0: grouping only (order inside a bucket unspecified: it depends on the order atomics land in).
 * stable=2: ORDERED grouping for few huge buckets (species / species-pair keys, nb <= 50000): items of a bucket in
 *           ascending id, no dependence on atomic ordering — every keyed reduction that walks perm is reproducible.  Replaces the argsort + CSR
 * machinery of torch_sparse.SparseTensor (reference call site lcaonet.py:462) and the implicit
 * sort inside torch_scatter-by-batch (lcaonet.py:293).  Bit-exact, deterministic. */
int lcao_bucket_sort(const int64_t* keys, const int64_t* sec, int64_t n, int64_t nb, int32_t* ptr,
                     int32_t* perm, int32_t* scratch, int32_t stable, void* stream);

/* Range check of the integer inputs of forward(batch) before they index device memory: *status (one int32, device)
 * receives bit 1 if some z is outside [1, max_z], bit 2 if some batch index is outside [0, n_graph), bit 4 if some
 * edge_index entry is outside [0, N); 0 = all valid.  z / batch may be NULL (skipped).  The reference raises IndexError
 * for such inputs (nn.Embedding / index_select: embed.py:41,91, base.py:38, lcaonet.py:462). */
int lcao_validate_graph(const int64_t* z, int64_t N, int64_t max_z, const int64_t* batch, int64_t n_graph,
                        const int64_t* edge_index, int64_t E, int32_t* status, void* stream);

/* Everything the fused kernels need from edge_index (2,E), in one call:
 *   src32/dst32 (E)            int32 copies of edge_index rows
 *   in_ptr (N+1), in_edge (E)  in-CSR;   in_src (E) = src32[in_edge]
 *   out_ptr (N+1), out_edge (E) out-CSR
 *   tri_ptr (E+1)  exclusive scan of the triplet count per edge, tri_ptr[E] = T
 *                  (T = sum_e indeg(s_e) - [s_e == t_e]; reference lcaonet.py:464-473); may be NULL (skipped:
 *                  only the reference's triplet LISTS need it, see lcao_triplet_offsets)
 * scratch: (2*N + 2*E + 8) int32. */
int lcao_graph_index_build(const int64_t* edge_index, int64_t E, int64_t N, int32_t* src32, int32_t* dst32,
                           int32_t* in_ptr, int32_t* in_edge, int32_t* in_src, int32_t* out_ptr,
                           int32_t* out_edge, int32_t* tri_ptr, int32_t* scratch, void* stream);

/* tri_ptr (E+1) alone, from an existing index; scratch: E + ceil(E / 4096) int32. */
int lcao_triplet_offsets(const int32_t* src32, const int32_t* dst32, const int32_t* in_ptr, int64_t E, int32_t* tri_ptr,
                         int32_t* scratch, void* stream);

/* Materialise the reference's triplet lists (lcaonet.py:468-485) and, if unit != NULL, the triplet
 * cosines (lcaonet.py:431-435): for edge e, for e' in in(s_e) with e' != e:
 *   tri_k = src[e'], e_ks = e', e_st = e, cos = unit[e].unit[e'].   T entries, int64 like the reference. */
int lcao_triplets_fill(const int32_t* src32, const int32_t* in_ptr, const int32_t* in_edge,
                       const int32_t* tri_ptr, int64_t E, int64_t* tri_k, int64_t* e_ks, int64_t* e_st,
                       const float* unit, float* cos_out, void* stream);

/* histogram of small integer keys (pair / species counts for the BatchNorm statistics) */
int lcao_histogram(const int64_t* keys, int64_t n, int64_t nb, float* counts, void* stream);

/* ---- neighbour list under PBC (data/convert.py:103-172 atoms2graphdata; ase.neighborlist.neighbor_list) -------- */
/* Two phases because E is data dependent.  Atoms of one structure are contiguous: graph_ptr (B+1) int32, batch (N)
 * int64 (PyG convention), lattice (B,3,3) rows = cell vectors, pbc (B,3) int32 flags.
 * count[i] = number of (j, image) within `cutoff` of atom i (NOT truncated).  The caller clamps to max_neighbors,
 * marks structures with no neighbour at all as `fallback` (fully linked graph, convert.py:154-157: count = n_atoms-1),
 * and scans into out_ptr (N+1, int64). */
int lcao_neighbor_count(const float* pos, const int64_t* batch, const int32_t* graph_ptr, const float* lattice,
                        const int32_t* pbc, int64_t N, double cutoff, int32_t* count, void* stream);
/* edge_index (2,E) int64 [centre, neighbour] grouped by centre ascending, each centre's neighbours ordered by
 * (distance, neighbour id, image) ascending and truncated to max_neighbors; edge_shift (E,3) = integer image offsets
 * as float32.  status (1 int32, zero-initialised by the caller) is set to 1 if a centre had more than 2048
 * neighbours within the cutoff (not supported). */
int lcao_neighbor_fill(const float* pos, const int64_t* batch, const int32_t* graph_ptr, const float* lattice,
                       const int32_t* pbc, const int32_t* fallback, const int64_t* out_ptr, int64_t N, int64_t E,
                       double cutoff, int32_t max_neighbors, int64_t* edge_index, float* edge_shift, int32_t* status,
                       void* stream);

/* ---- geometry + radial basis (base.py:27-43, rbf.py:92-103,129-142, cutoff.py:32-67) --------- */
/* dist (E), unit (E,3), rb (E,O), optional drb (E,O) = d rb / d r (for autograd forces).  An unknown
 * spec->cutoff_kind or spec->rbf_kind is LCAO_E_ARG. */
int lcao_geom_basis_fwd(const float* pos, const float* shift, const float* lattice, const int64_t* batch,
                        const int32_t* src32, const int32_t* dst32, int64_t E, const lcao_basis_spec* spec_host,
                        float* dist, float* unit, float* rb, float* drb, void* stream);
/* backward of the above w.r.t. positions: given d_dist (E, nullable), d_unit (E,3, nullable),
 * d_rb (E,O, nullable; needs drb) accumulates dvec per edge and reduces it to d_pos (N,3) without
 * atomics (out-CSR for -dvec at s, in-CSR for +dvec at t).  dvec_scratch: (E,3) float. */
int lcao_geom_basis_bwd(const float* dist, const float* unit, const float* drb, const float* d_dist,
                        const float* d_unit, const float* d_rb, int64_t E, int64_t N, int32_t O,
                        const int32_t* in_ptr, const int32_t* in_edge, const int32_t* out_ptr,
                        const int32_t* out_edge, float* dvec_scratch, float* d_pos, void* stream);
/* Cell derivatives of the energy, per graph g, from the dvec (E,3) = d E / d vec that lcao_geom_basis_bwd wrote, with
 * vec_e = pos[t] - pos[s] + shift_e . L_g (row vectors; the rows of L_g = lattice[g] are the cell vectors):
 *   d_lattice[g][i][j] = sum_{e in g} shift_e[i] dvec_e[j]              d E / d L_g          (B,3,3), nullable
 *   virial[g][i][j]    = sum_{e in g} vec_e[i]   dvec_e[j]              d E / d eps_g        (B,3,3), nullable
 * where eps_g is a strain acting as pos' = pos (I + eps), L' = L (I + eps); stress = virial / |det L_g|.  An edge belongs
 * to the graph of its source.  vec is recomputed in FP64 from pos / shift / lattice / batch exactly as the forward forms
 * it; both sums are accumulated in FP64 and rounded once, without atomics (bitwise reproducible): per-chunk partials
 * over the out-edges of LCAO_CELL_CHUNK nodes, then a per-graph sum in chunk order.  Graphs without nodes or edges get
 * zeros.  (seg_ptr (B+1), seg_perm (N, nullable = identity)) lists the nodes of each graph (lcao_bucket_sort of batch);
 * batch (N, nullable = all graph 0) selects the lattice row as in the forward.
 * scratch: (N / LCAO_CELL_CHUNK + B) * 18 doubles.  The gradient w.r.t. edge_shift is not computed. */
#define LCAO_CELL_CHUNK 128
int lcao_geom_cell_bwd(const float* pos, const float* shift, const float* lattice, const int64_t* batch,
                       const int32_t* dst32, const float* dvec, int64_t E, int64_t N, const int32_t* out_ptr,
                       const int32_t* out_edge, const int32_t* seg_ptr, const int32_t* seg_perm, int64_t B,
                       double* scratch, float* d_lattice, float* virial, void* stream);

/* ---- orbital contraction (the einsum "ed,edh->eh" sites lcaonet.py:180-183,200-203) ----------- */
/* B[e,l,:]  = sum_{o: l(o)=l} rb[e,o] * (A[e,o,:] + m[e,o] V[e,o,:])        l = 0..NL-1
 * B[e,NL,:] = sum_o rb[e,o] m[e,o] V[e,o,:]                                  (only if valence)
 * with cst1 (E,O,Cp) = [A | V], Cp = C or 2C; lgrp (O) = l of each orbital; vmask (E,O) 0/1 floats.
 * cst1 and B must be 16-byte aligned: LCAO_E_ARG otherwise. */
int lcao_coeff_contract_fwd(const float* cst1, const float* rb, const float* vmask, const int32_t* lgrp,
                            int64_t E, int32_t O, int32_t C, int32_t NL, int32_t valence, float* B, void* stream);
/* d_cst1 (E,O,Cp) from dB (E,NG,C); d_rb (E,O) written if non-NULL.  dB, d_cst1 and, when d_rb is given, cst1 must
 * be 16-byte aligned: LCAO_E_ARG otherwise. */
int lcao_coeff_contract_bwd(const float* cst1, const float* rb, const float* vmask, const int32_t* lgrp,
                            const float* dB, int64_t E, int32_t O, int32_t C, int32_t NL, int32_t valence,
                            float* d_cst1, float* d_rb, void* stream);

/* ---- orbital contraction against the species-pair table (lcaonet.py:170 f_coeffs + :180-183,:200-203) --- */
/* The coefficient rows cst[e] are a function of the element pair (z_s, z_t) only (embed.py:234-249) and
 * f_coeffs is a bias-free row-wise MLP, so f_coeffs is evaluated on the P-row pair table by the caller and
 *   B[e,l,:]  = sum_{o: l(o)=l} rb[e,o] * (tabA[pair[e],o,:] + m[e,o] tabV[pair[e],o,:])      l = 0..NL-1
 *   B[e,NL,:] = sum_o rb[e,o] m[e,o] tabV[pair[e],o,:]                                        (only if valence)
 * with tab (P,O,Cp) = [A | V].  gram (nullable): (E, NL(NL+1)/2) FP64 upper triangle of B[e,l,:].B[e,l',:]
 * over the first NL groups (consumed by lcao_threebody_*).  psum (nullable): (E, 1 + valence, C) =
 * [sum_{l<NL} B[e,l,:] | B[e,NL,:]] — the only part of B the two-body weight needs; lcao_twobody_fwd/bwd accept it
 * in place of B with NG = 1 + valence, NL = 1 (a third of the bytes).  tab, B and psum must be 16-byte aligned:
 * LCAO_E_ARG otherwise. */
int lcao_pair_contract_fwd(const float* tab, const int64_t* pair, const float* rb, const float* vmask,
                           const int32_t* lgrp, int64_t E, int32_t O, int32_t C, int32_t NL, int32_t valence,
                           float* B, double* gram, float* psum, void* stream);
/* d_tab (P,O,Cp) = keyed reduction of rb[e,o] dB[e,l(o),:] over the edges of each pair, deterministic
 * (two stages, no atomics); (kptr (P+1), kperm (E)) = edges grouped by pair (lcao_bucket_sort).
 * d_rb (E,O) written if non-NULL (autograd forces); d_tab may be NULL when only d_rb is wanted (the positions-only
 * pass of autograd forces).  scratch: lcao_pair_contract_bwd_scratch() BYTES.  dB, d_tab, scratch and, when d_rb is
 * given, tab must be 16-byte aligned: LCAO_E_ARG otherwise (every argument is checked before the first launch). */
int lcao_pair_contract_bwd(const float* tab, const int64_t* pair, const int32_t* kptr, const int32_t* kperm,
                           const float* rb, const float* vmask, const int32_t* lgrp, const float* dB, int64_t E,
                           int64_t P, int32_t O, int32_t C, int32_t NL, int32_t valence, float* d_tab, float* d_rb,
                           void* scratch, void* stream);
int64_t lcao_pair_contract_bwd_scratch(int64_t E, int64_t P, int32_t O, int32_t C, int32_t valence);
/* Gram matrices of an existing B (E,NG,C): gram (E, NL(NL+1)/2) FP64, for callers that built B themselves. */
int lcao_coeff_gram(const float* B, int32_t NG, int64_t E, int32_t C, int32_t NL, double* gram, void* stream);

/* ---- embedding block: count-weighted BatchNorm over table rows (embed.py:175,194,232,249) -------- */
/* nn.BatchNorm1d over a batch given as its R DISTINCT rows x (R,F) and their multiplicities counts (R) (the node rows
 * depend on the species, the coefficient rows on the species pair: DESIGN.md R6).  training != 0: batch statistics
 * (biased variance), running_mean / running_var (nullable together) updated with `momentum` and the unbiased variance,
 * *num_batches_tracked (nullable) incremented; training == 0: the running statistics normalise.  gamma / beta nullable
 * (affine=False).  save_mean / save_rstd (F) are kept for the backward pass. */
int lcao_table_norm_fwd(const float* x, const float* counts, const float* gamma, const float* beta, int64_t R, int32_t F,
                        float eps, float momentum, int32_t training, float* running_mean, float* running_var,
                        int64_t* num_batches_tracked, float* y, float* save_mean, float* save_rstd, void* stream);
/* dx (R,F), dgamma (F), dbeta (F) (the last two nullable) of the above; dy is the gradient w.r.t. every table row. */
int lcao_table_norm_bwd(const float* dy, const float* x, const float* counts, const float* gamma, const float* save_mean,
                        const float* save_rstd, int64_t R, int32_t F, int32_t training, float* dx, float* dgamma,
                        float* dbeta, void* stream);

/* Species-pair coefficient table before its BatchNorm (embed.py:234-249 evaluated on the (Zd x Zd) pair table):
 * pre[s,t,o,k] = fe[t,o,k] * (1 + za[s,k] + zb[t,k]);  fe (Zd,O,K), za / zb (Zd,K), pre (Zd,Zd,O,K); K % 4 == 0. */
int lcao_pair_outer_fwd(const float* fe, const float* za, const float* zb, int32_t Zd, int32_t O, int32_t K, float* pre,
                        void* stream);
/* gradients of the above (fixed-order sums: deterministic): d_fe (Zd,O,K), d_za (Zd,K), d_zb (Zd,K) */
int lcao_pair_outer_bwd(const float* dpre, const float* fe, const float* za, const float* zb, int32_t Zd, int32_t O,
                        int32_t K, float* d_fe, float* d_za, float* d_zb, void* stream);

/* ---- three-body message passing (lcaonet.py:173-189, shbf.py:75-87) --------------------------- */
/* gate[n,:] = sigmoid(xk[n,:]) per node (lcaonet.py:186-188), computed once per layer */
int lcao_sigmoid_rows(const float* x, int64_t ldx, float* out, int64_t ldo, int64_t M, int32_t C, void* stream);
/* tbw[e,:] = sum_{e' in in(s_e), e' != e} normalize( sum_l Y_l(unit[e].unit[e']) B[e',l,:] ) * gate[src[e'],:]
 * B has NG groups per edge (row stride NG*C); gram = its per-edge Gram matrices (|v|^2 = Y^T G Y);
 * gate (N,C) with row stride ldg.  B, gate and tbw (and d_tbw, dP, dB and q for the backward) must be 16-byte aligned:
 * LCAO_E_ARG otherwise. */
int lcao_threebody_fwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate,
                       int64_t ldg, const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src,
                       const int32_t* out_ptr, const int32_t* out_edge, int64_t N, int64_t E, int32_t C,
                       int32_t NL, float* tbw, void* stream);
/* backward: dB (E,NG,C) groups 0..NL-1 are OVERWRITTEN with the three-body contribution, including the
 * part that flows through the norms (gram is treated as a function of B); group NL is zeroed when
 * NG > NL.  q (E,C) = per in-edge gradient of the gate PRE-activation xk (the sigmoid derivative is
 * applied here): d_xk[k] = sum_{e' in out(k)} q[e'].  d_unit_ks / d_unit_st (E,3; both or neither):
 * gradient w.r.t. unit[e] from its role as in-edge (k->s) and as out-edge (s->t); d_unit = their sum
 * (autograd forces).  dP (nullable): the COMPACT two-body gradient of lcao_twobody_bwd (E, 1 + valence, C);
 * when given, dB = three-body part + dP[e,0,:] for every l < NL and dB[e,NL,:] = dP[e,1,:], i.e. the sum
 * autograd would otherwise form with a separate (E,NG,C) pass. */
int lcao_threebody_bwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate,
                       int64_t ldg, const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src,
                       const int32_t* out_ptr, const int32_t* out_edge, int64_t N, int64_t E, int32_t C,
                       int32_t NL, const float* d_tbw, const float* dP, float* dB, float* q, float* d_unit_ks,
                       float* d_unit_st, void* stream);

/* ---- two-body weight (lcaonet.py:192-204) ----------------------------------------------------- */
/* p = (1+g[:, :C]) * PA + (1+g[:, C:]) * PV ;  lw = p / max(|p|, 1e-12)
 * PA = sum_l B[e,l,:] - B[e,NL,:],  PV = B[e,NL,:] (valence) ;  PA = sum_l B[e,l,:] otherwise. */
int lcao_twobody_fwd(const float* B, int32_t NG, const float* g, int64_t E, int32_t C, int32_t NL,
                     int32_t valence, float* lw, void* stream);
/* compact = 0: dB is (E,NG,C) (the same row repeated for every l < NL, then the valence slot);
 * compact = 1: dB is (E, 1 + valence, C): [row shared by all l < NL | valence slot]. */
int lcao_twobody_bwd(const float* B, int32_t NG, const float* g, const float* d_lw, int64_t E, int32_t C,
                     int32_t NL, int32_t valence, int32_t compact, float* dB, float* d_g, void* stream);

/* ---- edge <- node gathers and node <- edge segment sums (torch_scatter sites lcaonet.py:208,293,307;
 *      ATen index sites lcaonet.py:209) --------------------------------------------------------- */
/* out[e,:] = act(a[src[e],:] + b[dst[e],:] + bias) ; pre[e,:] (nullable) = value before act */
int lcao_edge_pair_fwd(const float* a, int64_t lda, const float* b, int64_t ldb, const float* bias,
                       const int32_t* src32, const int32_t* dst32, int64_t E, int32_t C, int32_t act,
                       float* out, float* pre, void* stream);
/* out[r,:] = sum_{j in [ptr[r],ptr[r+1])} x[perm[j],:] * (y ? y[perm[j],:] : 1) * scale_r
 * `mean` is a flag word: bit 0: scale_r = 1/max(count,1) instead of 1; bit 1: y holds a pre-activation and the
 * factor is act(y) (the message sum then needs no stored copy of h = act(pre_h)); bit 2: the factor is act'(y)
 * (backward through an activation folded into the reduction that follows it); bits 4-7: the activation (LCAO_ACT_*,
 * 0 = SiLU).  Deterministic, no atomics.  x may be NULL when no segment
 * has any item (edge-less batch): out is zero-filled. */
int lcao_segment_sum(const float* x, int64_t ldx, const float* y, int64_t ldy, const int32_t* ptr,
                     const int32_t* perm, int64_t R, int32_t C, int32_t mean, float* out, int64_t ldo, void* stream);
/* backward of the message sum  agg[s] = sum_{e in out(s)} bw[e] * h[e],  h = act(pre_h)  (lcaonet.py:207-214):
 *   d_bw[e,:] = d_agg[src[e],:] * h[e,:] ;  d_pre_h[e,:] = d_agg[src[e],:] * bw[e,:] * act'(pre_h[e,:])
 * h may be NULL: it is then recomputed from pre_h. */
int lcao_msg_bwd(const float* d_agg, int64_t lda, const int32_t* src32, const float* h, const float* bw,
                 const float* pre_h, int64_t E, int32_t C, int32_t act, float* d_bw, float* d_pre_h, void* stream);
/* out[i,:] = table[idx[i],:] * (mul ? mul[i,:] : 1)   (idx int64 or int32 chosen by idx_is64) */
int lcao_gather_rows(const float* table, int64_t ldt, const void* idx, int32_t idx_is64, const float* mul, int64_t ldm,
                     int64_t n, int32_t W, float* out, int64_t ldo, void* stream);
/* acc[key[i],:] += x[i,:]   (keys int64, few distinct values: pair / species tables; acc pre-zeroed) */
int lcao_reduce_by_key(const float* x, int64_t ldx, const int32_t* kptr, const int32_t* kperm, int64_t nkeys,
                       int64_t n, int32_t W, float* acc, void* stream);

/* ---- dense layers (nn/base.py:11-81 = nn.Linear; sites listed in SURVEY.md §8 a-7) ------------- */
/* Y = act(X W^T + bias); X (M,K) ldx, W (Nout,K) contiguous, Y (M,Nout) ldy; pre (nullable) gets X W^T + bias.
 * The tcgen05 kernels split W into shared memory while the previous kernel of the stream may still run (programmatic
 * dependent launch), so W must not be written by this library's immediately preceding launch on the same stream (a
 * layer's weight is a parameter: no kernel of the pass writes it). */
int lcao_linear_fwd(const float* X, int64_t ldx, const float* W, const float* bias, float* Y, int64_t ldy,
                    float* pre, int64_t ldp, int64_t M, int32_t K, int32_t Nout, int32_t act, int32_t mode,
                    void* stream);
/* dX = (dY * act'(H)) W   (accumulate=1: dX += ...).  H (M,Nout) = the layer's pre-activation, or NULL /
 * act = NONE for a plain dY.  dY * act'(H) is first formed in `scratch` (lcao_linear_bwd_scratch() floats: M*Nout;
 * may be NULL when act == NONE).  W must not be written by this library's
 * immediately preceding launch on the same stream (see lcao_linear_fwd); nor for lcao_linear_dgrad_act. */
int lcao_linear_dgrad(const float* dY, int64_t ldy, const float* H, int64_t ldh, int32_t act, const float* W, float* dX,
                      int64_t ldx, int64_t M, int32_t K, int32_t Nout, int32_t accumulate, int32_t mode, float* scratch,
                      void* stream);
/* dX = (dY W) * act'(G): lcao_linear_dgrad of a layer whose INPUT is act(G), G (M,K) ldg being that activation's
 * pre-activation (nn.Sequential(Dense, act, Dense) chains: lcaonet.py:108-113,122-127,254-269).  Fuses the
 * lcao_act_bwd pass that would otherwise follow into the GEMM epilogue. */
int lcao_linear_dgrad_act(const float* dY, int64_t ldy, const float* W, const float* G, int64_t ldg, int32_t act,
                          float* dX, int64_t ldx, int64_t M, int32_t K, int32_t Nout, int32_t mode, void* stream);
/* dW (Nout,K) += (dY * act'(H))^T X ; db (Nout) += its column sums (db nullable).  dW/db zeroed by the caller. */
int lcao_linear_wgrad(const float* dY, int64_t ldy, const float* H, int64_t ldh, int32_t act, const float* X, int64_t ldx,
                      float* dW, float* db, int64_t M, int32_t K, int32_t Nout, int32_t mode, float* scratch, void* stream);
/* lcao_linear_wgrad (act = none) with its second stage — the deterministic sum of the per-CTA partial tiles into dW / db
 * — DEFERRED to lcao_wgrad_reduce_batch: a training step needs its weight gradients only at the optimizer, so the ~30
 * small reduction launches of a backward pass become one.  desc: HOST buffer of 6 int64 per 128-column pass
 * (ceil(Nout / 128) passes); *n_desc: descriptors written (0: the shape took the CUDA-core kernel and dW is final).
 * scratch: lcao_linear_bwd_scratch(...) floats PER PASS; it must stay untouched until the batch reduction has run. */
int lcao_linear_wgrad_deferred(const float* dY, int64_t ldy, const float* X, int64_t ldx, float* dW, float* db, int64_t M,
                               int32_t K, int32_t Nout, int32_t mode, float* scratch, int64_t* desc, int32_t* n_desc,
                               void* stream);
/* dW / db += the partial tiles of n deferred weight gradients (descriptors from lcao_linear_wgrad_deferred, HOST memory) */
int lcao_wgrad_reduce_batch(const int64_t* desc, int32_t n, void* stream);
/* number of floats of `scratch` the two calls above need for these arguments (0 when the act' factor is fused
 * into the tcgen05 prologue).  Pass X = NULL / dX = NULL for the call that will not be made. */
int64_t lcao_linear_bwd_scratch(const float* dY, int64_t ldy, const float* H, int64_t ldh, int32_t act, const float* W,
                                const float* X, int64_t ldx, const float* dX, int64_t lddx, int64_t M, int32_t K,
                                int32_t Nout, int32_t mode);
/* dH = dY * act'(H)  elementwise over (M,C) with row strides (in place allowed: dH == dY); any alignment and width */
int lcao_act_bwd(const float* dY, int64_t ldy, const float* H, int64_t ldh, float* dH, int64_t ldd, int64_t M,
                 int32_t C, int32_t act, void* stream);
/* Y = act(X) elementwise over (M,C) with row strides (in place allowed).  lcao_linear_fwd's tcgen05 epilogue fuses
 * SiLU; the other LCAO_ACT_* kinds run as this pass over the GEMM's output. */
int lcao_act_fwd(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t M, int32_t C, int32_t act, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LCAO_B200_H */
