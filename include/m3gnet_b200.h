/*
 * m3gnet_b200.h — C ABI of the B200 (sm_100a) energy+forces hot path of M3GNet.
 *
 * The reference (lan496/torch-m3gnet) is 100 % Python: it has no FFI/plugin layer to mirror, so this
 * header *defines* the boundary a maintainer would bind (ctypes stub in INTEGRATION.md).  Each entry
 * point names the reference code it replaces (paths relative to /root/reference/src/torch_m3gnet/).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; buffers are caller-owned
 *     (torch caching allocator); no entry point allocates, frees or synchronises;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = success, otherwise a negative M3G_ERR_* code; m3g_last_error() gives the
 *     message of the last failure on the calling thread;
 *   - floating tensors are float32 row-major; index tensors are int32 unless noted (the int64
 *     tensors of the reference API are narrowed once per batch by m3g_narrow_i64);
 *   - edges are grouped by source atom (ascending), `edge_ptr` (N+1) is that CSR;
 *     `in_ptr`/`in_perm` is the CSR of edge ids grouped by destination atom (ascending edge id
 *     inside a row); triplets are a CSR per bond: `tri_ptr` (E+1) rows = first bond e1,
 *     `tri_e2` (T) columns = second bond; `trt_ptr`/`trt_e1` is its transpose (rows = e2);
 *   - sizes: N atoms, E directed edges, T triplets, B structures, F feature width (node == edge),
 *     R = n_max radial functions, L = l_max, D = L*R.
 *   - accumulation order (stated, deterministic): every segmented sum is evaluated by one warp
 *     (or sub-warp group of G lanes): lane g adds elements g, g+G, g+2G, ... of the segment in
 *     ascending order, then lanes are combined by a butterfly (xor 16,8,4,2,1).  No float atomics
 *     on the default path.
 */
#ifndef M3GNET_B200_H
#define M3GNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define M3G_OK 0
#define M3G_ERR_INVALID (-1) /* bad argument (null pointer, unsupported size) */
#define M3G_ERR_CUDA (-2)    /* a CUDA runtime call / launch failed */
#define M3G_ERR_UNSUPPORTED (-3)

#define M3G_MAX_F 128 /* feature width supported by the kernels */
#define M3G_MAX_L 9   /* l_max supported by the kernels = the reference's range (nn/interaction.py:250-253) */
#define M3G_MAX_R 10  /* n_max supported by the three-body kernels = the reference's range */
#define M3G_MAX_RADIAL 10 /* n_max supported by the radial (edge) basis */

const char* m3g_last_error(void);
int m3g_abi_version(void);
/* Device properties the host side sizes grids with: out[0]=SM count, out[1]=cc major, out[2]=cc minor */
int m3g_device_info(int* out_host);

/* ---------------------------------------------------------------------------------------------
 * Graph preparation (once per batch; replaces nothing in the reference — it is the canonical
 * form the reference's `from_structure` output already has, data/material_graph.py:182-187,239-248)
 * ------------------------------------------------------------------------------------------- */
int m3g_narrow_i64(const int64_t* in, int32_t* out, int64_t n, void* stream);
/* flags[0] = 1 if keys is non-decreasing, flags[1] = 1 if every key is in [0, n_rows) */
int m3g_check_sorted(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* flags, void* stream);
/* row_ptr[r] = first position whose key >= r (keys sorted); row_ptr has n_rows+1 entries */
int m3g_csr_from_sorted(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* row_ptr, void* stream);
/* Stable counting sort of positions 0..n-1 by key: row_ptr (n_rows+1), perm (n) with ascending
 * positions inside each row.  `work` must hold n_rows+1 + m3g_scan_work_elems(n_rows) int32. */
int m3g_csr_by_key(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* row_ptr, int32_t* perm,
                   int32_t* work, void* stream);
/* out[p] = vals[perm[p]] */
int m3g_gather_i32(const int32_t* vals, const int32_t* perm, int64_t n, int32_t* out, void* stream);
/* every row of (row_ptr, cols) is sorted ascending in place (rows are short: one neighbour shell) */
int m3g_sort_rows(const int32_t* row_ptr, int64_t n_rows, int32_t* cols, void* stream);
/* flags[0] = 1 iff (ptr_a, col_a) == transpose(ptr_a, col_a), i.e. (e1,e2) occurs as often as (e2,e1); rows sorted */
int m3g_csr_is_symmetric(const int32_t* row_ptr, const int32_t* cols, int64_t n_rows, int32_t* flags,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * Graph construction on the GPU (replaces data/material_graph.py:168-193 [pymatgen
 * Structure.get_all_neighbors] and :196-254 [compute_threebody]).  Batched over B structures.
 *   lattice (B,3,3) f64 rows = lattice vectors, cart (N,3) f64, atom_ptr (B+1) int32.
 * Two-pass: count → caller allocates → fill.  Accept rule d^2 < r^2 + 1e-8 in float64, zero-length
 * self pairs dropped; images are relative to the unwrapped input coordinates; edges of atom i are
 * ordered by (j, s0, s1, s2) ascending.
 * ------------------------------------------------------------------------------------------- */
/* Optional cell list: bins (B,3) int32 = bins per lattice axis of each structure (0,0,0 = sweep the whole structure;
 * otherwise every axis needs >= 3 bins whose perpendicular width is >= cutoff), bin_base (B+1) = offset of each
 * structure's bins.  m3g_nbr_bin_count writes atom_bin (N) and adds to bin_count (zeroed by the caller); after an
 * exclusive scan into bin_ptr, m3g_nbr_bin_fill lists the atoms of every bin (bin_cursor zeroed by the caller).
 * The bins only restrict the candidate atoms: accept test, edge set and edge order are unchanged.  Pass
 * bins = NULL to m3g_nbr_count / m3g_nbr_fill for the plain sweep. */
int m3g_nbr_bin_count(const double* lattice, const double* cart, const int32_t* atom_ptr, int64_t B, int64_t N,
                      double cutoff, const int32_t* bins, const int32_t* bin_base, int32_t* atom_bin,
                      int32_t* bin_count, void* stream);
int m3g_nbr_bin_fill(const int32_t* atom_bin, const int32_t* bin_ptr, int64_t N, int32_t* bin_cursor,
                     int32_t* bin_atoms, void* stream);
int m3g_nbr_count(const double* lattice, const double* cart, const int32_t* atom_ptr, int64_t B, int64_t N,
                  double cutoff, const int32_t* bins, const int32_t* bin_base, const int32_t* bin_ptr,
                  const int32_t* bin_atoms, int32_t* edge_count /* (N) */, void* stream);
int m3g_exclusive_scan_i32(const int32_t* in, int32_t* out /* n+1 */, int64_t n, int32_t* work, void* stream);
int64_t m3g_scan_work_elems(int64_t n);
int m3g_nbr_fill(const double* lattice, const double* cart, const int32_t* atom_ptr, int64_t B, int64_t N,
                 double cutoff, double threebody_cutoff, const int32_t* bins, const int32_t* bin_base,
                 const int32_t* bin_ptr, const int32_t* bin_atoms, const int32_t* edge_ptr /* (N+1) */, int64_t E,
                 int64_t* edge_index /* (2,E) */, int32_t* edge_shift /* (E,3) */, float* edge_dist /* (E) */,
                 int32_t* member /* (E) 1 if float32(d) <= float32(r3) */, void* stream);

/* Verlet (skin) list for MD / relaxation loops (SURVEY.md 8(f) rank 2; the reference rebuilds the pymatgen neighbour
 * list for every structure it sees, data/material_graph.py:168-193).  The candidate list is an ordinary neighbour
 * list built once with cutoff + skin (m3g_nbr_count / m3g_nbr_fill): cand_ptr (N+1), cand_j (C) int32, cand_shift
 * (C,3).  m3g_verlet_displacement writes max_i |cart_i - ref_i|^2 (f32, rounded up; +inf for NaN input) so the host
 * rebuilds the candidates once it exceeds (skin/2)^2.  While it does not, m3g_verlet_count / m3g_verlet_fill give
 * exactly the output of m3g_nbr_count / m3g_nbr_fill on the new coordinates (same float64 accept test on the
 * candidates, same (j, s0, s1, s2) order).  The lattice must be the one the candidates were built with. */
int m3g_verlet_displacement(const double* cart, const double* ref_cart, int64_t N, float* max_d2 /* (1) */,
                            void* stream);
int m3g_verlet_count(const double* lattice, const double* cart, const int32_t* atom_ptr, int64_t B, int64_t N,
                     double cutoff, const int32_t* cand_ptr, const int32_t* cand_j, const int32_t* cand_shift,
                     int32_t* edge_count /* (N) */, void* stream);
int m3g_verlet_fill(const double* lattice, const double* cart, const int32_t* atom_ptr, int64_t B, int64_t N,
                    double cutoff, double threebody_cutoff, const int32_t* cand_ptr, const int32_t* cand_j,
                    const int32_t* cand_shift, const int32_t* edge_ptr, int64_t E, int64_t* edge_index /* (2,E) */,
                    int32_t* edge_shift /* (E,3) */, float* edge_dist /* (E) */, int32_t* member /* (E) */,
                    void* stream);
/* per-atom member degree n3 -> num_triplet_i (N) int64 = n3(n3-1), num_triplet_ij (E) int32,
 * tri_count (E) = triplets whose first bond is e (n3-1 for member edges else 0), and member_list (E):
 * the member edges of atom i compacted (ascending) at positions edge_ptr[i]..
 * Optional (NULL to skip): used_count (N) = bonds of atom i that head a triplet (n3 if n3 >= 2 else 0) and
 * stats int64[3], zeroed by the caller: += T, max n3, += sum of used_count — one read-back sizes tri_e2,
 * the per-atom kernels' capacity and the member-bond list */
int m3g_triplet_count(const int32_t* edge_ptr, const int32_t* member, int64_t N, int64_t E,
                      int64_t* num_triplet_i, int32_t* num_triplet_ij, int32_t* tri_count, int32_t* member_list,
                      int32_t* used_count, int64_t* stats, void* stream);
/* tri_ptr = exclusive scan of tri_count.  Fills tri_e2 (T) int32 CSR columns and, if triplet_index != NULL,
 * the reference's (2,T) int64 list in the reference's order (atom, e1, e2).  Optional: member_edges = ascending
 * list of the bonds that head a triplet, written at used_ptr (N+1) = exclusive scan of used_count */
int m3g_triplet_fill(const int32_t* edge_ptr, const int32_t* tri_ptr, const int32_t* tri_count,
                     const int32_t* member_list, int64_t N, int64_t T, int32_t* tri_e2, int64_t* triplet_index,
                     const int32_t* used_ptr, int32_t* member_edges, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Geometry + bases
 * ------------------------------------------------------------------------------------------- */
/* nn/scale.py:24-29 — out = in / length_scale (true division) */
int m3g_scale_fwd(const float* in, float* out, int64_t n, float length_scale, void* stream);
/* nn/invariant.py:44-59 — vec4[e] = (pos[dst]+shift·lattice[batch[src]]-pos[src], |v|), dist[e] = |v| */
int m3g_geometry_fwd(const float* pos, const float* lattice, const int32_t* batch, const int32_t* src,
                     const int32_t* dst, const int32_t* shift, int64_t E, float* vec4, float* dist, void* stream);
/* nn/invariant.py:33-40 — cos[t] = clamp(v1·v2/(r1 r2), -1, 1) in the caller's triplet order (int64 list) */
int m3g_angles_fwd(const float* vec4, const int64_t* tri_index /* (2,T) */, int64_t T, float* cos_out, void* stream);
/* adjoint of m3g_angles_fwd: adds into g_vec4 (E,4) with float atomics (rare path: only when a caller
 * differentiates through `triplet_angles`) */
int m3g_angles_bwd(const float* vec4, const int64_t* tri_index, const float* g_cos, int64_t T, float* g_vec4,
                   void* stream);
/* adjoint of m3g_geometry_fwd w.r.t. pos: g_e = g_vec4.xyz + (g_vec4.w + g_dist)·v/r;
 * g_pos[i] = scale * (sum_{e in in(i)} g_e - sum_{e in out(i)} g_e).  g_dist may be NULL. */
int m3g_geometry_bwd(const float* vec4, const float* g_vec4, const float* g_dist, const int32_t* edge_ptr,
                     const int32_t* in_ptr, const int32_t* in_perm, int64_t N, float scale, float* g_pos,
                     void* stream);
/* nn/featurizer.py:81-100 — h (E,R).  consts: [k_0..k_R | coeff_0..coeff_{R-1} | a_0..a_{R-1} | b_0..b_{R-1}]
 * with k_m = (m+1)·pi/rc, a_m = sqrt(e_m/d_{m-1}), b_m = sqrt(d_m), all produced on the host by the
 * reference's float32 op sequence. */
int m3g_radial_fwd(const float* dist, const float* consts, int64_t E, int R, float* h, void* stream);
int m3g_radial_bwd(const float* dist, const float* consts, const float* g_h, int64_t E, int R, float* g_dist,
                   void* stream);
/* nn/atom_ref.py:25-29 and nn/featurizer.py:33-38 (one-hot · Linear == column gather of W (F,num_types)) */
int m3g_atomref_fwd(const float* table, const int32_t* types, int64_t N, float* out, void* stream);
int m3g_embed_fwd(const float* weight /* (F,num_types) */, const int32_t* types, int64_t N, int F, int num_types,
                  float* x, void* stream);
/* nn/featurizer.py:128-132 — e0 = SiLU(h · Wt), Wt (R,F) = weight^T */
int m3g_edge_adjust_fwd(const float* h, const float* Wt, int64_t E, int R, int F, float* e0, void* stream);
int m3g_edge_adjust_bwd(const float* h, const float* Wt, const float* g_e0, int64_t E, int R, int F, float* g_h,
                        void* stream);

/* nn/interaction.py:284-350 (SphericalBessel fwd + its custom derivative), :353-382 (LegendreCosPolynomial
 * fwd / bwd with the reference's grad_output-per-level rule), :389-400 (cutoff_function) — elementwise,
 * kept for the operator API (`spherical_bessel`, `legendre_cos`, `cutoff_function`).  dout may be NULL. */
int m3g_sph_bessel(const float* x, int order, int64_t n, float* out, float* dout, void* stream);
int m3g_legendre(const float* x, int order, int64_t n, float* out, void* stream);
int m3g_legendre_bwd(const float* x, const float* go, int order, int64_t n, float* gx, void* stream);
int m3g_cutoff(const float* r, float rc, int64_t n, float* out, float* dout, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ThreeBodyInteration (nn/interaction.py:187-223) — D = L*R, d = l*R + n
 * tb_consts: [zeros_ln (D) | factors_ln (D) | rc | r3]  (2*D + 2 floats; chi = j_l(z r / rc) / factors)
 * ------------------------------------------------------------------------------------------- */
/* sig (N,D) = sigmoid(x · Ws^T + bs), Ws (D,F) = linear_sigmoid1.weight */
int m3g_tb_sigma_fwd(const float* x, const float* Ws, const float* bs, int64_t N, int F, int D, float* sig,
                     void* stream);
/* per edge: bas[e][d] = chi_d(r_e)·fc(r_e)·sig[dst[e]][d]   (chi uses rc, fc uses r3; quirk Q5) */
int m3g_tb_edge_basis_fwd(const float* vec4, const int32_t* dst, const float* sig, const float* tb_consts,
                          int64_t E, int L, int R, const int32_t* edge_list, int64_t n_list, float* bas, void* stream);
/* red[e1][d] = fc(r_e1)·sum_{e2 in tri(e1)} Y_l(cos(e1,e2))·bas[e2][d];
 * e_out = e_in + SiLU(red·WdT) * sigmoid(red·WgT), WdT/WgT (D,F) */
int m3g_tb_reduce_fwd(const float* vec4, const float* bas, const int32_t* tri_ptr, const int32_t* tri_e2,
                      const float* tb_consts, const float* WdT, const float* WgT, const float* e_in, int64_t E,
                      int L, int R, int F, int group, float* red, float* e_out, void* stream);
/* g_red (E,D) from g_e (E,F): adjoint of the bias-free 1-layer GatedMLP (forward recomputed from red); rows
 * of bonds without triplets (tri_ptr[e+1] == tri_ptr[e]) are zero */
int m3g_tb_gate_bwd(const float* red, const float* g_e, const float* WdT, const float* WgT, const int32_t* tri_ptr,
                    int64_t E, int D, int F, float* g_red, void* stream);
/* gather-form adjoint of the triplet sum (uses tri CSR for "e as first bond" and its transpose for
 * "e as second bond"; they may alias when the list is symmetric).  Outputs: g_vec4 (E,4) (xyz from
 * cos, w from cos and fc(r_e1)), g_bas (E,D).  Legendre backward follows the reference (quirk Q3). */
int m3g_tb_reduce_bwd(const float* vec4, const float* bas, const float* g_red, const int32_t* tri_ptr,
                      const int32_t* tri_e2, const int32_t* trt_ptr, const int32_t* trt_e1, const float* tb_consts,
                      int64_t E, int L, int R, int group, float* g_vec4, float* g_bas, void* stream);
/* adjoint of m3g_tb_edge_basis_fwd: g_vec4[e].w += d/dr terms; g_sig_e (E,D) per-edge sigma gradient.
 * edge_list (optional, both directions): only the n_list listed bonds (the member bonds of the triplet list) are
 * evaluated — bas rows of other bonds are never read by the reduce kernels; for the adjoint the caller zero-fills
 * g_sig_e, whose unlisted rows stay zero. */
int m3g_tb_edge_basis_bwd(const float* vec4, const int32_t* dst, const float* sig, const float* g_bas,
                          const float* tb_consts, int64_t E, int L, int R, const int32_t* edge_list, int64_t n_list,
                          float* g_vec4, float* g_sig_e, void* stream);
/* g_x (N,F) = base (N,F or NULL) + (sum_{e in in(k)} g_sig_e[e]) * sig(1-sig) · Ws, Ws (D,F) */
int m3g_tb_sigma_bwd(const float* g_sig_e, const int32_t* in_ptr, const int32_t* in_perm, const float* sig,
                     const float* Ws, const float* base, int64_t N, int F, int D, float* g_x, void* stream);

/* Canonical triplet layout (what compute_threebody, data/material_graph.py:239-248, emits): for every atom the
 * rows of its member bonds (bonds with a non-empty triplet row) list exactly all other member bonds of that atom,
 * ascending.  m3g_tri_dense_check: flags[0] = 1 if the CSR has that layout, flags[1] = max members per atom.
 * m3g_tb_atom_fwd / _bwd (csrc/threebody_atom.cu; replaces nn/interaction.py:187-223 and its autograd; l_max = n_max =
 * 3, F = 64, members per atom <=
 * m3g_tb_atom_capacity()) evaluate the three-body op with one warp per centre atom out of shared memory: no
 * triplet index list is read.  fwd writes red for member bonds only and e_out for all bonds; bwd writes g_vec4 for
 * all bonds (zeros for non-members) and g_bas for member bonds only (pair it with the member edge_list of
 * m3g_tb_edge_basis_bwd).  The gradient w.r.t. e_in is g_e itself. */
int m3g_tri_dense_check(const int32_t* src, const int32_t* edge_ptr, const int32_t* tri_ptr, const int32_t* tri_e2,
                        int64_t E, int32_t* flags, void* stream);
int m3g_tb_atom_capacity(void);
int m3g_tb_atom_fwd(const float* vec4, const float* bas, const int32_t* edge_ptr, const int32_t* tri_ptr, float r3,
                    const float* WdT, const float* WgT, const float* e_in, int64_t N, int n_sm, float* red,
                    float* e_out, void* stream);
int m3g_tb_atom_bwd(const float* vec4, const float* bas, const float* red, const float* g_e, const int32_t* edge_ptr,
                    const int32_t* tri_ptr, float r3, const float* WdT, const float* WgT, int64_t N, int n_sm,
                    float* g_vec4, float* g_bas, void* stream);

/* O(n3)-per-atom moment form of the same op (csrc/threebody_moment.cu; replaces nn/interaction.py:187-223, :353-382 and
 * their autograd for l_max = n_max = 3, F = 64 and the canonical triplet layout, members per atom <=
 * m3g_tb_mom_capacity()).  m3g_tb_radial (once per step; nn/interaction.py:226-281, :389-400): G[e][d] = chi_d(r_e) fc(r_e)
 * and dG/dr for the listed member bonds.  m3g_tb_mom_fwd: red (member bonds) and e_out (all bonds) with bas = G *
 * sig[dst] formed in-kernel.  m3g_tb_mom_bwd: g_vec4 (E,4) complete (cos, fc' and radial chain; zeros for
 * non-members; accumulate != 0 adds to the existing rows: the sum over the model's blocks) and g_sig_e (E,9) (zeros for
 * non-members, written by the accumulate == 0 call: with accumulate != 0 both buffers must come from such a call on the
 * same bond list), ready for m3g_tb_sigma_bwd.  The Legendre adjoint follows
 * the reference's quirk (Q3) through second-order moments.  max_members: upper bound of member bonds per atom. */
int m3g_tb_radial(const float* vec4, const float* tb_consts, int64_t E, int L, int R, const int32_t* edge_list,
                  int64_t n_list, float* G, float* dG, void* stream);
int m3g_tb_mom_capacity(void);
/* m3g_tb_sigma_fwd / _bwd specialised for F = 64, D = 9 (weights in registers, one shared butterfly for the nine sums,
 * warps striding over atoms; n_sm sizes the persistent grid) */
int m3g_tb_sigma64_fwd(const float* x, const float* Ws, const float* bs, int64_t N, int n_sm, float* sig, void* stream);
int m3g_tb_sigma64_bwd(const float* g_sig_e, const int32_t* in_ptr, const int32_t* in_perm, const float* sig,
                       const float* Ws, const float* base, int64_t N, int n_sm, float* g_x, void* stream);
int m3g_tb_mom_fwd(const float* vec4, const float* G, const float* sig, const int32_t* dst, const int32_t* edge_ptr,
                   const int32_t* tri_ptr, float r3, const float* WdT, const float* WgT, const float* e_in, int64_t N,
                   int max_members, int n_sm, float* red, float* e_out, void* stream);
/* the forward in two launches (default): m3g_tb_mom_red = the per-atom moment part only (red for member bonds), then
 * m3g_tb_edge_update = e_out = e_in + SiLU(red WdT) * sigmoid(red WgT) streamed over all bond rows (members by
 * tri_ptr), independent of the atom structure and bound by the 512 B per bond it moves */
int m3g_tb_mom_red(const float* vec4, const float* G, const float* sig, const int32_t* dst, const int32_t* edge_ptr,
                   const int32_t* tri_ptr, float r3, int64_t N, int max_members, int n_sm, float* red, void* stream);
int m3g_tb_edge_update(const float* red, const int32_t* tri_ptr, const float* WdT, const float* WgT, const float* e_in,
                       int64_t E, int n_sm, float* e_out, void* stream);
/* the same with e_in = SiLU(h WaT) (the EdgeAdjustor's output, nn/featurizer.py:84-96; h (E,3), WaT (3,64)) formed
 * in-kernel: the first block of the whole-step executor neither writes nor re-reads e0 (bit-identical to
 * m3g_edge_adjust_fwd followed by m3g_tb_edge_update) */
int m3g_tb_edge_update_h(const float* red, const int32_t* tri_ptr, const float* WdT, const float* WgT, const float* h,
                         const float* WaT, int64_t E, int n_sm, float* e_out, void* stream);
int m3g_tb_mom_bwd(const float* vec4, const float* G, const float* dG, const float* sig, const int32_t* dst,
                   const float* red, const float* g_e, const int32_t* edge_ptr, const int32_t* tri_ptr, float r3,
                   const float* WdT, const float* WgT, int64_t N, int max_members, int n_sm, int accumulate,
                   float* g_vec4, float* g_sig_e, void* stream);
/* the backward in two launches (default): m3g_tb_mlp_adj = adjoint of the 9 -> 64 gated MLP (nn/interaction.py:219-220,
 * nn/core.py:61-62) over the packed member-bond list, q[e] = dL/dred[e] (a lane owns a row: no cross-lane sums; q may
 * alias red); then m3g_tb_mom_bwd_q = the per-atom moment part of m3g_tb_mom_bwd reading q (no weights, no edge rows) */
int m3g_tb_mlp_adj(const float* red, const float* g_e, const int32_t* member_edges, int64_t n_members, const float* WdT,
                   const float* WgT, int n_sm, float* q, void* stream);
int m3g_tb_mom_bwd_q(const float* vec4, const float* G, const float* dG, const float* sig, const int32_t* dst,
                     const float* q, const int32_t* edge_ptr, const int32_t* tri_ptr, float r3, int64_t N,
                     int max_members, int n_sm, int accumulate, float* g_vec4, float* g_sig_e, void* stream);

/* Specialised variants for the default model shape l_max = n_max = 3, F = 64 (compile-time loops, gated-MLP
 * weights in shared memory, vector row I/O, persistent grid of 8 x n_sm blocks).  Same results and buffers as
 * the generic entry points above; r3 = three-body cutoff.  m3g_tb_reduce_bwd_sym requires a symmetric triplet
 * list ((e1,e2) present <=> (e2,e1) present — always true for graphs from from_structure). */
int m3g_tb_reduce_fwd_fast(const float* vec4, const float* bas, const int32_t* tri_ptr, const int32_t* tri_e2,
                           float r3, const float* WdT, const float* WgT, const float* e_in, int64_t E, int group,
                           int n_sm, float* red, float* e_out, void* stream);
int m3g_tb_gate_bwd_fast(const float* red, const float* g_e, const float* WdT, const float* WgT,
                         const int32_t* tri_ptr, int64_t E, int n_sm, float* g_red, void* stream);
int m3g_tb_reduce_bwd_sym(const float* vec4, const float* bas, const float* g_red, const int32_t* tri_ptr,
                          const int32_t* tri_e2, float r3, int64_t E, int group, int n_sm, float* g_vec4, float* g_bas,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Generic row-wise linear: out (n,M) = in (n,K) · Wt (K,M) + bias (M or NULL).  Used for the per-atom
 * first-layer projections of M3GNetConv (nn/conv.py:92-97 concat split: [x_i,x_j,e]·W = x_i·W_i + x_j·W_j + e·W_e)
 * ------------------------------------------------------------------------------------------- */
int m3g_linear_fwd(const float* in, const float* Wt, const float* bias, int64_t n, int K, int M, float* out,
                   void* stream);

/* ---------------------------------------------------------------------------------------------
 * Elementwise pieces of a GatedMLP called on its own (nn/core.py:45-62): activation kind 0 = SiLU, 1 = sigmoid;
 * m3g_act_bwd: out = g * act'(in); m3g_mul: out = a * b.  (csrc/elementwise.cu)
 * ------------------------------------------------------------------------------------------- */
int m3g_act_fwd(const float* in, int64_t n, int kind, float* out, void* stream);
int m3g_act_bwd(const float* in, const float* g, int64_t n, int kind, float* out, void* stream);
int m3g_mul(const float* a, const float* b, int64_t n, float* out, void* stream);
/* out = a + b (out may alias a or b) */
int m3g_add(const float* a, const float* b, int64_t n, float* out, void* stream);
/* out[i] = sum_k slices[k * n + i], k ascending */
int m3g_sum_slices(const float* slices, int K, int64_t n, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * M3GNetConv (nn/conv.py:63-97, nn/core.py:6-62).  One "gated MLP on edges":
 *   z1 = P[src][po .. po+2F) + P[dst][po+2F .. po+4F) + e · W1eT            (2F: dense | gate)
 *   a1 = SiLU(z1); z2d = a1d·W2dT + b2d; z2g = a1g·W2gT + b2g
 *   out = SiLU(z2d) * sigmoid(z2g) * (h · WhT)
 * P (N, ldp) holds the per-atom projections (bias of layer 1 folded into the src part).
 * mode 0 (edge update, conv.py:68-75): y = e + out, written to y (E,F)
 * mode 1 (node update, conv.py:77-89): y = out (messages); m3g_segment_sum_add then adds them per source atom
 * ------------------------------------------------------------------------------------------- */
int m3g_conv_mlp_fwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                     const float* h, const float* W1eT, const float* W2dT, const float* b2d, const float* W2gT,
                     const float* b2g, const float* WhT, int64_t E, int F, int R, int mode, float* y, void* stream);
/* out (N,F) = base (N,F) + sum_{e in [edge_ptr[i], edge_ptr[i+1])} msg[e] */
int m3g_segment_sum_add(const float* base, const float* msg, const int32_t* edge_ptr, int64_t N, int F,
                        float* out, void* stream);
/* the same sum from the partial rows of m3g_conv_tc_fwd(mode = 2): the tensor-core forward reduces the messages of every
 * 32-row block per source atom in its epilogue and writes one partial row per (block, atom) at the block's first row of
 * that atom (the other rows of `part` are never written nor read); out[i] = base[i] + sum_k part[max(b_i, 32 k)] */
int m3g_segment_sum_parts(const float* base, const float* part, const int32_t* edge_ptr, int64_t N, int F,
                          float* out, void* stream);
/* adjoint of one gated MLP on edges (activations recomputed).  Upstream gradient of `out`:
 *   mode 0: g_u[e] rows of g_up (E,F);   mode 1: g_u[e] = g_up[src[e]] rows of g_up (N,F).
 * Outputs: g_e (E,F) = g_e_base (may be NULL = 0) + d out/d e adjoint; g_z1 (E,2F); g_h (E,R) accumulated (+=)
 * W1e (2F,F) is the e-part of layer 1 in (out,in) layout; W2d/W2g (F,F) in (out,in) layout; Wh (F,R). */
int m3g_conv_mlp_bwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                     const float* h, const float* W1eT, const float* W2dT, const float* b2d, const float* W2gT,
                     const float* b2g, const float* WhT, const float* W1e, const float* W2d, const float* W2g,
                     const float* Wh, const float* g_up, const float* g_e_base, int64_t E, int F, int R, int mode,
                     float* g_e, float* g_z1, float* g_h, void* stream);
/* g_P (N, ldp)[po..po+2F) = sum_{out(i)} g_z1, [po+2F..po+4F) = sum_{in(i)} g_z1 */
int m3g_conv_gather_gz(const float* g_z1, const int32_t* edge_ptr, const int32_t* in_ptr, const int32_t* in_perm,
                       int64_t N, int F, int ldp, int po, float* g_P, void* stream);
/* out (n,K) = base (n,K or NULL) + g (n,M) · W (M,K)   — adjoint of m3g_linear_fwd w.r.t. its input */
int m3g_linear_bwd_input(const float* g, const float* W, const float* base, int64_t n, int K, int M, float* out,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core path of the same gated MLP for F = 64 (csrc/conv_tc.cu): tcgen05.mma kind::tf32 with the 3xTF32
 * split (passes = 3; passes = 1 is plain TF32), accumulators in TMEM, weight images resident in shared memory.
 * m3g_tc_pack_b writes the hi / lo SWIZZLE_128B operand images of a (rows x cols) row-major weight matrix
 * (rows % 8 == 0, cols % 32 == 0; each image rows*cols floats).  wimg = [W1e hi | W1e lo | W2d hi | W2d lo |
 * W2g hi | W2g lo] with W1e (128 x 64) = rows [dense | gate] of the e-part of layer 1, W2d/W2g (64 x 64), all in
 * the reference's (out,in) orientation.  n_sm = number of SMs (persistent grid: two warp groups per CTA ping-pong
 * two 128-edge tiles; R <= 4).
 * ------------------------------------------------------------------------------------------- */
int m3g_tc_pack_b(const float* W, int rows, int cols, float* img_hi, float* img_lo, void* stream);
/* debug: per-phase cycle sums of the backward kernel (HOST buffer of 16 int64; all zero unless the library was built
 * with -DM3G_TC_TIMING); synchronises the stream */
int m3g_debug_tc_timing(int64_t* out16, int reset, void* stream);
/* debug: cycles to issue / to complete n_mma back-to-back tcgen05.mma kind::tf32 (M = 128, K = 8) of width N with A
 * from shared (a_tmem = 0) or tensor memory (1); cycles2 = DEVICE buffer of two int64 */
int m3g_debug_mma_rate(int N, int a_tmem, int n_mma, int64_t* cycles2, void* stream);
/* same for tcgen05.mma.cta_group::2 (M = 256 over a two-CTA cluster, A and B from shared memory): cycles2[0] = issue
 * loop, cycles2[1] = until the multicast commit arrives in the leader CTA. */
int m3g_debug_mma_rate2(int N, int n_mma, int64_t* cycles2, void* stream);
/* dev tool (tools/pipe_rate.py): clock cycles of `iters` x 32 instructions of one kind per thread (8 independent
 * chains) with `threads` threads per SM — kinds in csrc/debug_rate.cu */
int m3g_debug_pipe_rate(int kind, int threads, int iters, int64_t* cycles, void* stream);
/* UMMA plumbing self test on one 128-row tile: out (128 x rows) = A (128 x cols) · W^T, W given as its image;
 * a_tmem = 1 feeds A from tensor memory (tcgen05.st + the [a_tmem] operand form) instead of shared memory */
int m3g_tc_selftest(const float* A, const float* img_hi, const float* img_lo, int rows, int cols, int passes,
                    int a_tmem, float* out, void* stream);
/* mode 0 / 1 as m3g_conv_mlp_fwd; mode 2 = mode 1 with the messages summed per source atom inside the epilogue: y then
 * holds one partial row per (32-row block, source atom) at the block's first row of that atom, for
 * m3g_segment_sum_parts (the other rows of y are not written) */
int m3g_conv_tc_fwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                    const float* h, const float* wimg, const float* b2d, const float* b2g, const float* WhT, int64_t E,
                    int R, int mode, int passes, int n_sm, float* y, float* save, void* stream);
/* (nn/conv.py:63-89 with nn/core.py:30-62 for m3g_conv_tc_fwd; the two functions below replace its autograd)
 * save (optional): activations for m3g_conv_tc_bwd_saved — m3g_conv_tc_save_floats(E) floats (1 KB per edge:
 * SiLU'(z1) and the layer-2 pre-activations, in a tile-private fragment-major layout).  With them the backward needs
 * neither the forward weights nor P / e: output adjoint -> two 64x64 adjoint GEMM pairs -> g_e, g_z1, g_h (same outputs
 * and conventions as m3g_conv_tc_bwd; src is only read for mode 1, where g_up is indexed by source atom).
 * gh_store != 0: the g_h rows are stored instead of added to the rows already there (a caller that gives every launch
 * its own (E,R) slice and sums them with m3g_sum_slices: no read-modify-write inside the kernel). */
int64_t m3g_conv_tc_save_floats(int64_t E);
int m3g_conv_tc_bwd_saved(const int32_t* src, const float* h, const float* wimgT, const float* WhT, const float* save,
                          const float* g_up, const float* g_e_base, int64_t E, int R, int mode, int passes, int n_sm,
                          float* g_e, float* g_z1, float* g_h, int gh_store, void* stream);
/* Both adjoints of one M3GNetConv block in one launch: the node-MLP call (mode 1, g_up = g_x2, g_e_base = g_e2) and
 * then the edge-MLP call (mode 0, g_up = g_e_base = its output ge2) of m3g_conv_tc_bwd_saved, with ge2 kept on chip.
 * g_e, gz_node / gz_edge (nullable) and the g_h rows are bitwise those of the two calls.  gh_mode 0: the node and the
 * edge launch's g_h rows are stored into g_h_node and g_h_edge (per-launch slices, as gh_store = 1); gh_mode 1: their
 * sum fl(node + edge) is stored into g_h_node (g_h_edge unused, may be NULL).  g_e2 may be NULL (no residual base). */
int m3g_conv_tc_block_bwd(const int32_t* src, const float* h, const float* n_wimgT, const float* n_WhT,
                          const float* save_n, const float* e_wimgT, const float* e_WhT, const float* save_e,
                          const float* g_x2, const float* g_e2, int64_t E, int R, int passes, int n_sm, float* g_e,
                          float* gz_node, float* gz_edge, float* g_h_node, float* g_h_edge, int gh_mode, void* stream);

/* adjoint of m3g_conv_tc_fwd (same outputs as m3g_conv_mlp_bwd; forward recomputed on the tensor cores).
 * wimgT = [W2d^T hi|lo, W2g^T hi|lo, W1e_dense^T hi|lo, W1e_gate^T hi|lo]: four 64x64 image pairs from
 * m3g_tc_pack_b of the transposed matrices (W1e_dense = rows 0..63 of W1e, W1e_gate = rows 64..127). R <= 3. */
int m3g_conv_tc_bwd(const float* P, int ldp, int po, const int32_t* src, const int32_t* dst, const float* e,
                    const float* h, const float* wimg, const float* wimgT, const float* b2d, const float* b2g,
                    const float* WhT, const float* g_up, const float* g_e_base, int64_t E, int R, int mode, int passes,
                    int n_sm, float* g_e, float* g_z1, float* g_h, void* stream);

/* ---------------------------------------------------------------------------------------------
 * AtomWiseReadout (nn/readout.py:39-58) + virial (nn/gradient.py:39-62)
 * weights: 3-layer gated MLP F→F→F→1; WT = (in,out) layout, W = (out,in) layout
 * ------------------------------------------------------------------------------------------- */
int m3g_readout_fwd(const float* x, const float* W0dT, const float* b0d, const float* W1dT, const float* b1d,
                    const float* w2d, const float* b2d, const float* W0gT, const float* b0g, const float* W1gT,
                    const float* b1g, const float* w2g, const float* b2g, const float* elemental, float scale,
                    int64_t N, int F, float* atomic, void* stream);
/* scaled_total[b] = sum_{i in [atom_ptr[b], atom_ptr[b+1])} atomic[i]; total = scale * scaled_total */
int m3g_structure_sum(const float* atomic, const int32_t* atom_ptr, int64_t B, float scale, float* scaled_total,
                      float* total, void* stream);
/* g_eps[i] = g_atomic[i] + g_scaled_total[b] + scale*g_total[b] (each may be NULL); g_x (N,F) */
int m3g_readout_bwd(const float* x, const float* W0dT, const float* b0d, const float* W1dT, const float* b1d,
                    const float* w2d, const float* b2d, const float* W0gT, const float* b0g, const float* W1gT,
                    const float* b1g, const float* w2g, const float* b2g, const float* W0d, const float* W1d,
                    const float* W0g, const float* W1g, const float* g_atomic, const float* g_scaled_total,
                    const float* g_total, const int32_t* batch, float scale, int64_t N, int F, float* g_x,
                    void* stream);
/* m3g_readout_fwd and m3g_readout_bwd in ONE launch for a caller that knows the upstream gradient beforehand (the
 * whole-step executor: g_total is an input): writes atomic (N) and g_x (N,F); same arithmetic as the two calls */
int m3g_readout_fwd_bwd(const float* x, const float* W0dT, const float* b0d, const float* W1dT, const float* b1d,
                        const float* w2d, const float* b2d, const float* W0gT, const float* b0g, const float* W1gT,
                        const float* b1g, const float* w2g, const float* b2g, const float* W0d, const float* W1d,
                        const float* W0g, const float* W1g, const float* elemental, const float* g_total,
                        const int32_t* batch, float scale, int64_t N, int F, float* atomic, float* g_x, void* stream);
/* forces = -g_pos; stresses (B,6) = Voigt(sum_i pos_i (x) F_i)/|det lattice| */
int m3g_forces_virial(const float* pos, const float* g_pos, const float* lattice, const int32_t* atom_ptr,
                      int64_t N, int64_t B, float* forces, float* stresses, void* stream);
/* Cell stress (extension, no reference counterpart; the reference's only stress is the origin-dependent virial row of
 * nn/gradient.py:25-64 above).  sigma (B,3,3) row-major, eV/A^3:
 *   sigma_b[a][c] = (1/V_b) sum_{e in structure b} v_e[a] g_e[c],   g_e = g_vec4.xyz + (g_vec4.w + g_dist)·v/r,
 * i.e. (1/V) dE_b/d(eps_ac) at eps = 0 for positions and lattice rows deformed as r -> r (I + eps); V_b = |det lattice_b|.
 * Same bond-gradient inputs as m3g_geometry_bwd (g_vec4 / g_dist may be NULL); vec4 and its gradient may be in scaled
 * lengths (v (x) dE/dv does not depend on the length unit), lattice must be in A.  ASE convention: Voigt order
 * [xx, yy, zz, yz, xz, xy] of sigma is ASE's "stress" (pressure = -tr(sigma)/3; positive = tensile).  The bonds of
 * structure b are edge_ptr[atom_ptr[b]] .. edge_ptr[atom_ptr[b+1]]; structures without bonds get sigma = 0.
 * Deterministic: float64 partial sums over fixed 2048-bond chunks, then a fixed-order sum per structure (two launches,
 * no atomics).  work: m3g_bond_virial_work_elems(E, B) doubles of caller-owned scratch. */
int64_t m3g_bond_virial_work_elems(int64_t E, int64_t B);
int m3g_bond_virial(const float* vec4, const float* g_vec4, const float* g_dist, const int32_t* edge_ptr,
                    const int32_t* atom_ptr, int64_t E, int64_t B, const float* lattice, double* work, float* sigma,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched FIRE relaxation step (csrc/relax.cu; extension, no reference counterpart): one step of calculator.py::Fire
 * for every running structure of a ragged batch, each with its own FIRE state.  Per structure b (rows
 * atom_ptr[b] .. atom_ptr[b+1]) whose status[b] == 0:
 *   - generalised forces g: forces (N,3) f32 as they are, or with the cell filter (sigma != NULL; ASE UnitCellFilter
 *     as Fire(relax_cell=True)): D = solve(L0_b, lattice_b)^T, atom rows F D, 3 cell rows
 *     -|det lattice_b| (sigma_b + pressure I) D^-T / cell_factor[b];
 *   - fmax[b] = max row |g| (+inf and status 3 = failed if any g is not finite); fmax[b] < fmax_target -> status 1
 *     (converged); else n_steps[b] >= max_steps -> status 2 (not converged); otherwise one FIRE step with Fire's
 *     parameters (P = g.v > 0: v = (1-a) v + a|v| g/max(|g|,1e-30), dt / a updated after n_min positive steps;
 *     else v = 0, a = a_start, dt *= f_dec), v += dt g, dr = dt v clipped to |dr| <= max_move (norm over the
 *     structure's rows), n_steps[b] += 1;
 *   - without the cell filter pos (N,3) += dr; with it the generalised positions x (N,3) and xc (B,3,3) (= cell_factor
 *     D; initially pos and cell_factor I) get dr, and pos = x Dn^T, lattice_b = L0_b Dn^T with Dn = xc_b / cell_factor[b];
 *   - e_frame[b] = energy[b] and sigma_frame = sigma (f64, cell filter only) of the frame just checked (e_frame may be
 *     NULL).  Together with pos / lattice / fmax these are the values of the frame at which a structure stopped.
 * Velocities v (N,3), vc (B,3,3); dt, a (B) f64; n_pos, n_steps, status (B) int32; L0, lattice (B,3,3) f64 row-major.
 * Structures with status != 0 are not touched.  Without the cell filter x, xc, vc, L0, lattice, cell_factor and
 * sigma_frame are not read (may be NULL).  One launch, one 256-thread block per structure; every sum runs over the
 * structure's rows in a fixed thread-row map and a fixed tree (no atomics, no scratch), so a structure's new state
 * depends only on its own rows, not on its position in the batch. */
int m3g_fire_step(const float* forces, const float* sigma, const float* energy, const int32_t* atom_ptr, int64_t B,
                  double dt_max, double max_move, int n_min, double f_inc, double f_dec, double a_start, double f_a,
                  double fmax_target, int max_steps, double pressure, const double* cell_factor, double* x, double* xc,
                  double* v, double* vc, double* dt, double* a, int32_t* n_pos, int32_t* n_steps, int32_t* status,
                  const double* L0, double* lattice, double* pos, double* fmax, double* e_frame, double* sigma_frame,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched climbing-image NEB step (csrc/neb.cu; extension, no reference counterpart): one FIRE step of every running
 * band of a ragged batch, improved tangent (Henkelman & Jonsson 2000) with an optional climbing image, as ASE's
 * NEB(method="improvedtangent") optimised by FIRE.  Band b has M_b = image_ptr[b+1] - image_ptr[b] interior images
 * (1 <= M_b <= M3G_NEB_MAX_IMAGES) of n_b = (end_ptr[b+1] - end_ptr[b]) / 2 atoms each: interior rows row_ptr[b] ..
 * row_ptr[b+1] (= M_b n_b rows, image-major) of pos / v / forces (f64 / f64 / f32, (rows,3)), interior energies
 * energy[image_ptr[b] ..] f32, endpoint positions ends rows end_ptr[b] .. (image 0's n_b rows, then image M_b+1's)
 * and endpoint energies e_end (B,2) f64, spring constant k[b] (eV/A^2).  For every band with status[b] == 0:
 *   - e_frame[image] = energy (f64); i_climb[b] = the interior image (1 .. M_b, band numbering) of highest energy,
 *     ties to the lowest index;
 *   - per interior image i, t+ = R_{i+1} - R_i, t- = R_i - R_{i-1} (raw differences) and the tangent t = t+ if
 *     E_{i+1} > E_i > E_{i-1}, t- if E_{i+1} < E_i < E_{i-1}, else dVmax t+ + dVmin t- when E_{i+1} > E_{i-1} and
 *     dVmin t+ + dVmax t- otherwise (dVmax / dVmin = max / min of |E_{i+1} - E_i|, |E_{i-1} - E_i|), t+ + t- when
 *     dVmax = 0; t^ = t / |t|;
 *   - G_i = F_i - (F_i.t^) t^ + k (|t+| - |t-|) t^, or F_i - 2 (F_i.t^) t^ for the climbing image when climb != 0;
 *   - status 3 (failed), fmax = +inf, if an energy is not finite or some |t| is 0 or not finite; otherwise
 *     m3g_fire_step's fixed-cell step on the band's M_b n_b rows of G as one structure (fmax = max row |G|, power,
 *     norms and the max_move clip over the band), with dt, a, n_pos, n_steps, status, fmax per band.
 * Bands with status != 0 are not touched.  max_images: the largest M_b of the launch (checked against the cap).  One
 * launch, one 256-thread block per band, relax.cu's thread-row map and fixed trees (no atomics, no scratch), so a
 * band's new state depends only on its own rows. */
#define M3G_NEB_MAX_IMAGES 64
int m3g_neb_step(const float* forces, const float* energy, const int32_t* row_ptr, const int32_t* image_ptr,
                 const int32_t* end_ptr, int64_t B, int max_images, const double* ends, const double* e_end,
                 const double* k, int climb, double dt_max, double max_move, int n_min, double f_inc, double f_dec,
                 double a_start, double f_a, double fmax_target, int max_steps, double* pos, double* v, double* dt,
                 double* a, int32_t* n_pos, int32_t* n_steps, int32_t* status, double* fmax, int32_t* i_climb,
                 double* e_frame, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched harmonic phonons (csrc/phonon.cu; extension, no reference counterpart).  Structure b has a unit cell of
 * n_b = atom_ptr[b+1] - atom_ptr[b] atoms (1 <= n_b <= M3G_PHONON_MAX_ATOMS), a diagonal supercell reps[b] (3 int32)
 * of L_b = r1 r2 r3 cells and N_b = n_b L_b atoms, supercell atom j = l n_b + k' with l = (i1 r2 + i2) r3 + i3.  Its
 * (k, j) pairs are pair_ptr[b] + k N_b + j; its force constants fc (pairs, 3, 3) f64 eV/A^2 hold
 * Phi(0k alpha; j beta) (phonopy's compact layout).  Everything is float64 and deterministic: sums run in a fixed
 * order that depends only on the structure's own data, so its output does not depend on the rest of the batch.
 *
 * m3g_phonon_force_constants: forces rows row_ptr[b] .. (f32, (6 n_b + 1) N_b rows: the undisplaced supercell, then
 *   for k = 0 .. n_b-1 and alpha = x, y, z the supercells with atom k of cell 0 moved by +h and by -h along alpha);
 *   Phi = -(F(+h) - F(-h)) / 2h, then `symmetrize` rounds of (a) Phi(0k; l k')_ab <- (Phi(0k; l k')_ab +
 *   Phi(0k'; -l k)_ba) / 2 (-l wrapped in the supercell) and (b) Phi(0k; 0k) -= sum_j Phi(0k; j) (acoustic sum
 *   rule).  status[b] = 0, residual[b] = max |F| of the undisplaced supercell; a structure with any non-finite force
 *   gets status 1, NaN force constants and residual.  One 256-thread block per structure.
 * m3g_phonon_dynmat: dmat (Q, ld, ld) complex128 (re, im interleaved), ld >= 3 max n: D(q) of q-point i (fractional
 *   coordinates of the unit cell's reciprocal lattice, q (Q,3) f64) of structure b (q_ptr[b] <= i < q_ptr[b+1],
 *   int32), D_{3k+a, 3k'+b}(q) = sum_l Phi(0k; l k')_ab (1/|M|) sum_{v in M} exp(2 pi i q.v) / sqrt(m_k m_k');
 *   M is the minimum-image set of the pair: vectors sv[sv_ptr[p] .. sv_ptr[p+1]] (unit-cell fractional coordinates of
 *   the lattice translation from cell 0 to the image's cell, (rows, 3) f64), sv_ptr (pairs + 1) int64; mass (atoms)
 *   f64 amu.  Entries outside 3 n_b x 3 n_b are zero.  One block per q-point.
 * m3g_phonon_frequencies: per q-point the same D(q), its Hermitian part (D + D^H) / 2 and its eigenvalues by a cyclic
 *   complex Jacobi method (round-robin pair order, 3n/2 disjoint rotations per round), until the off-diagonal
 *   Frobenius norm is <= 1e-13 ||D||_F.  eig (f64, eV/(amu A^2)) and freq = sign(eig) sqrt(|eig|) thz (THz), ascending,
 *   at f_ptr[b] + (i - q_ptr[b]) 3 n_b (f_ptr (B+1) int64); sweeps[i] = Jacobi sweeps, q_status[i] = 0.  A structure
 *   with status[b] != 0, a non-finite D or 30 sweeps without convergence give NaN and q_status 1.  One block per
 *   q-point, (3 max_atoms)^2 x 16 B of dynamic shared memory.
 * m3g_phonon_thermal: per structure b and temperature temps[t] (K), over the frequencies f >= cutoff (THz) of its
 *   q-points with e = h_thz f (eV), x = e / kT, kT = kB T: out[b, t, :] = (F, S, Cv, E) / N_q with
 *   F = sum e/2 + kT ln(1 - e^-x), S = kB sum x/(e^x - 1) - ln(1 - e^-x), Cv = kB sum x^2 e^x / (e^x - 1)^2,
 *   E = sum e (1/2 + 1/(e^x - 1)) (T = 0: F = E = sum e/2, S = Cv = 0); n_imag[b] = #{f < -cutoff},
 *   fmin[b] = min f.  NaN frequencies give NaN; a structure with status[b] != 0 gets NaN, n_imag -1.  One block per
 *   (structure, temperature); fixed-order block reductions.
 * ------------------------------------------------------------------------------------------- */
#define M3G_PHONON_MAX_ATOMS 32
int m3g_phonon_force_constants(const float* forces, const int64_t* row_ptr, const int32_t* atom_ptr,
                               const int32_t* reps, const int64_t* pair_ptr, int64_t B, int max_atoms, double h,
                               int symmetrize, double* fc, int32_t* status, double* residual, void* stream);
int m3g_phonon_dynmat(const double* fc, const int32_t* atom_ptr, const int32_t* reps, const int64_t* pair_ptr,
                      const int64_t* sv_ptr, const double* sv, const double* mass, const double* q,
                      const int32_t* q_ptr, int64_t B, int64_t Q, int max_atoms, int ld, double* dmat, void* stream);
int m3g_phonon_frequencies(const double* fc, const int32_t* atom_ptr, const int32_t* reps, const int64_t* pair_ptr,
                           const int64_t* sv_ptr, const double* sv, const double* mass, const int32_t* status,
                           const double* q, const int32_t* q_ptr, const int64_t* f_ptr, int64_t B, int64_t Q,
                           int max_atoms, double thz, double* eig, double* freq, int32_t* sweeps, int32_t* q_status,
                           void* stream);
int m3g_phonon_thermal(const double* freq, const int64_t* f_ptr, const int32_t* q_ptr, const int32_t* status,
                       int64_t B, const double* temps, int64_t T, double kB, double h_thz, double cutoff, double* out,
                       int32_t* n_imag, double* fmin, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched Langevin MD (csrc/md.cu; extension, no reference counterpart): BAOAB (Leimkuhler & Matthews 2013) on fixed
 * cells for every running structure of a ragged batch.  Positions pos (N,3) f64 A, velocities v (N,3) f64 A/fs,
 * inv_mass (N) f64 = ACC_UNIT / m (calculator.py), dt fs; per structure c1 = exp(-gamma dt), c2 = sqrt(1 - c1^2) and
 * kT (eV) f64, the stream id sid (int64; the structure's index in the caller's list), the step counter step and status
 * (0 = running, 1 = failed) int32, bath f64.
 *
 * Noise: Philox4x64-10 (numpy.random.Philox's generator) with key (seed, 0) (seed reinterpreted as uint64) and counter
 * (i, sid, k, tag): i = atom index within its structure, k = step, tag 0 = Langevin noise, 1 = starting velocities.
 * u = ((w >> 11) + 0.5) 2^-53; one call gives xi = (sqrt(-2 ln u0) cos(2 pi u1), sqrt(-2 ln u0) sin(2 pi u1),
 * sqrt(-2 ln u2) cos(2 pi u3)).  No generator state is stored; the noise names the structure, not its batch row.
 *
 * m3g_langevin_step: one launch per MD step with the forces (N,3) and energy (B) f32 of frame k = step[b], for every
 * structure with status 0:
 *   1. unless k == 0, the closing half kick v += dt/2 F inv_mass of step k - 1 gives v_k;
 *   2. the structure fails (status 1; pos, v, step and bath left as they were) if a force, v_k or the energy is not
 *      finite or max_i |v_k,i| dt > max_step_move; otherwise, when slot >= 0, obs[slot, b, :] (f64) =
 *      (E_pot, E_kin, T_kin = 2 E_kin / ((3 n_b - 3) kB), bath) with E_kin = sum |v_k|^2 / (2 inv_mass);
 *   3. advance != 0: B (v += dt/2 F inv_mass), A (x += dt/2 v), O (v = c1 v + c2 sqrt(kT inv_mass) xi, counter step k,
 *      tag 0, then the mass-weighted mean velocity removed), A (x += dt/2 v) -> x_{k+1}; bath += the kinetic energy the
 *      O step and the removal added; step = k + 1.  advance == 0 (the final frame): v = v_k.
 * One 256-thread block per structure; every sum runs in relax.cu's fixed thread-row map and tree (no atomics, no
 * scratch), so a structure's new state depends only on its own rows and sid.
 *
 * m3g_langevin_npt_step: m3g_langevin_step plus a stochastic cell-rescaling barostat (Bernetti & Bussi 2020), same
 * kernel body.  Extra inputs: the cell stress sigma (B,3,3) f32 of frame k (eV/A^3, ASE sign, P = -tr sigma / 3), the
 * lattice (B,3,3) f64 row-major (rows are lattice vectors; L_k in, L_{k+1} out), per structure P0 (eV/A^3), beta_T
 * (A^3/eV) and tau_p (fs) f64, coupling (0 = isotropic, 1 = per Cartesian axis) and max_step_strain.  After step 1:
 *   - V = |det L_k|, P_int = 2 E_kin / (3 V) - tr(sigma) / 3, per axis P_a = 2 K_aa / V - sigma_aa with
 *     K_aa = sum v_a^2 / (2 inv_mass);
 *   - d eps = -(beta_T dt / tau_p) (P0 - P) + sqrt(2 kT beta_T dt / (V tau_p)) xi with xi from counter
 *     (0, sid, k, tag 2): one step in ln V with P = P_int and xi_0 (isotropic, mu_a = exp(d eps / 3)), or one per axis
 *     with P = P_a and xi_a (mu_a = exp(d eps_a));
 *   - the structure also fails if an entry of sigma or V is not finite or any |ln mu_a| > max_step_strain (lattice left
 *     as it was too);
 *   - obs rows are (E_pot, E_kin, T_kin, bath, V, P_int), 6 columns isotropic, and per axis 9 with (P_x, P_y, P_z)
 *     appended: obs is (n_slots, B, 6) or (n_slots, B, 9);
 *   - advance != 0: after B A O A, x_{k+1} = x_{k+1} diag(mu), v = v diag(mu)^-1, L_{k+1} = L_k diag(mu).  bath keeps
 *     its meaning (the O step and the centre-of-mass removal; the barostat's work is not in it).
 * With beta_T = 0, mu = 1 exactly and pos, v, step, status, bath and obs[..., :4] are bitwise those of
 * m3g_langevin_step.
 *
 * m3g_md_maxwell_boltzmann: v = sqrt(kT inv_mass) xi (counter step 0, tag 1), then the mass-weighted mean velocity of
 * each structure removed; no rescaling.  One launch, one block per structure.
 *
 * m3g_debug_philox4x64: out (n,4) = philox4x64_10(ctr (n,4), key (n,2)), words as uint64 in int64 storage.
 * ------------------------------------------------------------------------------------------- */
int m3g_langevin_step(const float* forces, const float* energy, const int32_t* atom_ptr, int64_t B, double dt,
                      double max_step_move, int64_t seed, int advance, int slot, const double* inv_mass,
                      const double* c1, const double* c2, const double* kT, const int64_t* sid, double* pos, double* v,
                      int32_t* step, int32_t* status, double* bath, double* obs, void* stream);
int m3g_langevin_npt_step(const float* forces, const float* energy, const int32_t* atom_ptr, int64_t B, double dt,
                          double max_step_move, int64_t seed, int advance, int slot, const double* inv_mass,
                          const double* c1, const double* c2, const double* kT, const int64_t* sid, double* pos,
                          double* v, int32_t* step, int32_t* status, double* bath, double* obs, const float* sigma,
                          double* lattice, const double* P0, const double* beta_T, const double* tau_p, int coupling,
                          double max_step_strain, void* stream);
int m3g_md_maxwell_boltzmann(const int32_t* atom_ptr, int64_t B, int64_t seed, const double* inv_mass,
                             const double* kT, const int64_t* sid, double* v, void* stream);
int m3g_debug_philox4x64(const int64_t* ctr, const int64_t* key, int64_t n, int64_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Domain decomposition helpers (new; nothing in the reference — nn/gradient.py:26 TODO)
 * ------------------------------------------------------------------------------------------- */
/* out[r] = in[idx[r]] rows of width W floats (halo pack) ; in[idx[r]] += add[r] (reverse halo unpack) */
int m3g_rows_gather(const float* in, const int32_t* idx, int64_t n, int W, float* out, void* stream);
int m3g_rows_scatter_add(const float* add, const int32_t* idx, int64_t n, int W, float* inout, void* stream);
/* halo push over NVLink / NVSwitch peer memory: row idx[r] (or r when idx == NULL) of `in` (rows of W floats; 16-byte
 * aligned rows when W % 4 == 0) is stored at the absolute device address dst_addr[r], typically a slot of a PEER
 * GPU's landing buffer (peer-mapped symmetric memory).  Pack + transfer in one kernel, no collective call; the caller
 * orders it against the consumer with a device-side barrier (domain.py::DomainStep, exchange = "p2p"). */
int m3g_rows_put(const float* in, const int32_t* idx, const int64_t* dst_addr, int64_t n, int W, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Whole-step executor (csrc/step.cu): the launch sequence of  Gradient(Sequential[ScaleLength, AtomRef,
 * DistanceAndAngle, AtomFeaturizer, EdgeFeaturizer, EdgeAdjustor, (ThreeBodyInteration, M3GNetConv) x n_blocks,
 * AtomWiseReadout])  (model/build.py:37-83, nn/gradient.py:25-64) — forward kernels, then the hand-written adjoint
 * kernels in reverse order, then forces + virial — issued from C with one call instead of ~70 Python round trips and
 * an autograd pass.  Default model shape only (F = 64, l_max = n_max = 3, radial degree 3, canonical triplet layout);
 * everything else stays on the per-operator entry points above.  All buffers are caller-owned device memory; the
 * struct itself lives in HOST memory.  The sequence is cut into phases so that a caller can interleave its own work
 * (the halo exchanges of a domain-decomposed cell, csrc/geometry.cu m3g_rows_*):
 *
 *   M3G_PHASE_PROLOGUE              scale, atom reference, geometry (+ cos), embedding, radial basis, e0, G / dG
 *   M3G_PHASE_TB(b), M3G_PHASE_CONV(b)      b = 0 .. n_blocks-1   (x of block b+1 is blocks[b].x_out)
 *   M3G_PHASE_READOUT(n)            energies; adjoint of the readout -> g_x
 *   M3G_PHASE_CONV_BWD(n,b), M3G_PHASE_TB_BWD(n,b)   b = n_blocks-1 .. 0   (the adjoint w.r.t. blocks[b].x_in is
 *                                   left in g_x[cur]; block 0 skips the dead gradient w.r.t. the embedding)
 *   M3G_PHASE_EPILOGUE(n)           e0 / radial / geometry adjoints -> g_pos
 *   M3G_PHASE_FORCES(n)             forces = -g_pos, virial stress
 * ------------------------------------------------------------------------------------------- */
#define M3G_STEP_MAX_BLOCKS 8
#define M3G_PHASE_PROLOGUE 0
#define M3G_PHASE_TB(b) (1 + 2 * (b))
#define M3G_PHASE_CONV(b) (2 + 2 * (b))
#define M3G_PHASE_READOUT(n) (1 + 2 * (n))
#define M3G_PHASE_CONV_BWD(n, b) (2 + 2 * (n) + 2 * ((n)-1 - (b)))
#define M3G_PHASE_TB_BWD(n, b) (3 + 2 * (n) + 2 * ((n)-1 - (b)))
#define M3G_PHASE_EPILOGUE(n) (2 + 4 * (n))
#define M3G_PHASE_FORCES(n) (3 + 4 * (n))

typedef struct M3GStepBlock {
  /* ThreeBodyInteration weights (nn/interaction.py:138-185): Ws (9,64), bs (9), WdT / WgT (9,64), tb_consts (20) */
  const float *Ws, *bs, *WdT, *WgT, *tb_consts;
  /* M3GNetConv weights (nn/conv.py:25-61): per-atom projection WpT (64,512) / bp (512) / Wp (512,64); per gated MLP
   * the tcgen05 weight images (m3g_tc_pack_b), second-layer biases and the (3,64) radial weights */
  const float *WpT, *bp, *Wp;
  const float *e_wimg, *e_wimgT, *e_b2d, *e_b2g, *e_WhT;
  const float *n_wimg, *n_wimgT, *n_b2d, *n_b2g, *n_WhT;
  /* activations: G / dG (E,9) radial tables (blocks with equal constants share them; radial_owner = 1 computes),
   * sig (N,9), red (E,9), x_in (N,64), e_in (E,64), e_tb (E,64), e_out (E,64), x_out (N,64), saved activations of
   * the two gated MLPs (ceil(E/128)*128*256 floats each) */
  float *G, *dG;
  int radial_owner;
  float *sig, *red;
  const float *x_in, *e_in;
  float *e_tb, *e_out, *x_out, *save_e, *save_n;
} M3GStepBlock;

typedef struct M3GStepDesc {
  int64_t N, E, T, B;
  int n_blocks, n_sm, passes, max_members;
  int64_t n_members; /* member bonds (bonds inside the three-body cutoff) */
  float length_scale, energy_scale, r3;
  int num_types;
  /* plan (int32 CSR views, see "Conventions") */
  const int32_t *batch, *src, *dst, *shift, *types, *edge_ptr, *in_ptr, *in_perm, *tri_ptr, *atom_ptr, *member_edges;
  const int64_t* tri_index; /* (2,T) caller-order list for the triplet_angles output, or NULL */
  /* inputs */
  const float *pos, *lattice;
  /* layer weights outside the blocks */
  const float *embed_W, *atomref_table, *radial_consts, *adjust_Wt;
  const float *ro_W0dT, *ro_b0d, *ro_W1dT, *ro_b1d, *ro_w2d, *ro_b2d, *ro_W0gT, *ro_b0g, *ro_W1gT, *ro_b1g, *ro_w2g,
      *ro_b2g, *ro_W0d, *ro_W1d, *ro_W0g, *ro_W1g;
  const float* g_total; /* (B) upstream gradient of the structure energies (ones; owned / ghost weights for a domain) */
  /* outputs / step-level activations */
  float *scaled_pos, *scaled_lattice, *elemental, *vec4, *dist, *cos_t, *x0, *h, *e0;
  float *atomic, *scaled_total, *total, *forces, *stresses;
  /* scratch */
  float *P, *msg;                 /* (N,512), (E,64) */
  float *g_x[2];                  /* (N,64) ping-pong; g_x[cur] holds the running adjoint */
  float *g_e[2], *ge2;            /* (E,64); ge2 may be NULL with fuse_conv_bwd */
  float *gz_edge, *gz_node, *gP;  /* (E,128) x 2, (N,512) */
  float *g_h, *g_hs, *g_sig_e, *g_vec4, *g_dist, *g_pos; /* (E,3), (2 n_blocks + 1, E, 3) per-launch slices, (E,9), (E,4), (E), (N,3) */
  int cur_x, cur_e;               /* state carried between phases (updated by m3g_step_run) */
  int have_g_e;                   /* 0 until the first conv adjoint has produced g_e */
  int msg_reduce;                 /* 1: node MLP sums its messages per atom in-kernel (m3g_conv_tc_fwd mode 2) */
  int tb_split;                   /* 1: three-body forward as m3g_tb_mom_red + m3g_tb_edge_update */
  int tb_bwd_split;               /* 1: three-body backward as m3g_tb_mlp_adj (q overwrites red) + m3g_tb_mom_bwd_q */
  int fuse_e0;                    /* 1 (needs tb_split): e0 is formed inside block 0's m3g_tb_edge_update_h, never stored */
  int fuse_conv_bwd;              /* 1: each block's node + edge MLP adjoints in one m3g_conv_tc_block_bwd (ge2 unused) */
  M3GStepBlock blocks[M3G_STEP_MAX_BLOCKS];
} M3GStepDesc;

/* run phases first .. last (inclusive) on `stream`; returns the first non-zero status */
int m3g_step_run(M3GStepDesc* desc, int first_phase, int last_phase, void* stream);
/* sizeof(M3GStepDesc) as compiled (binding self-check) */
int64_t m3g_step_desc_size(void);

#ifdef __cplusplus
}
#endif
#endif /* M3GNET_B200_H */
