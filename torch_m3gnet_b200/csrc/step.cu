// Whole-step executor: the launch sequence of the default M3GNet energy + forces call, issued from C (see the
// M3GStepDesc comment in include/m3gnet_b200.h).  Host code only: every launch goes through the per-operator C ABI, so
// the arithmetic is exactly that of the torch.autograd.Function path (torch_m3gnet_b200/nn/_functions.py); what
// disappears is the per-launch Python / ctypes / autograd cost (~1.3 ms per step, which dominates systems below a few
// thousand atoms and the per-rank sub-domains of a decomposed cell) and the dead gradient w.r.t. the embedding.
#include "common.cuh"

using namespace m3g;

#define M3G_TRY(call)            \
  do {                           \
    int rc__ = (call);           \
    if (rc__ != M3G_OK) return rc__; \
  } while (0)

namespace {

constexpr int F = 64, D = 9, R = 3, L = 3;

int prologue(M3GStepDesc* d, void* s) {
  M3G_TRY(m3g_scale_fwd(d->pos, d->scaled_pos, 3 * d->N, d->length_scale, s));
  M3G_TRY(m3g_scale_fwd(d->lattice, d->scaled_lattice, 9 * d->B, d->length_scale, s));
  M3G_TRY(m3g_atomref_fwd(d->atomref_table, d->types, d->N, d->elemental, s));
  M3G_TRY(m3g_geometry_fwd(d->scaled_pos, d->scaled_lattice, d->batch, d->src, d->dst, d->shift, d->E, d->vec4, d->dist,
                           s));
  if (d->tri_index && d->cos_t) M3G_TRY(m3g_angles_fwd(d->vec4, d->tri_index, d->T, d->cos_t, s));
  M3G_TRY(m3g_embed_fwd(d->embed_W, d->types, d->N, F, d->num_types, d->x0, s));
  M3G_TRY(m3g_radial_fwd(d->dist, d->radial_consts, d->E, R, d->h, s));
  if (!(d->fuse_e0 && d->tb_split)) M3G_TRY(m3g_edge_adjust_fwd(d->h, d->adjust_Wt, d->E, R, F, d->e0, s));
  for (int b = 0; b < d->n_blocks; ++b)
    if (d->blocks[b].radial_owner)
      M3G_TRY(m3g_tb_radial(d->vec4, d->blocks[b].tb_consts, d->E, L, R, d->member_edges, d->n_members, d->blocks[b].G,
                            d->blocks[b].dG, s));
  d->cur_x = 0;
  d->cur_e = 0;
  d->have_g_e = 0;
  return M3G_OK;
}

int tb_fwd(M3GStepDesc* d, int b, void* s) {
  M3GStepBlock& k = d->blocks[b];
  M3G_TRY(m3g_tb_sigma64_fwd(k.x_in, k.Ws, k.bs, d->N, d->n_sm, k.sig, s));
  if (d->tb_split) {
    M3G_TRY(m3g_tb_mom_red(d->vec4, k.G, k.sig, d->dst, d->edge_ptr, d->tri_ptr, d->r3, d->N, d->max_members, d->n_sm,
                           k.red, s));
    if (b == 0 && d->fuse_e0)
      M3G_TRY(m3g_tb_edge_update_h(k.red, d->tri_ptr, k.WdT, k.WgT, d->h, d->adjust_Wt, d->E, d->n_sm, k.e_tb, s));
    else
      M3G_TRY(m3g_tb_edge_update(k.red, d->tri_ptr, k.WdT, k.WgT, k.e_in, d->E, d->n_sm, k.e_tb, s));
  } else {
    M3G_TRY(m3g_tb_mom_fwd(d->vec4, k.G, k.sig, d->dst, d->edge_ptr, d->tri_ptr, d->r3, k.WdT, k.WgT, k.e_in, d->N,
                           d->max_members, d->n_sm, k.red, k.e_tb, s));
  }
  return M3G_OK;
}

int conv_fwd(M3GStepDesc* d, int b, void* s) {
  M3GStepBlock& k = d->blocks[b];
  M3G_TRY(m3g_linear_fwd(k.x_in, k.WpT, k.bp, d->N, F, 8 * F, d->P, s));
  M3G_TRY(m3g_conv_tc_fwd(d->P, 8 * F, 0, d->src, d->dst, k.e_tb, d->h, k.e_wimg, k.e_b2d, k.e_b2g, k.e_WhT, d->E, R, 0,
                          d->passes, d->n_sm, k.e_out, k.save_e, s));
  // mode 2: messages reduced per source atom in the kernel's epilogue (one partial row per 32-row block and atom)
  M3G_TRY(m3g_conv_tc_fwd(d->P, 8 * F, 4 * F, d->src, d->dst, k.e_out, d->h, k.n_wimg, k.n_b2d, k.n_b2g, k.n_WhT, d->E,
                          R, d->msg_reduce ? 2 : 1, d->passes, d->n_sm, d->msg, k.save_n, s));
  if (d->msg_reduce) M3G_TRY(m3g_segment_sum_parts(k.x_in, d->msg, d->edge_ptr, d->N, F, k.x_out, s));
  else M3G_TRY(m3g_segment_sum_add(k.x_in, d->msg, d->edge_ptr, d->N, F, k.x_out, s));
  return M3G_OK;
}

int readout(M3GStepDesc* d, void* s) {
  const float* x = d->blocks[d->n_blocks - 1].x_out;
  // forward and adjoint in one launch: the upstream gradient g_total is an input of the step
  M3G_TRY(m3g_readout_fwd_bwd(x, d->ro_W0dT, d->ro_b0d, d->ro_W1dT, d->ro_b1d, d->ro_w2d, d->ro_b2d, d->ro_W0gT,
                              d->ro_b0g, d->ro_W1gT, d->ro_b1g, d->ro_w2g, d->ro_b2g, d->ro_W0d, d->ro_W1d, d->ro_W0g,
                              d->ro_W1g, d->elemental, d->g_total, d->batch, d->energy_scale, d->N, F, d->atomic,
                              d->g_x[0], s));
  M3G_TRY(m3g_structure_sum(d->atomic, d->atom_ptr, d->B, d->energy_scale, d->scaled_total, d->total, s));
  d->cur_x = 0;
  d->cur_e = 0;
  d->have_g_e = 0;
  return M3G_OK;
}

int conv_bwd(M3GStepDesc* d, int b, void* s) {
  M3GStepBlock& k = d->blocks[b];
  const bool need_x = b > 0;  // x of block 0 is the embedding: no dependence on the positions
  const float* g_x2 = d->g_x[d->cur_x];
  const float* g_e2 = d->have_g_e ? d->g_e[d->cur_e] : nullptr;
  float* g_e_new = d->g_e[d->have_g_e ? (d->cur_e ^ 1) : 0];
  // every backward launch stores its radial-weight adjoint into its own slice; the epilogue sums the slices
  float* gh_node = d->g_hs + (int64_t)(2 * (d->n_blocks - 1 - b)) * R * d->E;
  float* gh_edge = gh_node + (int64_t)R * d->E;
  if (d->fuse_conv_bwd) {
    M3G_TRY(m3g_conv_tc_block_bwd(d->src, d->h, k.n_wimgT, k.n_WhT, k.save_n, k.e_wimgT, k.e_WhT, k.save_e, g_x2, g_e2,
                                  d->E, R, d->passes, d->n_sm, g_e_new, need_x ? d->gz_node : nullptr,
                                  need_x ? d->gz_edge : nullptr, gh_node, gh_edge, 0, s));
  } else {
    M3G_TRY(m3g_conv_tc_bwd_saved(d->src, d->h, k.n_wimgT, k.n_WhT, k.save_n, g_x2, g_e2, d->E, R, 1, d->passes,
                                  d->n_sm, d->ge2, need_x ? d->gz_node : nullptr, gh_node, 1, s));
    M3G_TRY(m3g_conv_tc_bwd_saved(d->src, d->h, k.e_wimgT, k.e_WhT, k.save_e, d->ge2, d->ge2, d->E, R, 0, d->passes,
                                  d->n_sm, g_e_new, need_x ? d->gz_edge : nullptr, gh_edge, 1, s));
  }
  d->cur_e = d->have_g_e ? (d->cur_e ^ 1) : 0;
  d->have_g_e = 1;
  if (need_x) {
    M3G_TRY(m3g_conv_gather_gz(d->gz_edge, d->edge_ptr, d->in_ptr, d->in_perm, d->N, F, 8 * F, 0, d->gP, s));
    M3G_TRY(m3g_conv_gather_gz(d->gz_node, d->edge_ptr, d->in_ptr, d->in_perm, d->N, F, 8 * F, 4 * F, d->gP, s));
    M3G_TRY(m3g_linear_bwd_input(d->gP, k.Wp, g_x2, d->N, F, 8 * F, d->g_x[d->cur_x ^ 1], s));
    d->cur_x ^= 1;
  }
  return M3G_OK;
}

int tb_bwd(M3GStepDesc* d, int b, void* s) {
  M3GStepBlock& k = d->blocks[b];
  const bool need_x = b > 0;
  if (d->tb_bwd_split) {
    // q = dL/dred overwrites this block's red (dead after this phase)
    M3G_TRY(m3g_tb_mlp_adj(k.red, d->g_e[d->cur_e], d->member_edges, d->n_members, k.WdT, k.WgT, d->n_sm, k.red, s));
    M3G_TRY(m3g_tb_mom_bwd_q(d->vec4, k.G, k.dG, k.sig, d->dst, k.red, d->edge_ptr, d->tri_ptr, d->r3, d->N,
                             d->max_members, d->n_sm, b != d->n_blocks - 1, d->g_vec4, d->g_sig_e, s));
  } else {
    M3G_TRY(m3g_tb_mom_bwd(d->vec4, k.G, k.dG, k.sig, d->dst, k.red, d->g_e[d->cur_e], d->edge_ptr, d->tri_ptr, d->r3,
                           k.WdT, k.WgT, d->N, d->max_members, d->n_sm, b != d->n_blocks - 1, d->g_vec4, d->g_sig_e, s));
  }
  if (need_x) {
    M3G_TRY(m3g_tb_sigma64_bwd(d->g_sig_e, d->in_ptr, d->in_perm, k.sig, k.Ws, d->g_x[d->cur_x], d->N, d->n_sm,
                               d->g_x[d->cur_x ^ 1], s));
    d->cur_x ^= 1;
  }
  return M3G_OK;
}

int epilogue(M3GStepDesc* d, void* s) {
  M3G_TRY(m3g_edge_adjust_bwd(d->h, d->adjust_Wt, d->g_e[d->cur_e], d->E, R, F,
                              d->g_hs + (int64_t)(2 * d->n_blocks) * R * d->E, s));
  M3G_TRY(m3g_sum_slices(d->g_hs, 2 * d->n_blocks + 1, (int64_t)R * d->E, d->g_h, s));
  M3G_TRY(m3g_radial_bwd(d->dist, d->radial_consts, d->g_h, d->E, R, d->g_dist, s));
  M3G_TRY(m3g_geometry_bwd(d->vec4, d->g_vec4, d->g_dist, d->edge_ptr, d->in_ptr, d->in_perm, d->N,
                           1.0f / d->length_scale, d->g_pos, s));
  return M3G_OK;
}

}  // namespace

extern "C" {

int64_t m3g_step_desc_size(void) { return (int64_t)sizeof(M3GStepDesc); }

int m3g_step_run(M3GStepDesc* d, int first_phase, int last_phase, void* stream) {
  M3G_REQUIRE(d != nullptr, "m3g_step_run: null descriptor");
  const int n = d->n_blocks;
  M3G_REQUIRE(n >= 1 && n <= M3G_STEP_MAX_BLOCKS, "m3g_step_run: n_blocks=%d outside [1,%d]", n, M3G_STEP_MAX_BLOCKS);
  M3G_REQUIRE(d->N > 0 && d->E > 0 && d->B > 0, "m3g_step_run: empty batch (use the per-operator path)");
  M3G_REQUIRE(first_phase >= 0 && last_phase <= M3G_PHASE_FORCES(n) && first_phase <= last_phase,
              "m3g_step_run: phases %d..%d outside [0,%d]", first_phase, last_phase, M3G_PHASE_FORCES(n));
  for (int ph = first_phase; ph <= last_phase; ++ph) {
    if (ph == M3G_PHASE_PROLOGUE) {
      M3G_TRY(prologue(d, stream));
    } else if (ph < M3G_PHASE_READOUT(n)) {
      const int b = (ph - 1) / 2;
      if ((ph - 1) % 2 == 0) M3G_TRY(tb_fwd(d, b, stream));
      else M3G_TRY(conv_fwd(d, b, stream));
    } else if (ph == M3G_PHASE_READOUT(n)) {
      M3G_TRY(readout(d, stream));
    } else if (ph < M3G_PHASE_EPILOGUE(n)) {
      const int q = ph - (2 + 2 * n);
      const int b = n - 1 - q / 2;
      if (q % 2 == 0) M3G_TRY(conv_bwd(d, b, stream));
      else M3G_TRY(tb_bwd(d, b, stream));
    } else if (ph == M3G_PHASE_EPILOGUE(n)) {
      M3G_TRY(epilogue(d, stream));
    } else {
      M3G_TRY(m3g_forces_virial(d->pos, d->g_pos, d->lattice, d->atom_ptr, d->N, d->B, d->forces, d->stresses, stream));
    }
  }
  return M3G_OK;
}

}  // extern "C"
