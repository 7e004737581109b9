/* codlad_b200 -- C ABI of the B200-native reverse latent-diffusion sampling path of CODLAD.
 *
 * Plain C: opaque handles, raw pointers and sizes, no torch types.  Every function returns 0 on
 * success or a non-zero cudaError_t / error code; cb2_last_error() gives the message (thread-local).
 * Unless a parameter says "host", pointers are DEVICE pointers owned by the caller (inputs are
 * borrowed for the duration of the call, never retained or freed); `stream` is a cudaStream_t passed
 * as void* and all work is enqueued on it (no internal threads, no hidden synchronisation except in
 * the *_create / set_* functions that upload host data).
 *
 * The reference (xiaoxiaokuye/CODLAD) has no FFI layer: its boundary is the Python call surface.  Each
 * entry point below names the reference call it replaces; codlad_b200/*.py binds them with ctypes
 * behind the reference's own signatures (see INTEGRATION.md).
 */
#ifndef CODLAD_B200_H
#define CODLAD_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CB2_API __attribute__((visibility("default")))
#else
#define CB2_API
#endif

#define CB2_ABI_VERSION 4
#define CB2_PRECISION_F32 0   /* fp32 SIMT tier: tracks the fp32 reference to ~1e-6 */
#define CB2_PRECISION_F16 1   /* tcgen05 tier: fp16 operands / edge state, fp32 accumulation in TMEM */
#define CB2_MOD_WIDTH 6016    /* adaLN table row: 3*1152 (enc) + 3*768 (dec) + 256 (final) */

typedef struct cb2_denoiser cb2_denoiser;   /* packed weights of ProteinMPNN_diffusion_new */
typedef struct cb2_vae cb2_vae;             /* codebook + map_out + IC decoder weights */
typedef struct cb2_plan cb2_plan;           /* buffers + graph for one batch geometry */

typedef struct {
    const char* name;        /* reference state_dict key, e.g. "encoder_layers.0.W1.weight" */
    const float* data;       /* HOST pointer, fp32, contiguous, reference layout */
    long long numel;
} cb2_tensor;

CB2_API int cb2_abi_version(void);
CB2_API const char* cb2_last_error(void);

/* ---- model objects ------------------------------------------------------------------------- */

/* Replaces: MPNN_models['mpnn_diffusion'](...) + load_state_dict (models/latent_model.py:78-165,276-281;
 * test.py:262-288).  `tensors` = the 108 state_dict entries (host).  `freqs128` (host) = the sinusoid
 * frequencies exp(-ln(1e4) k/128) as the caller's torch computes them (latent_model.py:59-61). */
CB2_API int cb2_denoiser_create(const cb2_tensor* tensors, int n_tensors, const float* freqs128, int k_neighbors,
                        cb2_denoiser** out);
CB2_API void cb2_denoiser_destroy(cb2_denoiser* m);

/* Replaces: the decode-side state of get_vae_model (utils/model_module.py:20-123): quantize._codebook.embed,
 * map_out.*, equivaraintconv.* (IC_Decoder or, angle_variant=1, IC_Decoder_angle), and the latent
 * mean/std 3-vectors of datasets/miu_and_sigma/ (utils/dataset_module.py:248-249).  All host pointers. */
CB2_API int cb2_vae_create(const cb2_tensor* tensors, int n_tensors, const float* mean3, const float* std3,
                   int angle_variant, cb2_vae** out);
CB2_API void cb2_vae_destroy(cb2_vae* v);

/* ---- plan: one batch geometry ------------------------------------------------------------------
 * F frames (distinct C-alpha traces) padded to L residues, NB batch members; member b denoises over
 * frame frame_of[b] (an ensemble = several members on one frame).  K = min(k_neighbors, L).
 * m may be NULL: a decode-only plan (set_frames / set_topology / decode work; forward / sample refuse). */
CB2_API int cb2_plan_create(const cb2_denoiser* m, int F, int NB, int L, int precision, int keep_debug, cb2_plan** out);
CB2_API void cb2_plan_destroy(cb2_plan* p);
CB2_API int cb2_plan_K(const cb2_plan* p);
CB2_API long long cb2_plan_launches(const cb2_plan* p);   /* kernels launched through this plan so far */

/* Replaces: CA_ProteinFeatures.forward + W_e (models/protein_mpnn_utils.py:447-523, latent_model.py:208,216),
 * hoisted out of the step loop: k-NN graph, edge features and h_E0 for every frame.
 * X [F,L,3] fp32 (zero beyond each frame's length), lengths [F] int32, cg_z [F,L] int32, frame_of [NB] int32. */
CB2_API int cb2_plan_set_frames(cb2_plan* p, const float* X, const int* lengths, const int* cg_z, const int* frame_of,
                        void* stream);

/* Replaces: ProteinMPNN_diffusion_new.forward (models/latent_model.py:175-268) for the geometry set above.
 * x [NB,L,3], t [NB] fp32 timesteps (already mapped to the original 0..999 scale) -> out [NB,L,6]. */
CB2_API int cb2_plan_forward(cb2_plan* p, const float* x, const float* t, float* out, void* stream);

/* Debug / parity: the first `stop_after` kernels of cb2_plan_forward (1 = node init, then per encoder layer
 * node-message, node-update, edge-update; then per decoder layer message, node-update); inspect the state with
 * cb2_plan_buffer. */
CB2_API int cb2_plan_forward_partial(cb2_plan* p, const float* x, const float* t, int stop_after, void* stream);

/* Replaces: SpacedDiffusion/GaussianDiffusion coefficient tables + _WrappedModel timestep remap
 * (diffusion_and_flow/respace.py:73-129, gaussian_diffusion.py:175-209).  HOST arrays: t_of_step [T] =
 * timestep_map, coef [T][8] = {posterior_log_variance_clipped, log(beta), sqrt(1/acp), sqrt(1/acp - 1),
 * posterior_mean_coef1, posterior_mean_coef2, (step != 0), 0} as fp32.  Builds the [T, 6016] adaLN table. */
CB2_API int cb2_plan_set_schedule(cb2_plan* p, const float* t_of_step, const float* coef, int T, void* stream);

/* DDIM counterpart of cb2_plan_set_schedule (IDDPM gaussian_diffusion.py ddim_sample, clip_denoised=False; the reference
 * itself has no DDIM sampler).  HOST arrays: t_of_step [T] = timestep_map, ddim_coef [T][8] = {sqrt(1/acp), sqrt(1/acp - 1),
 * sqrt(acp_prev), sqrt(max(0, 1 - acp_prev - sigma^2)), sigma * (step != 0), 0, 0, 0} as fp32, with
 * sigma = eta sqrt((1 - acp_prev) / (1 - acp)) sqrt(1 - acp / acp_prev).  Builds the adaLN table; cb2_plan_sample then applies
 * the DDIM update until the next cb2_plan_set_schedule. */
CB2_API int cb2_plan_set_ddim_schedule(cb2_plan* p, const float* t_of_step, const float* ddim_coef, int T, void* stream);

/* Replaces: GaussianDiffusion.p_sample_loop (gaussian_diffusion.py:451-547): T denoiser forwards + p_sample
 * updates, steps T-1 .. 0.  x [NB,L,3] in/out; noise [T,NB,L,3] (noise[s] is used at step s; the reference
 * draws it with randn_like at :440).  use_graph != 0 captures the whole loop in one CUDA graph and replays it.
 * After cb2_plan_set_ddim_schedule the updates are DDIM steps; noise may then be NULL when every sigma is zero (eta = 0).
 * With inpainting on (cb2_plan_set_inpaint) the kept rows follow their latent and T must equal the inpainting table's. */
CB2_API int cb2_plan_sample(cb2_plan* p, float* x, const float* noise, int use_graph, void* stream);

/* Latent inpainting for the following cb2_plan_sample calls (the replacement method; the reference has no such sampler):
 * the rows marked in keep [NB*L] (u8, non-zero = keep) follow their normalised latent x0 [NB,L,3], every other row is
 * regenerated, conditioned on the kept ones through the denoiser.  With eps = the kept rows of the initial noise x, a kept
 * row starts at q_coef[T] and after the update of step s is overwritten with q_coef[s], where a row {a, b} means
 * a * x0 + b * eps (fp32, two rounded products and one rounded sum).  q_coef [T+1][2] is a HOST array:
 * rows 0..T-1 = {sqrt(acp_prev), sqrt(1 - acp_prev)} of each step, row T = {sqrt(acp[T-1]), sqrt(1 - acp[T-1])}, so that
 * kept rows end at x0 exactly.  It serves DDPM and DDIM schedules alike.  keep and x0 are copied into plan-owned buffers
 * (x0 may therefore be the x later passed to cb2_plan_sample); new contents need no graph recapture.  keep == NULL turns
 * inpainting off (x0 and q_coef are then ignored).  Each sample call with inpainting on launches one more kernel. */
CB2_API int cb2_plan_set_inpaint(cb2_plan* p, const unsigned char* keep, const float* x0, const float* q_coef, int T,
                         void* stream);

/* Decode-side geometry.  ca_full [F,L+2,3] device (untrimmed trace); HOST OR DEVICE (copied with
 * cudaMemcpyDefault): csr_row_ptr [F*L+1] / csr_col [E]
 * = directed 21 A radius graph per frame (local column indices; make_directed, models/gcn_nn.py:54-64),
 * atom_orders [F,L,10,3] int8 and slot_atom [F,L*14] int32 (inverse of info's atom_idx[permute],
 * utils/protein_module.py:455-494), out_offset [NB] int64 = first output atom row of each member. */
CB2_API int cb2_plan_set_topology(cb2_plan* p, const cb2_vae* v, const float* ca_full, const int* csr_row_ptr,
                          const int* csr_col, int n_edges, const signed char* atom_orders, const int* slot_atom,
                          const long long* out_offset, void* stream);

/* Replaces: get_norm_feature(norm_in=False) + VAE.latent_decode + ic_to_xyz (test.py:548-582;
 * utils/dataset_module.py:230-256; models/vae_model.py:830-839; utils/utils_ic.py:242-268).
 * latent [NB,L,3]; denorm != 0 applies x*std+mean first.  Outputs (any may be NULL): idx [NB,L] int32 (-1 at
 * padded positions), zq [NB,L,3], ic_recon [NB,L,13,3], xyz [sum Na,3]. */
CB2_API int cb2_plan_decode(cb2_plan* p, const cb2_vae* v, const float* latent, int denorm, int* idx, float* zq,
                    float* ic_recon, float* xyz, void* stream);

/* Not in the reference: per-residue form of clash_result's criterion (test.py:118-139) on a decoded sample, with no reference
 * structure and no dataset pair lists.  xyz [sum Na,3] is laid out as cb2_plan_decode writes it (slot_atom / out_offset of
 * cb2_plan_set_topology, which must have been called).  counts [NB*L] int32: counts[b*L+i] = number of atom pairs (a in residue
 * i, c in another residue j of member b) with d(a, c) < threshold, where d = sqrt(|a - c|^2 + 1e-7) in fp32 exactly as
 * cb2_pair_losses forms it, leaving out the peptide pair C(i)-N(i+1) (slots 2 and 1); a pair counts once for each of its two
 * residues; padded rows get 0.  Every pair is tested (bounding-sphere pruning that never drops one), so the counts equal a
 * brute-force pass.  keep [NB*L] u8 or NULL: 0 where residue i or one of its `grow` nearest other residues (the plan's k-NN
 * rows, distance order) has a clash, 1 elsewhere and on padded rows -- the keep mask of cb2_plan_set_inpaint that resamples the
 * clashing residues.  threshold must be finite and positive (the reference uses 1.2 A), 0 <= grow < K (grow = 0 on a decode-only
 * plan).  Deterministic; two launches, three with keep. */
CB2_API int cb2_plan_residue_clashes(cb2_plan* p, const float* xyz, float threshold, int grow, int* counts, unsigned char* keep,
                             void* stream);

/* Debug / parity access to plan-owned buffers: "nbr_idx" "nbr_dist" "E" "hE0" "hE" "hV" "S" "out6" "mod".
 * Copies the first dst_bytes of the buffer into the caller's device memory (error if it is smaller). */
CB2_API int cb2_plan_buffer(cb2_plan* p, const char* name, void* dst, long long dst_bytes, void* stream);

/* Measurement hook (bench.py roofline): launches ONE per-edge kernel of the denoiser on the plan's current
 * state.  mode 0 = encoder node message, 1 = encoder edge update, 2 = decoder message; layer 0..2. */
CB2_API int cb2_plan_run_edge_kernel(cb2_plan* p, int mode, int layer, void* stream);

/* Measurement hook (bench.py roofline_all): launches ONE stage of the path on the plan's current buffers, exactly as the
 * step loop / the per-frame precompute / the decode launch it (results land in the plan's own buffers and are not meant to be
 * read).  stage: 0-2 = per-edge kernels as above; 3 = node update of phase `layer` (0-2 encoder, 3-5 decoder, 5 includes
 * FinalLayer + p_sample; reference protein_mpnn_utils.py:247-259,307-317); 4 = k-NN graph (:447-459); 5 = edge featuriser
 * (:369-523); 6 = de-normalise + VQ lookup + map_out (vae_model.py:835); 7 = IC decoder (vae_model.py:467-503); 8 = ic_to_xyz
 * (utils_ic.py:242-268, needs `xyz_scratch` of [total atoms, 3]); 9 = IC distance filters (gcn_nn.py:222-338).
 * Stages 6-9 need cb2_plan_set_topology. */
CB2_API int cb2_plan_run_stage(cb2_plan* p, const cb2_vae* v, int stage, int layer, float* xyz_scratch, void* stream);

/* ---- stand-alone kernels (same code the plan uses) ---------------------------------------------- */

/* Replaces: CA_ProteinFeatures._dist (protein_mpnn_utils.py:447-459).  D [F,L,K] fp32, idx [F,L,K] int32,
 * sorted ascending by (distance, index).  lengths may be NULL (all L valid). */
CB2_API int cb2_knn_topk(const float* X, const int* lengths, int F, int L, int K, float* D, int* idx, void* stream);

/* Replaces: VectorQuantize.forward eval (vae_model.py:835) for N = NB*L rows with per-frame lengths. */
CB2_API int cb2_vq_lookup(const cb2_vae* v, const float* x, int NB, int L, const int* lengths, const int* frame_of,
                  int denorm, int* idx, float* zq, void* stream);

/* Replaces: one p_sample update (gaussian_diffusion.py:404-449) on a model output the caller produced.
 * x, noise, x_next [rows,C]; model_out [rows,2C]; coef [T,8] device; step_of_member [NB] int32 device;
 * rows = NB*rows_per_member. */
CB2_API int cb2_p_sample(const float* x, const float* model_out, const float* noise, const float* coef,
                 const int* step_of_member, int rows_per_member, int rows, int C, float* x_next, void* stream);

/* One DDIM update (IDDPM ddim_sample, clip_denoised=False) on a model output the caller produced; same conventions as
 * cb2_p_sample with coef = the [T,8] rows of cb2_plan_set_ddim_schedule.  noise may be NULL (no noise term). */
CB2_API int cb2_ddim_sample(const float* x, const float* model_out, const float* noise, const float* coef,
                 const int* step_of_member, int rows_per_member, int rows, int C, float* x_next, void* stream);

/* Replaces: ic_to_xyz (utils_ic.py:242-268) alone; same conventions as cb2_plan_set_topology but all DEVICE. */
CB2_API int cb2_ic_to_xyz(const float* ca_full, const float* ic_recon, int NB, int L, const int* frame_of,
                  const int* lengths, const signed char* atom_orders, const int* slot_atom,
                  const long long* out_offset, float* xyz, void* stream);

/* ---- evaluation step right after the path (SURVEY.md section 8f-4) --------------------------------------------------
 * Replaces: eval_sample_qualities / count_valid_graphs / get_bond_graphs / compute_rmsd (utils/protein_module.py:245-364),
 * called per structure by valid_ratio_and_cut_off_result (test.py:168-188) with two dense [Na, Na] matrices on the CPU.
 * All pointers are DEVICE: xyz_ref / xyz_gen [sum Na, 3], atomic_num [sum Na], offsets [n_struct + 1] (atom ranges of the
 * structures), cov_radius [max_z + 1] (COVCUTOFFTABLE, protein_module.py:128); max_atoms = the largest structure.  Outputs:
 *   counts [n_struct, 6] = {differing adjacency entries, reference bonds, generated bonds} over all atoms, then over heavy atoms
 *   sums   [n_struct, 4] = {sum ||x_gen - x_ref||^2 over all atoms, Na, the same over heavy atoms, number of heavy atoms}
 * bond(i, j) = i != j and ||x_i - x_j|| < (r[z_i] + r[z_j]) * scale in fp32, entries counted over the full symmetric matrix. */
CB2_API int cb2_eval_bond_graphs(const float* xyz_ref, const float* xyz_gen, const int* atomic_num, const long long* offsets, int n_struct,
                         int max_atoms, const float* cov_radius, int max_z, float scale, long long* counts, double* sums, void* stream);

/* Replaces: md.rmsd(Trajectory(a), Trajectory(b)) as the diversity score uses it (compute_rmsd_ref / compute_rmsd_gen / compute_div,
 * test.py:37-96): the minimum RMSD under rigid superposition of structure pairs.  A, B [sum Na, 3] DEVICE (pair s = atoms
 * offsets[s] .. offsets[s+1] of both), out [n_struct] double.  Sums in double, largest eigenvalue of Horn's quaternion matrix.
 * mdtraj is absent from the build container: parity is against a float64 Kabsch (SVD) restatement, i.e. unpinned against mdtraj itself. */
CB2_API int cb2_superposed_rmsd(const float* A, const float* B, const long long* offsets, int n_struct, double* out, void* stream);

/* Replaces: the pair-list reductions of inter_result / clash_result / ged_result (test.py:97-146).  xyz [Na, 3] DEVICE; xyz_data the
 * reference coordinates (DEVICE) or NULL; idx [n_rows, width] int64 DEVICE, width 2 = atom pairs, width 4 = (a, b, c, e) quads whose
 * distance is between the centres (x_a + x_b)/2 and (x_c + x_e)/2 (pi-pi stacking, test.py:113-116).  d = sqrt(|.|^2 + 1e-7) in fp32.
 * out4 (DEVICE, double): {#(d < thr_count), sum max(d - thr_hinge, 0), sum (d - d_data)^2 (0 without xyz_data), n_rows}. */
CB2_API int cb2_pair_losses(const float* xyz, const float* xyz_data, const long long* idx, int width, long long n_rows, float thr_count,
                    float thr_hinge, double* out4, void* stream);

/* Replaces: the `uniques[counts == 1]` selection of clash_result (test.py:121-123) on a SORTED int64 key list (key = a * Na + b):
 * once[i] = 1 where the key occurs exactly once.  DEVICE pointers. */
CB2_API int cb2_keys_once(const long long* sorted_keys, long long n, unsigned char* once, void* stream);

#ifdef __cplusplus
}
#endif
#endif
