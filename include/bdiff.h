/*
 * bdiff.h — C ABI of libbdiff_sm100.so: the B200-native GCPNet denoiser hot path of GCDM.
 *
 * The reference (BioinfoMachineLearning/bio-diffusion) has no FFI for this path; its seam is the Python
 * class contract `dynamics_network.forward(batch, xh, t) -> (batch, net_out)` selected in
 * src/models/qm9_mol_gen_ddpm.py:101-105,125-131 (and geom_mol_gen_ddpm.py) and called from
 * src/models/components/variational_diffusion.py:873,1042,1116,1236.  The entry points below are what a
 * binding for that seam needs; each cites the reference interface it replaces.  Host mirror:
 * bio-diffusion_b200/bdiff/dynamics.py (class GCPNetDynamicsB200); binding recipe: INTEGRATION.md.
 *
 * Conventions
 *   - plain C, no torch types; every data pointer is a DEVICE pointer owned by the caller unless the name
 *     ends in _host; float = fp32, indices int64 at the boundary (like the reference), mask = uint8 (0/1);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); nothing synchronises the
 *     device except bdiff_plan_topology (one D2H of batch_index/mask + one H2D of the plan);
 *   - return 0 on success, a negative BDIFF_E* code otherwise; never throws; bdiff_last_error(h) gives text;
 *   - one handle per (device, stream); not thread-safe; the handle owns packed weights and workspace.
 */
#ifndef BDIFF_H_
#define BDIFF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BDIFF_OK 0
#define BDIFF_EINVAL (-1)   /* bad argument / unsupported configuration            */
#define BDIFF_ECUDA (-2)    /* a CUDA runtime call or kernel launch failed         */
#define BDIFF_ESTATE (-3)   /* call order violated (weights missing, no plan, ...) */
#define BDIFF_ENOMEM (-4)

#define BDIFF_ABI_VERSION 1

#if defined(__GNUC__)
#define BDIFF_API __attribute__((visibility("default")))
#else
#define BDIFF_API
#endif

/* Compute modes.  PARITY: every multiply-add in fp32 FFMA (differs from the reference only by
 * summation order).  TENSOR: the per-edge message GEMMs run on tcgen05 tensor cores
 * (operands rounded to the tensor format, fp32 accumulation in TMEM). */
#define BDIFF_MODE_PARITY_FP32 0
#define BDIFF_MODE_TENSOR 1

typedef struct bdiff_handle bdiff_handle;

/* Dims of the denoiser; mirrors what GCPNetDynamics.__init__ derives from its five Hydra configs
 * (src/models/components/gcpnet.py:933-1039).  Only the shipped option set is supported (GCP2,
 * vector_gate, no frame_gate, bottleneck 4, 4 residual message GCPs, scalar message attention, one
 * feed-forward GCP, no GCP norm / dropout, no self-conditioning); anything else -> BDIFF_EINVAL. */
typedef struct bdiff_config {
  int32_t num_h;          /* F: node scalar features in xh = [x(3) | h(F)] = num_atom_types + include_charges */
  int32_t num_context;    /* len(module_cfg.conditioning): context columns appended after the time column     */
  int32_t num_layers;     /* model_cfg.num_encoder_layers (9 QM9, 4 GEOM)                                      */
  int32_t h_hidden;       /* model_cfg.h_hidden_dim   — must be 256                                            */
  int32_t chi_hidden;     /* model_cfg.chi_hidden_dim — must be 32                                             */
  int32_t e_hidden;       /* model_cfg.e_hidden_dim   (64 QM9, 16 GEOM), multiple of 4, <= 64                   */
  int32_t xi_hidden;      /* model_cfg.xi_hidden_dim  (16 QM9, 8 GEOM), multiple of 4, <= 16                    */
  int32_t mode;           /* BDIFF_MODE_*                                                                       */
} bdiff_config;

BDIFF_API int32_t bdiff_abi_version(void);

/* Replaces: GCPNetDynamics.__init__ (gcpnet.py:933-1039) — allocates packed-weight storage. */
BDIFF_API int32_t bdiff_create(const bdiff_config* cfg, bdiff_handle** out);
BDIFF_API void bdiff_destroy(bdiff_handle* h);
BDIFF_API const char* bdiff_last_error(const bdiff_handle* h);   /* h may be NULL: last creation error */

/* Replaces: nn.Module.load_state_dict on the reference module.  `name` is the reference parameter name
 * relative to the denoiser (e.g. "interaction_layers.3.interaction.message_fusion.0.scalar_out.weight"),
 * `data` a contiguous fp32 device tensor of `shape`.  The tensor is repacked (transposed to K-major,
 * split, zero-padded) into the kernel layout immediately on `stream`; the caller may free it afterwards. */
BDIFF_API int32_t bdiff_set_weight(bdiff_handle* h, void* stream, const char* name, const float* data,
                         const int64_t* shape, int32_t ndim);
/* Number of reference parameter tensors still missing (0 = ready); -errno on error. */
BDIFF_API int32_t bdiff_weights_missing(const bdiff_handle* h);

/* Finishes weight preparation once every parameter is set (tensor mode: builds the pre-swizzled bf16 weight
 * K-blocks the TMA producer streams).  Called by the host after load_state_dict so that nothing but the forward
 * kernels runs inside a captured CUDA graph.  Idempotent. */
BDIFF_API int32_t bdiff_prepare(bdiff_handle* h, void* stream);

/* Hardware self test of the split-bf16 machinery of the tensor mode (csrc/bdiff_selftest.cu): hi/lo A blocks,
 * un-swizzled K=16 weight slabs, three (variant bit 1: four, node-tile row views) products per K step, TMEM pair
 * exchange.  C[128,336] <- [A W^T (320 cols; the last 32 negated) | exchange (16 cols)] for A fp32[128,128],
 * W fp32[320,128] (device pointers).  variant bit 0 swaps LBO/SBO (must then FAIL the comparison).  Synchronises. */
BDIFF_API int32_t bdiff_selftest_split(void* stream, int32_t variant, const float* A, const float* W, float* C);

/* Hardware self test of the CTA-pair (cta_group::2) machinery: a two-CTA cluster, TMEM allocated for the pair, every weight
 * plane split between the two shared memories, the peer's TMA completion relayed by a remote mbarrier arrive, one commit
 * multicast to both CTAs.  C[256,320] <- A W^T for A fp32[256,128], W fp32[320,128] (device pointers), split-bf16 operands.
 * Synchronises. */
BDIFF_API int32_t bdiff_selftest_pair(void* stream, const float* A, const float* W, float* C);

/* Weight-stream layout of one layer's edge pass in tensor mode, for edge / xi hidden sizes (e_hidden, xi_hidden); no GPU
 * needed.  out[0] = bytes packed per layer, out[1] = TMA chunks per CTA and edge tile (streamed by the producer lane,
 * relayed by the peer CTA), out[2] = bytes of those chunks summed over both CTAs (must equal out[0]).  Returns
 * BDIFF_EINVAL for sizes the tensor mode does not support. */
BDIFF_API int32_t bdiff_tc_edge_stream_layout(int32_t e_hidden, int32_t xi_hidden, int64_t* out);

/* Replaces: GCPNetDynamics.get_fully_connected_edge_index (gcpnet.py:1054-1066) — as an implicit plan.
 * batch_index int64[N] (sorted molecule ids, as every caller provides), mask uint8[N].  Builds the
 * per-molecule offsets the kernels enumerate edges from; *num_edges_host receives E = sum_k nact_k^2.
 * Synchronises `stream` (one small D2H + H2D).  Re-plan whenever batch_index / mask change. */
BDIFF_API int32_t bdiff_plan_topology(bdiff_handle* h, void* stream, int32_t num_mols, int64_t num_nodes,
                            const int64_t* batch_index, const uint8_t* mask, int64_t* num_edges_host);

/* Materialises the reference's edge_index int64[2,E] ((row,col)-sorted, self loops, masked nodes dropped)
 * from the current plan — only for callers/tests that want it; the kernels never read it. */
BDIFF_API int32_t bdiff_edge_index(bdiff_handle* h, void* stream, int64_t* edge_index);

/* Replaces: GCPNetDynamics.forward / atom_types_and_coords_forward (gcpnet.py:1042-1052, 1069-1232).
 * xh fp32[N,3+F], t fp32[N] (per node, the reference's t[batch_index]), context fp32[N,C] or NULL,
 * net_out fp32[N,3+F] = [vel (CoG-free) | h_final].  xh is not modified. */
BDIFF_API int32_t bdiff_denoise_forward(bdiff_handle* h, void* stream, const float* xh, const float* t,
                              const float* context, float* net_out);

/* Same as bdiff_denoise_forward, but records CUDA events on `stream` around every kernel class and, after
 * synchronising the stream, writes milliseconds to ms_host[0..6] = {prep+node_frames, edge_embed, node_embed,
 * edge_message (sum over layers), node_update (sum over layers), finalize, whole forward}; ms_host[7] = number
 * of edge_message launches.  Measurement hook for bench.py's roofline block (not on the product path). */
BDIFF_API int32_t bdiff_profile_forward(bdiff_handle* h, void* stream, const float* xh, const float* t,
                                        const float* context, float* net_out, float* ms_host);

/* Optional taps of the last forward, for parity tests: which = "f_ij" [E,9], "e" [E,e_hidden],
 * "xi" [E,xi_hidden*3], "h" [N,256], "chi" [N,96], "x" [N,3], "fbar" [N,12], "chi_in" [N,6] (state after the
 * last layer).  Writes the shape to rows/cols and, if dst != NULL, copies rows*cols floats to dst (device) on
 * `stream`.  Returns BDIFF_EINVAL for unknown names. */
BDIFF_API int32_t bdiff_debug_tap(bdiff_handle* h, void* stream, const char* which, float* dst, int64_t* rows,
                                  int64_t* cols);

/* Replaces: the arithmetic of EquivariantVariationalDiffusion.sample_p_zs_given_zt
 * (variational_diffusion.py:1204-1278) around the denoiser call:
 *   eps = denoiser(z, t);  mu = z/alpha_ts - c_eps*eps;  z' = mu + sigma*noise;  z'[:, :3] re-centred.
 * noise_x fp32[N,3] and noise_h fp32[N,F] hold the two RAW randn draws of
 * sample_combined_position_feature_noise (:795-819); masking and the centring of noise_x happen inside.
 * z is updated in place.  coef_table: DEVICE array of rows {alpha_ts, c_eps, sigma, t_value} with
 * c_eps = sigma2_ts/alpha_ts/sigma_t and sigma = sigma_ts*sigma_s/sigma_t; the row used is
 * coef_table[*step_index] (step_index: DEVICE int32, or NULL for row 0), so one captured CUDA graph can be
 * replayed for every step while the host only bumps the device counter. */
BDIFF_API int32_t bdiff_reverse_step(bdiff_handle* h, void* stream, float* z, const float* context,
                                     const float* noise_x, const float* noise_h, const float* coef_table,
                                     const int32_t* step_index);

/* Replaces: sample_p_xh_given_z0 up to the normal sample (variational_diffusion.py:840-885):
 *   eps = denoiser(z0, 0);  xh = (1/alpha0)*(z0 - sigma0*eps) + sigma_x*noise (noise masked, x-part centred).
 * coef = {1/alpha0, sigma0, sigma_x, 0} (device).  Writes xh fp32[N,3+F]. */
BDIFF_API int32_t bdiff_decode_z0(bdiff_handle* h, void* stream, const float* z0, const float* context,
                                  const float* noise_x, const float* noise_h, const float* coef, float* xh);

/* Masks two raw randn draws and centres the x-part per molecule (variational_diffusion.py:795-819): z_T. */
BDIFF_API int32_t bdiff_center_noise(bdiff_handle* h, void* stream, const float* noise_x, const float* noise_h,
                                     float* z);

/* Synchronises `stream` and reports deferred device-side conditions of the work issued so far on this handle.
 * Today: the tile scheduler of the all-layers tensor-core kernel (replaces the kernel boundaries between
 * GCPInteractions layers, gcpnet.py:1161-1176) raises a flag if a dependency wait ever times out; that is an internal
 * error (BDIFF_ECUDA), never expected.  Call after a chain of bdiff_reverse_step / before trusting a result. */
BDIFF_API int32_t bdiff_check(bdiff_handle* h, void* stream);

/* ---- optimiser side of a training step (SURVEY.md §8 a21): adaptive gradient-norm clipping + AdamW(amsgrad) + EMA --
 * Replaces, per step: get_grad_norm + Queue statistics + clip_gradients (qm9_mol_gen_ddpm.py:1267-1304,
 * src/models/__init__.py:90-113,442-466), torch.optim.AdamW(lr 1e-4, weight_decay 1e-12, amsgrad) (configs/model/
 * *_mol_gen_ddpm.yaml:3-8) and the EMA callback (src/utils/__init__.py:125-142) by three multi-tensor kernels with
 * no host synchronisation.  All pointers are device pointers owned by the caller.
 *   tensors_dev       one record per parameter tensor (max_exp_avg_sq / ema may be NULL)
 *   chunk_*_dev       the tensors cut into chunks of bdiff_optimizer_chunk() elements: chunk c covers elements
 *                     [chunk_start[c], chunk_start[c] + chunk) of tensor chunk_tensor[c]
 *   partial_dev       scratch, num_chunks doubles
 *   state_dev         BDIFF_OPT_STATE_WORDS 32-bit words, zero-initialised once by the caller and then owned by the
 *                     library: [0] step count (int), [1] history length (int), [2] ring position (int), [3] last
 *                     gradient norm (float), [4] last allowed norm (float), [5] last clip coefficient (float),
 *                     [6] clipped? (int), [8 ...] norm history (floats).  Seed the history like the reference
 *                     (one entry of 3000.0: state[1] = 1, state[2] = 1 % queue_len, state[8] = 3000.0f). */
#define BDIFF_OPT_MAX_QUEUE 120
#define BDIFF_OPT_STATE_WORDS (8 + BDIFF_OPT_MAX_QUEUE)
typedef struct bdiff_opt_tensor {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  float* max_exp_avg_sq;
  float* ema;
  int64_t numel;
} bdiff_opt_tensor;
typedef struct bdiff_opt_hyper {
  float lr, beta1, beta2, eps, weight_decay, ema_decay;
  int32_t amsgrad;     /* 1: keep the running maximum of exp_avg_sq */
  int32_t clip;        /* 1: clip to 1.5 * mean + 2 * std of the norm history, then push min(norm, limit) */
  int32_t queue_len;   /* history length (reference: 50) */
} bdiff_opt_hyper;
BDIFF_API int32_t bdiff_optimizer_chunk(void);
BDIFF_API int32_t bdiff_optimizer_step(void* stream, const bdiff_opt_tensor* tensors_dev, const int32_t* chunk_tensor_dev,
                                       const int64_t* chunk_start_dev, int32_t num_chunks, double* partial_dev,
                                       int32_t* state_dev, const bdiff_opt_hyper* hyper);

/* ---- post-sampling stability check (SURVEY.md §8 f1) ----------------------------------------------------------------
 * Batched `check_molecular_stability` (src/datamodules/components/edm/__init__.py:91-124 with get_bond_order_batch
 * :61-88): for every molecule k (atoms mol_off[k] .. mol_off[k+1]) the bond order of each atom pair from the three
 * bond-length tables [num_types x num_types] (pm; 0 = no such bond) and margins, the per-atom bond count, and whether
 * that count is allowed for the atom's type (bit c of allowed_mask[type] set <=> c bonds allowed).  Outputs:
 * nr_bonds[N], nr_stable[B] (atoms with an allowed count), mol_stable[B] (1 iff all atoms).  The tables are data of
 * the caller's dataset (the reference keeps them in dataset_info / edm/constants.py); all pointers are device pointers. */
BDIFF_API int32_t bdiff_check_stability(void* stream, const float* x, const int32_t* atom_types, const int32_t* mol_off,
                                        int32_t num_mols, int32_t num_types, const float* bonds1, const float* bonds2,
                                        const float* bonds3, float margin1, float margin2, float margin3,
                                        const uint32_t* allowed_mask, int32_t limit_bonds_to_one, int32_t* nr_bonds,
                                        int32_t* nr_stable, int32_t* mol_stable);

/* Bond-order matrix of `make_mol_edm` (src/datamodules/components/edm/rdkit_functions.py:276-321 with
 * get_bond_order_batch, edm/__init__.py:61-88): for molecule k, bond_order[pair_off[k] + i*n + j] = bond type (0 none, 1, 2, 3)
 * of the pair (i, j) for i > j and 0 otherwise (E = tril(E_full, -1): the directed graph the reference adds to the RWMol),
 * with limit_bonds_to_one = ("GEOM" in dataset_info["name"]).  pair_off int64[B] = exclusive prefix sum of n_k^2.  Same
 * tables / margins as bdiff_check_stability; all pointers are device pointers. */
BDIFF_API int32_t bdiff_bond_orders(void* stream, const float* x, const int32_t* atom_types, const int32_t* mol_off,
                                    const int64_t* pair_off, int32_t num_mols, int32_t num_types, const float* bonds1,
                                    const float* bonds2, const float* bonds3, float margin1, float margin2, float margin3,
                                    int32_t limit_bonds_to_one, int8_t* bond_order);

/* ---- packed training collation (SURVEY.md §8 f3) ---------------------------------------------------------------------
 * Replaces: ProcessedDataset._featurize_as_graph + PyG collation (datamodules/components/edm_dataset.py:187-216: molecules
 * padded to `pad` atoms, mask = charges > 0) and prepare_context (datamodules/components/edm/utils.py:333-382).  The dataset
 * stays on the device in padded form (positions f32[M,pad,3], charges i32[M,pad], one_hot u8[M,pad,A]); a batch = molecule
 * ids idx i64[B].  bdiff_collate_count: counts[k] = present atoms of molecule idx[k].  bdiff_collate_packed: with
 * mol_off i32[B+1] = exclusive prefix sum of the counts, writes the present atoms of the selected molecules in order:
 * x f32[N,3], one_hot f32[N,A], charges f32[N] and batch_index i64[N] — the reference batch restricted to mask == True.
 * bdiff_prepare_context: context[n,c] = (props[c][idx[batch_index[n]]] - mean[c]) / mad[c] for per-molecule properties
 * props f32[C,M] (the reference's global-property branch; the node mask is all ones in a packed batch). */
BDIFF_API int32_t bdiff_collate_count(void* stream, const int32_t* charges, const int64_t* idx, int32_t num_mols, int32_t pad,
                                      int32_t* counts);
BDIFF_API int32_t bdiff_collate_packed(void* stream, const float* positions, const int32_t* charges, const uint8_t* one_hot,
                                       const int64_t* idx, const int32_t* mol_off, int32_t num_mols, int32_t pad,
                                       int32_t num_types, float* x, float* one_hot_out, float* charges_out,
                                       int64_t* batch_index);
BDIFF_API int32_t bdiff_prepare_context(void* stream, const float* props, const int64_t* idx, const int64_t* batch_index,
                                        const float* mean, const float* mad, int64_t dataset_size, int64_t num_nodes,
                                        int32_t num_props, float* context);

/* ---- training pass of the denoiser (SURVEY.md §8 a20) ---------------------------------------------------------------
 * Replaces: loss.backward() through GCPNetDynamics.forward (src/models/components/gcpnet.py:1069-1232) inside
 * EquivariantVariationalDiffusion.forward in .train() mode (variational_diffusion.py:955-1160) — what the Lightning
 * training_step triggers (src/models/qm9_mol_gen_ddpm.py:340-362).
 *
 * Parameters and gradients travel as ONE flat fp32 buffer each, in a canonical layout: the reference tensors (same
 * names and shapes as bdiff_set_weight, nn.Linear weights [out,in] row-major) in ascending name order, each starting at
 * a multiple of 64 floats.  bdiff_param_floats = length of such a buffer; bdiff_param_layout = {offset, count} of one
 * tensor.  A host keeps its nn.Parameters as views of the flat parameter buffer (bdiff/dynamics.py does), so an
 * optimiser step needs no re-upload.
 *
 * bdiff_train_forward: net_out = denoiser(params_flat; xh, t, context) on the current topology plan, same arguments and
 *   result as bdiff_denoise_forward (fp32), and keeps every intermediate the derivative needs (the "tape", device memory
 *   owned by the handle; one tape at a time).
 * bdiff_train_backward: grads_flat <- d/dparams sum(net_out * d_net_out) for the tape of the last bdiff_train_forward
 *   (the buffer is overwritten, not accumulated into).  No atomics: results are bit-reproducible.
 * bdiff_train_precision: tf32 = 0 (default) fp32 GEMMs, 1 = TF32 tensor-core GEMMs (the reference's bf16-mixed training
 *   configuration is the looser of the two).
 * bdiff_train_variant: 1 (default) = message GCP 0 in split form (node-level h.Wsi^T / h.Wsj^T instead of the [E, 512+Ed]
 *   gather + GEMM), activations kept on the tape and input gradients written straight into their consumers; 0 = the
 *   reference's operator graph one to one (same mathematics, 17 % slower; kept as the cross-check of variant 1).  Takes
 *   effect at the next bdiff_train_forward.
 * All on `stream`, no host synchronisation.  Errors: BDIFF_ESTATE without a plan / tape, BDIFF_ENOMEM for the tape. */
BDIFF_API int64_t bdiff_param_floats(const bdiff_handle* h);
BDIFF_API int32_t bdiff_param_layout(bdiff_handle* h, const char* name, int64_t* offset, int64_t* count);
BDIFF_API int32_t bdiff_train_precision(bdiff_handle* h, int32_t tf32);
BDIFF_API int32_t bdiff_train_variant(bdiff_handle* h, int32_t variant);
/* Per-operation timing of the training pass: enable = 1 starts recording a CUDA event pair around every kernel and GEMM of
 * the following bdiff_train_forward / bdiff_train_backward calls (on their stream); enable = 0 synchronises `stream`, stops
 * and writes a table (operation, calls, total ms, share; sorted) into report[report_bytes] (NUL-terminated, truncated). */
BDIFF_API int32_t bdiff_train_timing(bdiff_handle* h, void* stream, int32_t enable, char* report, int64_t report_bytes);
BDIFF_API int32_t bdiff_train_forward(bdiff_handle* h, void* stream, const float* params_flat, const float* xh, const float* t,
                                      const float* context, float* net_out);
BDIFF_API int32_t bdiff_train_backward(bdiff_handle* h, void* stream, const float* d_net_out, float* grads_flat);

/* Replaces: the warn-and-zero NaN guard of gcpnet.py:1214-1216 as an observable.  *count_host <- number of denoiser
 * forwards (since the last reset / re-plan of the workspace) in which a NaN position appeared and `vel` was zeroed.
 * Synchronises `stream`.  bench.py reports it for every timed chain. */
BDIFF_API int32_t bdiff_nan_guard_count(bdiff_handle* h, void* stream, int64_t* count_host, int32_t reset);

/* Counters for bench.py: kernels launched by this handle since creation. */
BDIFF_API int64_t bdiff_launch_count(const bdiff_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* BDIFF_H_ */
