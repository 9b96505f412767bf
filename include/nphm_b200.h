/* nphm_b200.h - C ABI of libnphm_b200.so, the B200-native engine behind NPHM's hot path.
 *
 * The reference (SimonGiebenhain/NPHM) has no FFI layer: its hot path sits behind Python call signatures
 * (SURVEY.md 8b).  This header is the boundary a binding would target; the Python mirror of the reference
 * modules in nphm_b200/ binds it with ctypes (nphm_b200/_native.py), see INTEGRATION.md.
 *
 * Conventions
 *   - every function returns NPHM_OK (0) or a negative error code; nphm_last_error() gives the message of the
 *     last failure on the calling thread.
 *   - pointers named *_dev are CUDA device pointers on the current device, *_host are host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are asynchronous on that
 *     stream unless stated otherwise.  No torch types appear in any signature.
 *   - all network arithmetic is fp32 in / fp32 out; weights are given in the reference's state_dict layout.
 *   - handles are not thread safe; use one handle per host thread / stream.
 */
#ifndef NPHM_B200_H
#define NPHM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define NPHM_OK               0
#define NPHM_ERR_INVALID     -1   /* bad argument */
#define NPHM_ERR_CUDA        -2   /* a CUDA runtime call failed */
#define NPHM_ERR_UNSUPPORTED -3   /* configuration not supported by the requested kernel */
#define NPHM_ERR_CAPACITY    -4   /* caller-provided buffer too small */

/* kernel selection for the network queries */
#define NPHM_IMPL_AUTO   0   /* tcgen05 kernel when the configuration allows it, else SIMT */
#define NPHM_IMPL_SIMT   1   /* fp32 FFMA kernel (any configuration) */
#define NPHM_IMPL_TC     2   /* tcgen05 / TMEM kernel, 3-pass fp16 split (fp32-equivalent accuracy) */
#define NPHM_IMPL_TC_PRUNED 3 /* OPT-IN: tcgen05 kernel that skips, per compact tile of 128 points, the ensemble members whose
                                normalised Gaussian blend weight is < tau for every point of the tile.  Not the dense
                                reference computation: |error| <= n_members * tau * max_k |s_k| (tau default 1e-8). */

const char *nphm_last_error(void);
int nphm_abi_version(void);
/* sm count and compute capability of the current device */
int nphm_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* ------------------------------------------------------------------------------------------------
 * Identity SDF ensemble  == FastEnsembleDeepSDFMirrored (reference src/NPHM/models/EnsembledDeepSDF.py:153-267)
 * ---------------------------------------------------------------------------------------------- */
typedef struct nphm_ensemble nphm_ensemble;

typedef struct {
    int n_loc;          /* facial anchors (39); ensemble size is n_loc + 1              (:183)      */
    int n_symm_pairs;   /* mirrored anchor pairs sharing weights (16)                   (:184,:43)  */
    int lat_dim_glob;   /* 64                                                                        */
    int lat_dim_loc;    /* 32; latent = [z_glob, z_0 .. z_{n_loc-1}, z_global_member]   (:210-212)  */
    int hidden_dim;     /* 200                                                                       */
    int n_layers;       /* 4 hidden layers -> 5 linear layers, skip at n_layers/2       (:80-96)    */
    int pos_mlp_dim;    /* hidden width of mlp_pos (256)                                (:194-200)  */
} nphm_ensemble_config;

int nphm_ensemble_create(const nphm_ensemble_config *cfg, nphm_ensemble **out);
void nphm_ensemble_destroy(nphm_ensemble *h);
/* threshold tau of NPHM_IMPL_TC_PRUNED (relative blend weight below which a member is skipped), 0 <= tau < 1 */
int nphm_ensemble_set_prune_threshold(nphm_ensemble *h, float tau);

/* Replaces `load_state_dict` for the engine.  lin_w_dev[l]: (n_sets, out_l, in_l) row-major, lin_b_dev[l]:
 * (n_sets, out_l) for l = 0..n_layers (keys ensembled_deep_sdf.lin{l}.weight/bias, n_sets = n_loc+1-n_symm_pairs);
 * pos_w_dev/pos_b_dev: the three nn.Linear of mlp_pos (keys mlp_pos.{0,2,4}); mean_anchors_dev: n_loc*3.
 * Packs/splits the weights for every kernel; must be called again after the parameters change. */
int nphm_ensemble_load_weights(nphm_ensemble *h,
                               const float *const *lin_w_dev, const float *const *lin_b_dev,
                               const float *const *pos_w_dev, const float *const *pos_b_dev,
                               const float *mean_anchors_dev, void *stream);

/* == FastEnsembleDeepSDFMirrored.forward(xyz, lat_rep, None) for lat_rep constant over the points of a query.
 *   xyz_dev       n_queries * n_points * 3
 *   latents_dev   n_queries * lat_dim
 *   quirk_period  eval-mode quirk of :260-261 (`sdf_pred[:, :, -1, 0] = 1` hits the LAST POINT of a call):
 *                 0 = train mode (off); p > 0 = points with (i % p == p-1) or i == n_points-1 get s_k = 1 for all
 *                 members.  A plain forward call uses p = n_points; get_logits (models/reconstruction.py:13) uses
 *                 p = nbatch_points.
 *   out_sdf_dev   n_queries * n_points           out_anchors_dev  n_queries * n_loc * 3 (may be NULL)        */
int nphm_ensemble_query(nphm_ensemble *h, const float *xyz_dev, const float *latents_dev,
                        int n_queries, long long n_points, long long quirk_period,
                        float *out_sdf_dev, float *out_anchors_dev, int impl, void *stream);

/* Same for ONE latent over (a contiguous range of) the regular grid of
 * create_grid_points_from_bounds (utils/reconstruction.py:5-20): point g = first + i, i < count, has
 * (ix,iy,iz) = unravel(g, res^3), z fastest, coordinates float32(linspace_f64(min,max,res)[i*]).  The points are
 * generated in the kernel (no xyz traffic).  The quirk uses the GLOBAL index g, so shards agree with a
 * single-GPU run.  out_sdf_dev: count floats. */
int nphm_ensemble_query_grid(nphm_ensemble *h, const float *latent_dev,
                             const double grid_min[3], const double grid_max[3], int res,
                             long long first, long long count, long long quirk_period,
                             float *out_sdf_dev, float *out_anchors_dev, int impl, void *stream);

/* Host-buffer convenience used for end-to-end timing: latent_host (lat_dim floats) -> device, grid query of the
 * whole res^3 grid, volume -> out_host (res^3 floats).  Synchronous. */
int nphm_ensemble_get_logits_host(nphm_ensemble *h, const float *latent_host,
                                  const double grid_min[3], const double grid_max[3], int res,
                                  long long quirk_period, float *out_host, int impl);

/* ------------------------------------------------------------------------------------------------
 * Plain DeepSDF MLP == DeepSDF.forward (reference src/NPHM/models/deepSDF.py:6-89), also the backbone of
 * DeformationNetwork (:118-239) whose condition vector the host builds (compressor Linear, :218-223).
 * ---------------------------------------------------------------------------------------------- */
typedef struct nphm_mlp nphm_mlp;

typedef struct {
    int lat_dim;      /* condition width (232 for the deformation backbone)  */
    int hidden_dim;   /* 512                                                 */
    int n_layers;     /* hidden layers (6) -> n_layers+1 linear, skip at n_layers/2 */
    int out_dim;      /* 3                                                   */
} nphm_mlp_config;

int nphm_mlp_create(const nphm_mlp_config *cfg, nphm_mlp **out);
void nphm_mlp_destroy(nphm_mlp *h);
/* w_dev[l]: (out_l, in_l) row-major, b_dev[l]: (out_l), l = 0..n_layers (keys lin{l}.weight/bias). */
int nphm_mlp_load_weights(nphm_mlp *h, const float *const *w_dev, const float *const *b_dev, void *stream);
/* xyz_dev n_queries*n_points*3, cond_dev n_queries*lat_dim -> out_dev n_queries*n_points*out_dim.
 * impl: NPHM_IMPL_AUTO picks the tcgen05 kernel for the deformation-backbone configuration (hidden 512, 6 hidden layers,
 * condition 232, 3 outputs) and the fp32 FFMA kernel otherwise; NPHM_IMPL_SIMT / NPHM_IMPL_TC force one. */
int nphm_mlp_query(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries,
                   long long n_points, float *out_dev, int impl, void *stream);

/* Batched Broyden search for canonical correspondences: roots of  x + F(x; cond) - obs  per point, F = this MLP
 * (3 outputs).  Replaces the Python loop of models/iterative_root_finding.py:5-71 (`broyden`) with the residual of
 * `search` (:142-147): same update rule, thresholds and freeze logic, one fused-MLP launch per step, no host
 * round trips except a 4-byte "still active?" read every 3 steps (the reference's early exit).
 *   x_dev          in: start points, out: 'result' (n_queries*n_points*3) - like the reference this is the point at
 *                  which a sample stopped, not the best one seen (its x_opt aliases x)
 *   jinv_init_dev  n_queries*n_points*9 row-major initial inverse Jacobians (not modified)
 *   diff_dev       out: smallest residual norm seen per sample; valid_dev out: diff < cvg_thresh (1 byte each)
 *   steps_done     host int.  NULL = sync-free call (CUDA-graph capturable): no early-exit read-back, all max_steps run; frozen
 *                  samples do not move any more, so the result is identical.
 *   workspace_dev: nphm_broyden_workspace_bytes(n_queries*n_points) bytes. */
long long nphm_broyden_workspace_bytes(long long n_total);
int nphm_mlp_broyden_search(nphm_mlp *h, const float *cond_dev, int n_queries, long long n_points,
                            const float *obs_dev, float *x_dev, const float *jinv_init_dev, int max_steps,
                            float cvg_thresh, float dvg_thresh, float eps, float *diff_dev,
                            unsigned char *valid_dev, int *steps_done, void *workspace_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Marching cubes == mcubes.marching_cubes(volume, iso) as called at utils/reconstruction.py:30
 * (PyMCubes semantics restated in oracle/mc_oracle.c: x-major cell order, `<=` classification, one vertex per
 * crossed grid edge numbered in creation order, double-precision interpolation, classic 256-case table).
 * The volume is a slab of nx planes (x slowest, z fastest) that may be a shard of a larger grid.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int nx, ny, nz;       /* planes / rows / columns of vol_dev                                               */
    int x_global0;        /* global x index of plane 0 (0 for a whole volume)                                 */
    int ghost_lo;         /* 1: the first cell layer belongs to the previous shard; it is classified so that
                             shared vertices resolve to the right ids, but emits nothing                      */
    int negate;           /* 1: run on -vol (mesh_from_logits negates the SDF, utils/reconstruction.py:25)    */
    double iso;
} nphm_mc_params;

/* bytes of scratch the two calls below need for this slab */
long long nphm_mc_workspace_bytes(const nphm_mc_params *p);
/* Pass 1: classify + count.  Writes the number of vertices / triangles this slab emits to the two host
 * integers (synchronises the stream). */
int nphm_mc_count(const float *vol_dev, const nphm_mc_params *p, void *workspace_dev,
                  long long *n_verts_host, long long *n_tris_host, void *stream);
/* Pass 2 (after nphm_mc_count on the same workspace): emit.  verts_dev: n_verts*3 doubles in GLOBAL index units;
 * tris_dev: n_tris*3 int64 vertex ids offset by vert_id_base (the number of vertices emitted by all earlier
 * shards; 0 for a whole volume). */
int nphm_mc_emit(const float *vol_dev, const nphm_mc_params *p, void *workspace_dev,
                 long long vert_id_base, double *verts_dev, long long *tris_dev, void *stream);
/* Host-buffer convenience == mcubes.marching_cubes on a host volume: two-call protocol, call with
 * verts_host == NULL to get the counts. Synchronous. */
int nphm_marching_cubes_host(const float *vol_host, int nx, int ny, int nz, double iso, int negate,
                             double *verts_host, long long *tris_host,
                             long long *n_verts, long long *n_tris);

/* ------------------------------------------------------------------------------------------------
 * Identity-space fitting step == one iteration of inference_identity_space
 * (reference src/NPHM/models/fitting.py:197-279): ensemble forward on the sampled observation points, clamped
 * |sdf| loss, latent regularisers, analytic gradient w.r.t. the latent (through the member inputs, the
 * anchors/mlp_pos and the blend weights), torch.optim.Adam update.  No autograd graph.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    float lambda_surface, lambda_reg_global, lambda_reg_loc, lambda_reg_unobserved, lambda_symm_dist;
    float clamp;          /* keep |sdf| < clamp (0.1 / 0.05 / 0.0075 by iteration, :239-246)                */
    float lr;             /* current Adam lr                                                                 */
    int   step;           /* 1-based Adam step count                                                         */
} nphm_fit_params;

/* bytes of scratch for n_points observation points */
long long nphm_fit_workspace_bytes(const nphm_ensemble *h, long long n_points);
/* latent_dev (lat_dim) is updated in place; adam_m_dev / adam_v_dev are the optimiser state (lat_dim each,
 * zero-initialised by the caller).  loss_terms_dev (may be NULL) receives
 * [surface, reg_global, reg_loc, reg_unobserved, symm_dist, n_kept].  grad_out_dev (may be NULL) receives the
 * latent gradient (lat_dim). If `apply_update` is 0 only loss/gradient are produced. */
int nphm_fit_identity_step(nphm_ensemble *h, const float *points_dev, long long n_points,
                           float *latent_dev, float *adam_m_dev, float *adam_v_dev,
                           const nphm_fit_params *fp, int apply_update,
                           float *loss_terms_dev, float *grad_out_dev,
                           void *workspace_dev, void *stream);

/* Surface term of the joint fitter with gradients w.r.t. BOTH the identity code and the query points
 * (reference src/NPHM/models/fitting.py:114-125: `sdf = decoder(xc, lat_rep_shape)`, `sdf[valid_ids]`, `l[l < clamp].mean()`):
 *   loss = mean over { p : mask[p] != 0 and |sdf_p| < clamp } of |sdf_p|        (training-mode forward, no eval quirk)
 * mask_dev (n_points bytes, may be NULL = all valid).  loss_terms_dev[0] = loss (NaN if nothing is kept, like torch),
 * [5] = number of kept points, [1..4] = the latent regularisers (unweighted).  grad_latent_dev (lat_dim) and
 * grad_points_dev (n_points*3, may be NULL) receive d loss / d latent (member inputs + anchors/mlp_pos + blend weights) and
 * d loss / d point (local coordinates of every member + blend weights); both are zero when nothing is kept.
 * The latent is not modified.  Same workspace as nphm_fit_identity_step.  Needs the tensor-core configuration when
 * grad_points_dev is given. */
int nphm_fit_surface_grad(nphm_ensemble *h, const float *points_dev, long long n_points, const float *latent_dev,
                          const unsigned char *mask_dev, float clamp, float *loss_terms_dev,
                          float *grad_latent_dev, float *grad_points_dev, void *workspace_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * DeepSDF-style stacks layer by layer on the generic fp32-accurate tcgen05 linear layer (csrc/tc_linear.cu, mlp_chain.cu).
 * ---------------------------------------------------------------------------------------------- */
/* == nphm_mlp_query for ANY width (DeepSDF.forward, reference src/NPHM/models/deepSDF.py:64-89; e.g. the NPM baseline
 * 515 -> 1024 x 8 of scripts/configs/npm.yaml:2-4, which no fused kernel takes). */
int nphm_mlp_query_layers(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                          float *out_dev, void *stream);
/* Value and input Jacobian in one forward-mode pass == `jac` (reference src/NPHM/models/diff_operators.py:26-54: three
 * autograd passes) without the identity term:  out_dev [q][n][out_dim] (may be NULL), jac_dev [q][n][out_dim][3] = d out / d xyz.
 * Callers: iterative_root_finding.py:123 (initial inverse Jacobian of the Broyden search), fitting.py:104 (implicit
 * differentiation of the root). */
int nphm_mlp_jacobian(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                      float *out_dev, float *jac_dev, void *stream);
/* Adjoint pass == what loss.backward() (reference src/NPHM/models/fitting.py:167) propagates through the deformation
 * network:  grad_cond_dev [q][lat_dim] = sum_n (d out_n / d cond_q)^T grad_out_n  (may be NULL),
 *           grad_xyz_dev [q][n][3]    = (d out_n / d xyz_n)^T grad_out_n            (may be NULL).   grad_out_dev: [q][n][out_dim].
 * xyz_dev == NULL: reuse the activations of the preceding nphm_mlp_jacobian / nphm_mlp_inverse_jacobian call on this handle
 * (same points, same condition) instead of recomputing the value pass. */
int nphm_mlp_backward_inputs(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                             const float *grad_out_dev, float *grad_cond_dev, float *grad_xyz_dev, void *stream);
/* (I + d out / d xyz)^-1 per point for a 3-output stack == `jac(decoder_expr, x, ...).inverse()` of the reference
 * (iterative_root_finding.py:123, fitting.py:104): out_dev [q][n][3] (may be NULL), jinv_dev [q][n][3][3]. */
int nphm_mlp_inverse_jacobian(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                              float *out_dev, float *jinv_dev, void *stream);

/* First-order training of a layer-chain stack (the deformation network of stage-2 training, reference
 * scripts/training/train_corresp.py).  The condition of query q at point n is cond_q + (noise_qn, 0): noise_dev
 * [q][n][noise_dim] is added to the first noise_dim condition columns (noise_dim 0: none; at most 36).
 * nphm_mlp_train_workspace_bytes: size of the device workspace one training forward needs (-1 on bad arguments). */
long long nphm_mlp_train_workspace_bytes(const nphm_mlp *h, int n_queries, long long n_points, int noise_dim);
/* == DeepSDF.forward on [xyz | cond_q + (noise_qn, 0)]: out_dev [q][n][out_dim]; keeps what the backward needs in workspace_dev */
int nphm_mlp_forward_train(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, const float *noise_dev, int noise_dim,
                           int n_queries, long long n_points, float *out_dev, void *workspace_dev, void *stream);
/* Gradients of sum(out * grad_out) for the forward held in workspace_dev (same arguments): grad_w_dev[l] [N_l][in_l] and
 * grad_b_dev[l] [N_l] in the state_dict layout (condition columns included), grad_cond_dev [q][cond_dim], grad_xyz_dev [q][n][3].
 * Every output may be NULL (grad_w_dev == NULL: no weight GEMMs; a NULL entry skips that layer); outputs are overwritten, not
 * accumulated, and the weight gradients are bitwise reproducible.  A workspace of another shape, another handle or of weights
 * loaded before the forward is refused with NPHM_ERR_INVALID, and so is a result that is not finite (an adjoint beyond the fp16
 * range of the packed activation format, or non-finite weights / inputs).  Synchronises the stream twice: to read the workspace
 * header and the scale of grad_out, and to check the outputs. */
int nphm_mlp_backward_train(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, const float *noise_dev, int noise_dim,
                            int n_queries, long long n_points, const float *grad_out_dev, float *const *grad_w_dev,
                            float *const *grad_b_dev, float *grad_cond_dev, float *grad_xyz_dev, void *workspace_dev,
                            void *stream);

/* anchors_dev [n_queries][n_loc][3] = mlp_pos(z_glob) + mean anchors (reference src/NPHM/models/EnsembledDeepSDF.py:228-229)
 * without evaluating the ensemble - what the fitters read from `decoder(zeros(1,1,3), lat)[1]` (fitting.py:59, :211). */
int nphm_ensemble_anchors(nphm_ensemble *h, const float *latents_dev, int n_queries, float *anchors_dev, void *stream);

/* Vector-Jacobian product of the ensemble forward w.r.t. its inputs == what torch.autograd computes for
 * `decoder(xyz, lat)[0].backward(grad_sdf)` on FastEnsembleDeepSDFMirrored in training mode (reference
 * src/NPHM/models/EnsembledDeepSDF.py:203-267; used by fitting.py:111-167 through loss.backward()):
 *   grad_points_dev[p] = grad_sdf[p] * d sdf_p / d xyz_p      (n_points * 3, may be NULL)
 *   grad_latent_dev    = sum_p grad_sdf[p] * d sdf_p / d latent  (lat_dim: member inputs + anchors/mlp_pos + blend weights)
 * sdf_out_dev (n_points, may be NULL) receives the forward values.  Same workspace as nphm_fit_identity_step. */
int nphm_ensemble_backward_inputs(nphm_ensemble *h, const float *points_dev, long long n_points, const float *latent_dev,
                                  const float *grad_sdf_dev, float *sdf_out_dev, float *grad_latent_dev,
                                  float *grad_points_dev, void *workspace_dev, void *stream);

/* Second half of a fitting iteration (regularisers of fitting.py:252-268 + torch.optim.Adam, :278-279) for a surface
 * gradient that was evaluated elsewhere: the point-sharded fit of one head over several GPUs (north_star / SURVEY.md 8e)
 * evaluates nphm_fit_surface_grad on every rank's share of the sampled points, combines [n_r * grad_r, n_r * loss_r, n_r]
 * with ONE all-reduce and then calls this on every rank with the identical global result.
 * surface_grad_dev: d(mean |sdf| over the kept points)/d latent (lat_dim, un-weighted: lambda_surface is applied here);
 * surface_stats_dev: [n_kept, sum |sdf| over the kept points]; loss_terms_dev as in nphm_fit_identity_step (may be NULL).
 * grad_anchors_dev (n_loc*3, may be NULL): an additional gradient w.r.t. the anchors, back-propagated through mlp_pos into
 * z_glob (joint fitter: the deformation network is conditioned on the anchors, deepSDF.py:218-219); also scaled by
 * lambda_surface.  apply_update = 0: only the total gradient (grad_out_dev, lat_dim, may be NULL) and the loss terms. */
int nphm_fit_apply_gradient(nphm_ensemble *h, float *latent_dev, float *adam_m_dev, float *adam_v_dev,
                            const nphm_fit_params *fp, const float *surface_grad_dev, const float *surface_stats_dev,
                            const float *grad_anchors_dev, int apply_update, float *loss_terms_dev, float *grad_out_dev,
                            void *stream);
/* torch.optim.Adam.step() (lr, betas 0.9/0.999, eps 1e-8) on a dense fp32 tensor: the expression codes of the joint fitter
 * (reference src/NPHM/models/fitting.py:36,169).  step is the 1-based step count. */
int nphm_adam_step(float *param_dev, const float *grad_dev, float *adam_m_dev, float *adam_v_dev, long long n, float lr,
                   int step, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation metrics (SURVEY.md 8f-4): nearest-neighbour distances between two point clouds ==
 * scipy.spatial.cKDTree(tgt).query(src) as used by `distance_p2p` (reference src/NPHM/evaluation/metrics.py:171-194) on
 * 250 k-point clouds (scripts/evaluation/eval.py:111).  dist_dev: n_src fp64, idx_dev: n_src int64.
 * ---------------------------------------------------------------------------------------------- */
int nphm_nearest_neighbors(const float *src_dev, long long n_src, const float *tgt_dev, long long n_tgt,
                           double *dist_dev, long long *idx_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NPHM_B200_H */
