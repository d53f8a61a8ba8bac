/* nbody_b200.h — C ABI of the B200-native EGNO / SEGNO hot path.
 *
 * The reference (simone7monaco/NO-NODE-comparison) has no FFI or plugin layer: its
 * boundary for this path is two torch.nn.Module classes called from Python
 * (SURVEY.md §8b).  This header is the C-ABI a drop-in replacement binds instead:
 * plain pointers and sizes, no torch types.  Each entry point cites the reference
 * code it replaces (paths relative to the reference root).
 *
 * Conventions
 *  - all tensors fp32, contiguous, row-major, on ONE CUDA device; indices int64.
 *  - the callee never allocates, frees or retains device memory: outputs, the
 *    saved-for-backward buffer and the scratch workspace are caller-owned
 *    (sizes from the *_floats() queries).
 *  - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no host
 *    synchronisation) and are safe under CUDA-graph capture.
 *  - every function returns 0 on success, <0 on error (nb_last_error() gives a
 *    thread-local message).  No CPU fallback exists.
 *  - graphs are the reference's canonical fully connected lists: per graph
 *    `for i: for j != i`, graphs offset by N*b (EGNO/simulation/dataset_simple.py:64-71,
 *    :101-111).  nb_check_canonical_edges validates an edge_index on the device.
 *  - parameters are ONE flat fp32 buffer in the order of the reference module's
 *    named_parameters() (layouts below); gradients use the same layout.
 */
#ifndef NBODY_B200_H
#define NBODY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB_HIDDEN 64      /* hidden_nf the kernels are specialised for (model_confs.yaml:3,23) */
#define NB_MAX_EDGE_FEA 4 /* in_edge_nf upper bound (reference uses 2) */
#define NB_MAX_T 16       /* num_timesteps upper bound for EGNO's temporal convolution */
#define NB_MAX_NODES 100  /* bodies per graph upper bound (BASELINE.json config 5) */

/* Error codes */
#define NB_OK 0
#define NB_ERR_INVALID (-1)  /* bad shape / unsupported configuration */
#define NB_ERR_CUDA (-2)     /* CUDA runtime error */

/* EGNO(**params) as resolved by main.py:133-134 / model_confs.yaml:1-13 (EGNO/model/egno.py:9-35). */
typedef struct NbEgnoConfig {
  int32_t B;             /* trajectories (graphs) in the batch */
  int32_t N;             /* bodies per graph */
  int32_t T;             /* num_timesteps */
  int32_t n_layers;
  int32_t num_modes;     /* after the ctor clamp, <= T/2+1 */
  int32_t in_node_nf;    /* node features BEFORE the time embedding is appended (2) */
  int32_t in_edge_nf;    /* 2 */
  int32_t time_emb_dim;  /* 32 */
  int32_t use_time_conv; /* 1 */
  int32_t num_inputs;    /* 0 / 1: one input frame; L > 1: L input frames (egno.py:13-16,42-47: the embedding then takes
                            in_node_nf + 2 * time_emb_dim features and frame t reads input min(t / (T / L), L - 1)) */
} NbEgnoConfig;

/* SEGNO(**params) as resolved by main.py:110-114 / model_confs.yaml:20-29 (SEGNO/models/model.py:7-26). */
typedef struct NbSegnoConfig {
  int32_t B;
  int32_t N;
  int32_t T;            /* integration sub-steps of this call (forward_step sets n_layers := T, model.py:96-97) */
  int32_t in_node_nf;   /* 1 */
  int32_t in_edge_nf;   /* 2 */
  int32_t recurrent;    /* h += phi_h(...) (gcl.py:93-94) */
  float coords_weight;  /* gcl.py:102 */
  int32_t h_given;      /* 0: `his` are raw node features, embedded inside (single-input forward, model.py:73);
                           1: `his` IS the hidden state h0[BN,64] of forward_step (the segments of the multi-input forward,
                              model.py:79-90): no embedding, and the backward returns dL/dh0 in g_h_in */
} NbSegnoConfig;

int nb_version(void);
const char* nb_last_error(void);

/* --- parameter layout ------------------------------------------------------------
 * EGNO (EGNO/model/basic.py:189-203, egno.py:28-33), H = 64, F = in_node_nf + time_emb_dim,
 * E = 1 + 2H + in_edge_nf:
 *   (note: `layers` is registered before `embedding` in the reference, so it comes first)
 *   per layer i: edge_message_net.scalar_net.mlp.0.weight[H,E] .bias[H]  (cols: radial | h_row | h_col | edge_fea)
 *                edge_message_net.scalar_net.mlp.2.weight[H,H] .bias[H]
 *                coord_net.mlp.0.weight[H,H] .bias[H]  coord_net.mlp.2.weight[1,H] .bias[1]
 *                node_v_net.mlp.0.weight[H,H] .bias[H] node_v_net.mlp.2.weight[1,H] .bias[1]
 *                node_net.mlp.0.weight[H,2H] .bias[H]  node_net.mlp.2.weight[H,H] .bias[H]
 *   embedding.weight[H,F] .bias[H]
 *   per layer i: time_conv_modules.i.t_conv.weights1[H,H,modes,2]
 *   per layer i: time_conv_x_modules.i.t_conv.weights1[2,2,modes,2]
 * SEGNO (SEGNO/models/model.py:19-25, SEGNO/models/models/gcl.py:39-67), E = 2H + 1 + in_edge_nf:
 *   embedding.weight[H,in_node_nf] .bias[H]
 *   module.edge_mlp.0.weight[H,E] .bias[H]   (cols: h_row | h_col | radial | edge_attr)
 *   module.edge_mlp.2.weight[H,H] .bias[H]
 *   module.node_mlp.0.weight[H,2H] .bias[H]  module.node_mlp.2.weight[H,H] .bias[H]
 *   module.coord_mlp.0.weight[H,H] .bias[H]  module.coord_mlp.2.weight[1,H] .bias[1]
 *   module.coord_mlp_vel.0.weight[H,H] .bias[H] module.coord_mlp_vel.2.weight[1,H] .bias[1]  (inert; grads stay 0)
 */
int64_t nb_egno_param_count(const NbEgnoConfig* cfg);
int64_t nb_segno_param_count(const NbSegnoConfig* cfg);

/* floats the caller must provide.  `mode` of the workspace queries: 0 = forward without a `saved` buffer (inference:
 * includes the two ping-pong layer sets that stand in for it), 1 = backward, 2 = forward WITH a `saved` buffer
 * (training: no ping-pong region). */
#define NB_WS_FORWARD_INFER 0
#define NB_WS_BACKWARD 1
#define NB_WS_FORWARD_TRAIN 2
int64_t nb_egno_saved_floats(const NbEgnoConfig* cfg);
int64_t nb_egno_workspace_floats(const NbEgnoConfig* cfg, int mode);
int64_t nb_segno_saved_floats(const NbSegnoConfig* cfg);
int64_t nb_segno_workspace_floats(const NbSegnoConfig* cfg, int mode);

/* Replaces EGNO.forward (EGNO/model/egno.py:37-111, num_inputs == 1) including every
 * EGNN_Layer.forward (EGNO/model/basic.py:167-186), aggregate (basic.py:6-31),
 * TimeConv / TimeConv_x (EGNO/model/layer_no.py:80-178) and get_timestep_embedding (:8-17).
 *   x[BN,3] nodes[BN,in_node_nf] edge_fea[B*N*(N-1),in_edge_nf] v[BN,3] loc_mean[BN,3]
 *   timesteps_out[B,T] (int64)  ->  x_out[T*BN,3] v_out[T*BN,3] h_out[T*BN,H]  (t-major)
 * `saved` may be NULL for inference (then nothing is kept for backward). */
int nb_egno_forward(const NbEgnoConfig* cfg, const float* params, const float* x, const float* nodes,
                    const float* edge_fea, const float* v, const float* loc_mean, const int64_t* timesteps_out,
                    const int64_t* timesteps_in, float* x_out, float* v_out, float* h_out, float* saved,
                    float* workspace, void* stream);
/* num_inputs = L > 1: x, v, loc_mean are [L][BN][3], nodes [L][BN][in_node_nf], edge_fea [L][B*N*(N-1)][in_edge_nf],
 * timesteps_in [B][L] int64 (NULL otherwise); the backward's g_x_in / g_v_in are then [L][BN][3]. */

/* Backward of the above (the reference relies on autograd).  g_*_out may be NULL (= zero).
 * grad_params (same layout as params) is OVERWRITTEN; g_x_in / g_v_in [BN,3] may be NULL. */
int nb_egno_backward(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                     const float* loc_mean, const int64_t* timesteps_out, const int64_t* timesteps_in,
                     const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                     float* grad_params, float* g_x_in, float* g_v_in, float* workspace, void* stream);

/* nb_egno_backward plus the gradients of the other inputs (num_inputs = 1 only; the reference's autograd gives them):
 *   g_nodes[BN, in_node_nf], g_edge_fea[B*N*(N-1), in_edge_nf], g_loc_mean[BN, 3], each nullable (NULL: not formed).
 * Every other output is bitwise what nb_egno_backward writes.  g_nodes or g_edge_fea (in_edge_nf > 0) need
 * `input_grad_workspace` of nb_egno_input_grad_workspace_floats(cfg) floats: the edge-feature gradient of every replicated
 * edge row of every layer, n_layers * T * B*N(N-1) * in_edge_nf floats, reduced in a fixed order at the end.  With all
 * three NULL this is nb_egno_backward (same launches, same results). */
int64_t nb_egno_input_grad_workspace_floats(const NbEgnoConfig* cfg);
int nb_egno_backward_ex(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                        const float* loc_mean, const int64_t* timesteps_out, const int64_t* timesteps_in,
                        const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                        float* grad_params, float* g_x_in, float* g_v_in, float* g_nodes, float* g_edge_fea,
                        float* g_loc_mean, float* workspace, float* input_grad_workspace, void* stream);

/* The same forward and backward with floating-point times: timesteps_out[B,T] and (num_inputs > 1) timesteps_in[B,L] are
 * fp32, the reference's `timesteps.float()`, and may be non-integral.  Integral values give the int64 entry points'
 * results bit for bit.  The workspaces, the saved buffer and the other arguments are those of nb_egno_forward /
 * nb_egno_backward_ex, including the num_inputs = 1 restriction on g_nodes / g_edge_fea / g_loc_mean.  The backward adds
 * the time gradients, each nullable and allowed for every num_inputs:
 *   g_t_out[B,T] = dL/dtimesteps_out, g_t_in[B,L] = dL/dtimesteps_in (num_inputs > 1 only; NULL otherwise)
 * through the sinusoidal embeddings, from the embedding-output gradient the backward forms anyway.  They need no
 * workspace; with time_emb_dim = 0 the times are unused and g_t_out is zero.  With both NULL the backward launches what
 * nb_egno_backward_ex launches (with k_time_table_f for k_time_table). */
int nb_egno_forward_ft(const NbEgnoConfig* cfg, const float* params, const float* x, const float* nodes,
                       const float* edge_fea, const float* v, const float* loc_mean, const float* timesteps_out,
                       const float* timesteps_in, float* x_out, float* v_out, float* h_out, float* saved,
                       float* workspace, void* stream);
int nb_egno_backward_ft(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                        const float* loc_mean, const float* timesteps_out, const float* timesteps_in,
                        const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                        float* grad_params, float* g_x_in, float* g_v_in, float* g_nodes, float* g_edge_fea,
                        float* g_loc_mean, float* g_t_out, float* g_t_in, float* workspace,
                        float* input_grad_workspace, void* stream);

/* Replaces SEGNO.forward_step applied to embedding(his) (SEGNO/models/model.py:73,95-102) with
 * SEGNO_GCL.forward (SEGNO/models/models/gcl.py:111-119), unsorted_segment_sum / _mean (:7-23).
 *   his[BN,in_node_nf] x[BN,3] v[BN,3] edge_attr[B*N*(N-1),in_edge_nf] -> x_out[BN,3] h_out[BN,H] v_out[BN,3] */
int nb_segno_forward(const NbSegnoConfig* cfg, const float* params, const float* his, const float* x, const float* v,
                     const float* edge_attr, float* x_out, float* h_out, float* v_out, float* saved,
                     float* workspace, void* stream);

int nb_segno_backward(const NbSegnoConfig* cfg, const float* params, const float* his, const float* edge_attr,
                      const float* saved, const float* g_x_out, const float* g_h_out, const float* g_v_out,
                      float* grad_params, float* g_x_in, float* g_v_in, float* g_h_in, float* workspace, void* stream);

/* nb_segno_backward plus g_his[BN, in_node_nf] (h_given = 0 only; with h_given = 1 the input gradient is g_h_in) and
 * g_edge_attr[B*N*(N-1), in_edge_nf], both nullable.  g_edge_attr (in_edge_nf > 0) needs `input_grad_workspace` of
 * nb_segno_input_grad_workspace_floats(cfg) floats: one slice of per-row gradients per sub-step, T * B*N(N-1) *
 * in_edge_nf floats, reduced in a fixed order.  With both NULL this is nb_segno_backward. */
int64_t nb_segno_input_grad_workspace_floats(const NbSegnoConfig* cfg);
int nb_segno_backward_ex(const NbSegnoConfig* cfg, const float* params, const float* his, const float* edge_attr,
                         const float* saved, const float* g_x_out, const float* g_h_out, const float* g_v_out,
                         float* grad_params, float* g_x_in, float* g_v_in, float* g_h_in, float* g_his,
                         float* g_edge_attr, float* workspace, float* input_grad_workspace, void* stream);

/* Multi-input SEGNO (SEGNO.forward with x[BN, L, 3], SEGNO/models/model.py:65-90): the reference embeds every observed
 * frame, integrates from frame i to frame i + 1 (forward_step = nb_segno_forward with cfg.h_given = 1) and merges the
 * integrated state with the observed frame i + 1 ('sum', model.py:82-85; InvariantTemporalAttention +
 * prepare_node_inputs, model.py:86-90, 105-139).  These entry points are everything around the segments.
 *   nb_segno_embed_forward : h[rows, H] = his[rows, in_node_nf] embedding.weight^T + embedding.bias   (model.py:73)
 *   nb_segno_embed_backward: grad_params[embedding.*] = its weight / bias gradients (overwritten; workspace:
 *                            nb_segno_embed_backward_workspace_floats)
 *   nb_segno_merge_forward : mode 0 = observed frame `frame` of h_all[n, L, H] / x_all[n, L, 3] / v_all[n, L, 3];
 *                            mode 1 = observed + integrated; mode 2 = attention-weighted pair, attn_params =
 *                            attn_mlp.0.weight[H][H+1] | attn_mlp.0.bias[H] | attn_mlp.2.weight[H] | attn_mlp.2.bias,
 *                            alpha[n, 2] = the softmax weights, kept for the backward
 *   nb_segno_merge_backward: gradients of the merged state -> slice [:, frame, :] of g_*_all and g_*_int; mode 2 also
 *                            writes (accumulate = 0) or adds (1) the 64*65 + 64 + 64 + 1 attention-parameter gradients
 *                            into g_attn (workspace: nb_segno_merge_backward_workspace_floats)
 *   nb_accumulate          : dst[0:n] += src[0:n] (sum of the segments' gradients of the shared parameters) */
int nb_segno_embed_forward(const NbSegnoConfig* cfg, const float* params, int64_t rows, const float* his, float* h,
                           void* stream);
int64_t nb_segno_embed_backward_workspace_floats(const NbSegnoConfig* cfg, int64_t rows);
int nb_segno_embed_backward(const NbSegnoConfig* cfg, int64_t rows, const float* his, const float* g_h, float* grad_params,
                            float* workspace, void* stream);
int nb_segno_merge_forward(int32_t mode, int64_t n, int32_t L, int32_t frame, const float* h_all, const float* x_all,
                           const float* v_all, const float* h_int, const float* x_int, const float* v_int,
                           const float* attn_params, float* h_out, float* x_out, float* v_out, float* alpha, void* stream);
int64_t nb_segno_merge_backward_workspace_floats(int64_t n);
int nb_segno_merge_backward(int32_t mode, int64_t n, int32_t L, int32_t frame, const float* h_all, const float* x_all,
                            const float* v_all, const float* h_int, const float* x_int, const float* v_int,
                            const float* attn_params, const float* alpha, const float* g_h, const float* g_x,
                            const float* g_v, float* g_h_all, float* g_x_all, float* g_v_all, float* g_h_int,
                            float* g_x_int, float* g_v_int, float* g_attn, int32_t accumulate, float* workspace,
                            void* stream);
int nb_accumulate(int64_t n, float* dst, const float* src, void* stream);

/* Validates that (row, col) is the canonical fully connected list for B graphs of N bodies.
 * Writes 0 to *flag_dev if so, else the (1-based) index of a mismatching edge.  No host sync. */
int nb_check_canonical_edges(const int64_t* row, const int64_t* col, int64_t n_edges, int32_t B, int32_t N,
                             int32_t* flag_dev, void* stream);

/* --- building blocks (exported for unit tests and for callers that fuse their own graph) --------- */

/* Fused E_GCL edge tile, forward.  Replaces basic.py:168-175,182 / gcl.py:104-109,74-83,97-102,87:
 * coord_diff, radial, phi_e (2 layers, SiLU), phi_x (64->64->1), f = rij*c, and the per-receiver
 * reductions  M_i = sum_j m_ij ,  Fsum_i = sum_j f_ij  (SEGNO: f clamped to +-100 per edge).
 * P, Q are the per-node pre-projections of the first edge layer (P = W1[:,h_row] h + b1, Q = W1[:,h_col] h).
 *   n_gt graph-instances of N bodies (EGNO: T*B, SEGNO: B); edge features indexed by (gt % B).
 *   w_rad[H], w_ef[in_edge_nf][H] column slices of the first edge layer (stride ldw between output rows). */
int nb_egcl_edge_forward(int32_t n_gt, int32_t B, int32_t N, int32_t n_edge_fea, int32_t clamp_per_edge,
                         const float* x, const float* P, const float* Q, const float* edge_fea, const float* w1,
                         int32_t ldw1, int32_t col_rad, int32_t col_ef, const float* W2, const float* b2,
                         const float* W3, const float* b3, const float* w4, const float* b4, float* M, float* Fsum,
                         void* stream);

/* Fused E_GCL edge tile, backward with edge-tile recompute (nothing per-edge is ever stored).
 * Inputs gM[nodes,H], gFsum[nodes,3]; outputs gP, gQ [nodes,H] (overwritten), gx[nodes,3] (ACCUMULATED into),
 * and weight gradients written/accumulated into a slice laid out as the parameter buffer (see .cu). */
int64_t nb_egcl_edge_backward_workspace_floats(int32_t n_gt, int32_t N);
/* gw (output, overwritten): [gW2 64x64 | gW3 64x64 | gb2 64 | gb3 64 | gw4 64 | G1[64][1+n_edge_fea] | gb4 1] where
 * G1[c][0] is the gradient of w_rad[c] and G1[c][1+f] that of w_ef[f][c]. */
int nb_egcl_edge_backward(int32_t n_gt, int32_t B, int32_t N, int32_t n_edge_fea, int32_t clamp_per_edge,
                          const float* x, const float* P, const float* Q, const float* edge_fea, const float* w1,
                          int32_t ldw1, int32_t col_rad, int32_t col_ef, const float* W2, const float* b2,
                          const float* W3, const float* b3, const float* w4, const float* b4, const float* gM,
                          const float* gFsum, float* gP, float* gQ, float* gx, float* gw, float* workspace,
                          void* stream);

/* --- accounting --------------------------------------------------------------------------------- */
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long nb_launch_count(void);
/* CUDA-event timing of the dominant kernels on their launch stream: categories
 * 0 = edge tile forward, 1 = edge tile backward, 2 = node GEMMs (k_gemm64_tc, k_egno_pair, SEGNO node chain), 3 = wgrad64,
 * 4 = fused temporal convolution, 5 = fused SEGNO forward (all T sub-steps in one kernel), 6 = EGNO per-layer node kernel
 * forward, 7 = its backward.
 * enable(1) resets the counters; read() synchronises the recorded events and returns total milliseconds and launch
 * counts per category (arrays of NB_PROFILE_CATEGORIES entries). */
#define NB_PROFILE_CATEGORIES 8
int nb_profile_enable(int enable);
int nb_profile_read(double* ms /*[NB_PROFILE_CATEGORIES]*/, long long* counts /*[NB_PROFILE_CATEGORIES]*/);

/* Edge-tile implementation: 2 = tcgen05 tensor-core tiles whose node gathers and receiver / sender reductions are
 * one-hot MMAs (default, product path; graphs with more than 27 nodes are walked in receiver x sender blocks by the same
 * kernels, template parameter BLK), 1 = tcgen05 tiles with CUDA-core gathers / reductions, 0 = fp32 SIMT tiles (kept as
 * an independent cross-check and for the host emulator of the test suite).  All are CUDA kernels of this library.
 * The three nb_set_* switches below are process-wide TEST hooks (variant cross-checks); they are not meant to be flipped
 * while another thread is inside a forward / backward call. */
int nb_set_edge_impl(int impl);
int nb_get_edge_impl(void);
/* Edge impl 2, forward: 1 (default) = units of one graph-instance with at least three 128-edge tiles (N = 17 .. 27) run
 * three tiles in flight per SM (k_edge_fwd_sel3), 0 = they run the two-CTA-per-SM kernel every other shape runs
 * (cross-check).  M and Fsum are bitwise equal either way. */
int nb_set_edge_fwd3(int on);
int nb_get_edge_fwd3(void);
/* Node-level 64-wide GEMMs and weight-gradient reductions: 1 = tcgen05 kernels (default, product path), 0 = fp32 SIMT
 * kernels (cross-check; the variant the host emulator runs). */
int nb_set_node_impl(int impl);
int nb_get_node_impl(void);
/* EGNO: 1 (default) = one fused node kernel per layer and direction, 0 = the generic node GEMM launches (cross-check). */
int nb_set_node_fused(int on);
int nb_get_node_fused(void);
/* SEGNO forward: 1 = all T integration sub-steps fused into one kernel, node state resident in shared memory (default;
 * needs edge impl 2, node impl 1 and N <= 27), 0 = one kernel sequence per sub-step. */
int nb_set_segno_fused(int on);
int nb_get_segno_fused(void);

/* --- caller-side helpers that keep training / rollout loops on the device (SURVEY.md 8f-1, 8f-2) -----------------
 * nb_nbody_features: the featurisation of one frame — EGNO prepare_inputs (EGNO/main_simulation_simple_no.py:326-338)
 * and SEGNO's (SEGNO/train_nbody.py:119-123, :228-233) — for the canonical fully connected edge order:
 *   nodes[B*N][1 + with_charge] = |v| (, charge);  loc_mean[B*N][3] = per-trajectory mean position (nullable);
 *   edge_attr[B*N*(N-1)][2] = (edge_attr_o or q_i q_j, |x_i - x_j|^2).
 * nb_nbody_energy: conserved energy per frame and trajectory, energy[F][B] — kind 0 charged
 * (utils.py:126-144: K + 1/2 sum_{i!=j} q_i q_j / r_ij), kind 1 gravity (utils.py:175-195: 1/2 sum m v^2 -
 * G sum_{i<j} m_i m_j / r_ij); loc / vel are [F][B*N][3], charges (or masses) [B*N]. */
int nb_nbody_features(int32_t B, int32_t N, int32_t with_charge, const float* loc, const float* vel, const float* charges,
                      const float* edge_attr_o, float* nodes, float* loc_mean, float* edge_attr, void* stream);
int nb_nbody_energy(int32_t kind, int32_t F, int32_t B, int32_t N, float G, const float* loc, const float* vel,
                    const float* charges, float* energy, void* stream);

/* Trajectory MSE and its gradient (SURVEY.md 8f-4): the callers' loss
 *   losses[t] = mean over (rows, xyz) of (pred - target)^2,   loss = mean_t losses[t]  (only_first: losses[0])
 * (EGNO/main_simulation_simple_no.py:273-276: MSELoss(reduction='none')(...).mean((0, 1, 3)) then .mean() / [0];
 * SEGNO/train_nbody.py:163-165 is the T = 1 case) with grad = d loss / d pred written in the same pass (nullable).
 * pred is [T][rows][3] (the models' frame-major output); target_layout 0: [T][rows][3], 1: [rows][T][3] (the data
 * loader's [B, N, T, 3]).  workspace: nb_traj_mse_workspace_floats(T) floats.  Two launches, deterministic. */
int64_t nb_traj_mse_workspace_floats(int32_t T);
int nb_traj_mse(int32_t T, int64_t rows, int32_t target_layout, int32_t only_first, const float* pred, const float* target,
                float* losses, float* loss, float* grad, float* workspace, void* stream);

/* Trajectory simulators (SURVEY.md 8f-4, data generation): float64 leapfrog integration of B independent systems of
 * N <= 128 bodies, one CTA per trajectory; random draws stay on the host, in the reference's order.
 * nb_sim_charged = ChargedParticlesSim.sample_trajectory (synthetic_sim.py:220-296): loc0 / vel0 [B][3][N], charges
 *   [B][N] -> loc / vel [B][T / sample_freq - 1][3][N] (the frames the reference keeps; velocities at half steps);
 *   the reference's constants are dt = 1e-3, strength = 1, max_force = 0.1 / dt, box_size = 5.
 * nb_sim_gravity = GravitySim.sample_trajectory (synthetic_sim.py:360-405): pos0 / vel0 [B][N][3], mass [B][N] ->
 *   pos / vel / force [B][T / sample_freq][N][3]; reference constants dt = 1e-3, G = 1, softening = 0.1. */
int nb_sim_charged(int32_t B, int32_t N, int32_t T, int32_t sample_freq, double dt, double strength, double max_force,
                   double box_size, const double* loc0, const double* vel0, const double* charges, double* loc, double* vel,
                   void* stream);
int nb_sim_gravity(int32_t B, int32_t N, int32_t T, int32_t sample_freq, double dt, double G, double softening,
                   const double* pos0, const double* vel0, const double* mass, double* pos, double* vel, double* force,
                   void* stream);

/* Fused Adam over flat buffers (SURVEY.md 8f-4): torch.optim.Adam semantics (amsgrad = False), one launch for n
 * elements; `step` is a device float counting the steps taken (incremented first when tick != 0), so the call is
 * CUDA-graph capturable.  Replaces the per-tensor optimizer launches of main.py:150 for models whose parameters and
 * gradients are the flat buffers of this ABI.  grad_scale multiplies the gradients first: 1 / world size when the bucket
 * holds the all-reduced SUM (the data-parallel mean costs no launch of its own), 1 otherwise. */
int nb_adam_step(int64_t n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* step,
                 int32_t tick, double lr, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                 void* stream);
/* Data-parallel variant: gradient all-reduce and optimizer update as ONE kernel over peer memory.  peer_grads[r] (host
 * array of npeer <= 8 device pointers) is rank r's flat gradient buffer as mapped into this process (NVLink / NVSwitch
 * peer access, e.g. torch's symmetric memory); every rank sums them in rank order (bit-identical replicas) and applies
 * grad_scale (1 / world for the mean).  The caller orders the launch after every rank's backward (a device-side
 * barrier) and keeps the buffers unchanged until every rank has passed a second barrier.  Replaces the
 * dist.all_reduce + optimizer.step pair of a data-parallel main.py:150. */
int nb_adam_step_peers(int64_t n, float* params, const void* const* peer_grads, int32_t npeer, float* exp_avg,
                       float* exp_avg_sq, float* step, int32_t tick, double lr, double beta1, double beta2, double eps,
                       double weight_decay, double grad_scale, void* stream);

/* tcgen05 self test: one 128-thread CTA evaluates, with split-bf16 operands and fp32 TMEM accumulation,
 *   mode 0: A[128x64] * W[64x64]^T   mode 1: A[128x64] * W[64x64]   mode 2: A[128x64]^T * W[128x64]
 * and dumps the raw 128 TMEM lanes x 64 columns into out[128*64]. */
int nb_tc_selftest(int32_t mode, const float* A, const float* W, float* out, void* stream);

/* SiLU self test: out_mufu[i] = x sigmoid(x) with ex2.approx + rcp.approx (two MUFU operations), out_fma[i] = the same
 * with the reciprocal on the FMA pipe (bit-trick seed + three Newton steps), the variant the forward edge tile uses for
 * a measured share of its elements (EGNO/model/basic.py:46-51: SiLU after every edge / coordinate MLP layer). */
int nb_silu_selftest(int64_t n, const float* x, float* out_mufu, float* out_fma, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NBODY_B200_H */
