/*
 * windgnn_b200.h — C-ABI of the B200-native WindGNN forward hot path.
 *
 * This is the drop-in boundary.  Every entry point is `extern "C"`, takes plain
 * pointers and sizes (no torch / C++ types) and names the reference interface it
 * replaces.  Reference paths are relative to NagsTheProgrammer/WindGNN.
 *
 * Conventions
 *   - All tensors are dense, row-major ("C-contiguous") fp32 unless stated.
 *   - "device pointer" = memory of CUDA device `device`; the call is asynchronous
 *     on `stream` (a cudaStream_t passed as void*; NULL = the legacy default stream).
 *   - The caller owns every buffer, including `workspace`; the library keeps no
 *     pointer after the call returns.  Its only state is thread-local: the last-error
 *     string and, for the host-buffer entry points, a cache of internal streams / events.
 *   - Return value: 0 (WG_OK) on success, a negative WG_ERR_* code otherwise;
 *     `wg_last_error()` then describes the failure.  Nothing throws.
 *   - There is no CPU fallback: without a CUDA device every compute entry point
 *     returns WG_ERR_CUDA.
 */
#ifndef WINDGNN_B200_H
#define WINDGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WG_ABI_VERSION 4

/* `flags` of the GCN-GRU entry points */
#define WG_FLAG_TENSOR_CORES 1 /* GRU input projection and recurrent product on tcgen05 (split fp16 operands) */

enum {
    WG_OK = 0,
    WG_ERR_BAD_ARG = -1,     /* null pointer, non-positive size, inconsistent dims        */
    WG_ERR_UNSUPPORTED = -2, /* dims outside what the sm_100a kernels are built for       */
    WG_ERR_WORKSPACE = -3,   /* workspace too small or misaligned (needs 256 B alignment) */
    WG_ERR_CUDA = -4         /* CUDA runtime error (message holds cudaGetErrorString)     */
};

/* Library / ABI identification. */
int wg_abi_version(void);
/* Thread-local description of the last failure on this thread ("" if none). */
const char* wg_last_error(void);

/* ------------------------------------------------------------------------------------
 * GCN-GRU forward — replaces `GCN_GRU.forward(adj_matrix, attr_matrix)`
 * (src/step6_gcn_gru_combined_model.py:13-27; called at src/main.py:66,102), i.e.
 *   conv1 -> conv2 (src/step5_gcn_layer_model.py:13-23) -> flatten [T, S*F_out]
 *   -> nn.GRU(batch_first, h0 = 0) -> every hidden state.
 *
 *   adj   [S, S]                 normalised adjacency (src/step2_graph_builder.py:38 -> main.py:26)
 *   x     [B, T, S, F_in]        step4 window layout (src/step4_sequence_preparer.py:13)
 *   w1    [F_in, F_hid], b1 [F_hid]      conv1.weight / conv1.bias   (in x out, not transposed)
 *   w2    [F_hid, F_out], b2 [F_out]     conv2.weight / conv2.bias
 *   w_ih  [3H, S*F_out]          gru.weight_ih_l0  (gate rows r, z, n)
 *   w_hh  [3H, H]                gru.weight_hh_l0
 *   b_ih  [3H], b_hh [3H]        gru.bias_ih_l0 / gru.bias_hh_l0
 *   out   [B, T, H]              (the reference, batch 1 only, returns out[0])
 *
 * The reference accepts B == 1 only (step6:20); this entry point is batch-generalised:
 * sequences are independent (h0 = 0 for each).
 *
 * `chunk` = sequences processed per internal pass (bounds the workspace); 0 = default.
 * `flags`: 0 = every contraction as FP32 FMA (the reference's arithmetic, different summation
 *   order).  WG_FLAG_TENSOR_CORES = the GRU input projection (65 % of the FLOPs) and, for H <= 128,
 *   the recurrent product h.W_hh^T run on the tcgen05 tensor cores: each operand row (a row of
 *   U = the GCN output, of W_ih, of W_hh; h as a whole) is scaled by a power of two that puts its
 *   largest magnitude in [2^14, 2^15), then split into two fp16 parts (x = hi + lo, 22 significant
 *   bits for every element down to 2^-17 of its row's largest), and a product is hi*hi + hi*lo +
 *   lo*hi with fp32 accumulation, unscaled once in fp32.  The error against fp64 is therefore the
 *   same size as the FP32 path's at any operand scale (row maxima from 2^-49 to 2^78; beyond, the
 *   scale stops at 2^+-63), no operand overflows fp16, and rescaling a model's operands by powers
 *   of two leaves the result bit-identical.  The path is held to the same 1e-5 parity bar.  Results
 *   do not depend on how a batch is split.  The workspace must be sized with the same flags.
 *
 * The workspace queries of the forward (this one, the CSR and the host-buffer ones below) return 0
 * for every shape (dims, chunk and flags) their entry point rejects, and wg_last_error() says why.
 * The entry point checks the shape first and returns the same code and text before it looks at
 * pointers or the workspace and before it launches anything.
 * ---------------------------------------------------------------------------------- */
size_t wg_gcn_gru_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                  int64_t chunk, int flags);

int wg_gcn_gru_forward_f32(const float* adj, const float* x, const float* w1, const float* b1,
                           const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                           const float* b_ih, const float* b_hh, float* out, int64_t B, int T, int S,
                           int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                           size_t workspace_bytes, int device, void* stream);

/* Same forward with the adjacency given as CSR (int32 row pointers [S+1], column indices and fp32
 * values [nnz], device pointers): the scaled-shape path — thousands of stations with a few
 * neighbours each, GCN hidden width up to 512 (F_in, F_out <= 16).  Used for BASELINE.json's
 * 4096-station kNN configuration; the dense entry point above is the tuned path for the shipped
 * 7- / 34-station models. */
size_t wg_gcn_gru_csr_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                      int64_t chunk, int flags);
int wg_gcn_gru_forward_csr_f32(const int32_t* rowptr, const int32_t* colidx, const float* vals,
                               const float* x, const float* w1, const float* b1, const float* w2,
                               const float* b2, const float* w_ih, const float* w_hh, const float* b_ih,
                               const float* b_hh, float* out, int64_t B, int T, int S, int F_in,
                               int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                               size_t workspace_bytes, int device, void* stream);

/* Rolling forecasts from one table — every window's last hidden state, without materialising the windows.
 * Stands in for the reference's windowing (src/step4_sequence_preparer.py:7-27) followed by its evaluation
 * (src/main.py:101-116, which reads the last timestep of each window), for windows that may overlap:
 *   table  [Ttot, S, F_in]  device: the pivoted table (wg_pivot_table_f32)
 *   starts int64 [N]        HOST: window n is table[starts[n] : starts[n] + L]; any order, repeats allowed
 *   out    [N, H]           device: out[n] = h_{L-1} of window n
 * out[n] is bit-identical to out[n, L-1, :] of wg_gcn_gru_forward_f32 (same flags) on the materialised window:
 * GCN and input projection depend only on a table row, so they run once per row of [min start, max start + L),
 * in pieces of at most chunk * L rows, and each window's recurrence (h0 = 0) reads its L rows of input-gate values in
 * place, on the kernel the forward would choose for the same N and chunk.
 *
 * The shapes, chunk and flags are planned as for the forward with T = L and B = N, and rejected with the
 * forward's code and text; the workspace query also returns 0 for N < 0, L < 1 and L > Ttot.  N == 0 returns
 * WG_OK.  The entry point validates `starts` before it looks at the workspace: NULL (N > 0) or a start outside
 * [0, Ttot - L] returns WG_ERR_BAD_ARG naming the window and the value.  The starts are copied to the
 * workspace on `stream` before the call returns, so the caller may reuse the array at once.
 * Workspace: the forward's packed parameters and U scratch of one piece, input-gate values of up to Ttot
 * rows (Ttot * 3H floats, rounded up), N int64 starts. */
size_t wg_gcn_gru_forecast_workspace_bytes(int64_t N, int64_t Ttot, int L, int S, int F_in, int F_hid, int F_out,
                                           int H, int64_t chunk, int flags);
int wg_gcn_gru_forecast_f32(const float* adj, const float* table, const int64_t* starts, const float* w1,
                            const float* b1, const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                            const float* b_ih, const float* b_hh, float* out, int64_t N, int64_t Ttot, int L, int S,
                            int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                            size_t workspace_bytes, int device, void* stream);
/* The same with the adjacency as CSR (rowptr, colidx, vals as for wg_gcn_gru_forward_csr_f32). */
size_t wg_gcn_gru_forecast_csr_workspace_bytes(int64_t N, int64_t Ttot, int L, int S, int F_in, int F_hid,
                                               int F_out, int H, int64_t chunk, int flags);
int wg_gcn_gru_forecast_csr_f32(const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* table,
                                const int64_t* starts, const float* w1, const float* b1, const float* w2,
                                const float* b2, const float* w_ih, const float* w_hh, const float* b_ih,
                                const float* b_hh, float* out, int64_t N, int64_t Ttot, int L, int S, int F_in,
                                int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                                size_t workspace_bytes, int device, void* stream);

/* Same computation with HOST buffers for x (pinned for full overlap) and out: the batch is
 * streamed through the device in `chunk`-sized pieces, H2D copy / compute / D2H copy of
 * consecutive pieces overlapped on internal streams (two compute lanes, so the latency-bound
 * recurrence of one piece overlaps the GCN / projection of the next).  `chunk` = 0 selects pieces of
 * 256 sequences.  Parameters and adj are device
 * pointers (they are the model, resident on the GPU as in src/main.py:27,43).  Blocks
 * until `out_host` is complete.  Replaces the per-window loop of src/main.py:101-103
 * (`model(adj, batch_x)` followed by `.cpu()`). */
size_t wg_gcn_gru_host_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                       int64_t chunk, int flags);

int wg_gcn_gru_forward_host_f32(const float* adj, const float* x_host, const float* w1,
                                const float* b1, const float* w2, const float* b2,
                                const float* w_ih, const float* w_hh, const float* b_ih,
                                const float* b_hh, float* out_host, int64_t B, int T, int S,
                                int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags,
                                void* workspace, size_t workspace_bytes, int device);

/* The evaluation loop of src/main.py:101-116 in one call: the same host-buffer pipeline, but only what the
 * reference's statistics read leaves the GPU — the LAST timestep of every window, de-normalised,
 *   pred_host [B, H] = out[:, T-1, :] * (vmax - vmin) + vmin      (src/main.py:103,116,131,146)
 * i.e. 3S floats per window instead of T*3S.  Workspace: wg_gcn_gru_host_workspace_bytes. */
int wg_gcn_gru_predict_host_f32(const float* adj, const float* x_host, const float* w1,
                                const float* b1, const float* w2, const float* b2,
                                const float* w_ih, const float* w_hh, const float* b_ih,
                                const float* b_hh, float* pred_host, int64_t B, int T, int S,
                                int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags,
                                double vmin, double vmax, void* workspace, size_t workspace_bytes,
                                int device);

/* ------------------------------------------------------------------------------------
 * Single GCN layer — replaces `GraphConvLayer.forward(adj_matrix, attr_matrix)`
 * (src/step5_gcn_layer_model.py:13-23):  out = relu((adj @ attr) @ weight + bias).
 *   attr [R, S, F_in] (R = product of the leading dims),  out [R, S, F_out].
 * No workspace.
 * ---------------------------------------------------------------------------------- */
int wg_gcn_layer_f32(const float* adj, const float* attr, const float* weight, const float* bias,
                     float* out, int64_t R, int S, int F_in, int F_out, int device, void* stream);

/* ------------------------------------------------------------------------------------
 * Stage entry points (the three kernels wg_gcn_gru_forward_f32 chains).  Exposed so the
 * benchmark can time, and the tests can check, each kernel alone.  `workspace` must have
 * been sized by wg_gcn_gru_workspace_bytes for the same dims and flags and must already hold the
 * packed parameters (wg_stage_pack_f32) before stages 2 and 3.
 *   stage_pack  : re-lay w_ih / w_hh / biases for the kernels
 *   stage_gcn   : x [Bc,T,S,F_in] -> U [Bc*T, IP]        (two GCN layers, fused)
 *   stage_inproj: U -> GI [Bc*T, GP] = U . w_ih^T + b     (the GRU input projection)
 *   stage_recur : GI -> out [Bc,T,H]                      (the serial GRU recurrence)
 * Bc must be <= the chunk the workspace was sized for.
 * ---------------------------------------------------------------------------------- */
int wg_stage_pack_f32(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                      int T, int S, int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags,
                      void* workspace, size_t workspace_bytes, int device, void* stream);
int wg_stage_gcn_f32(const float* adj, const float* x, const float* w1, const float* b1,
                     const float* w2, const float* b2, int64_t Bc, int T, int S, int F_in, int F_hid,
                     int F_out, int H, int64_t chunk, int flags, void* workspace, size_t workspace_bytes,
                     int device, void* stream);
int wg_stage_inproj_f32(int64_t Bc, int T, int S, int F_in, int F_hid, int F_out, int H,
                        int64_t chunk, int flags, void* workspace, size_t workspace_bytes, int device,
                        void* stream);
int wg_stage_recur_f32(float* out, int64_t Bc, int T, int S, int F_in, int F_hid, int F_out, int H,
                       int64_t chunk, int flags, void* workspace, size_t workspace_bytes, int device,
                       void* stream);

/* ------------------------------------------------------------------------------------
 * Graph build — replaces `build_graph(df)` after its Mercator step
 * (src/step2_graph_builder.py:16-40; the libm log/tan of :8-13 stay on the host).
 *   xy        [S, 2] fp64 device pointer: (northing, easting) metres per station
 *   adj_f64   [S, S] fp64 out (may be NULL)   D^-1/2 (A+I) D^-1/2, bit-identical to SciPy's
 *             evaluation order (see DESIGN.md)
 *   adj_f32   [S, S] fp32 out (may be NULL)   the `.float()` cast of src/main.py:26
 *   k         0 = dense reference graph; k > 0 = symmetrised k-nearest-neighbour pattern
 *             (edge (i,j) kept iff j in kNN(i) or i in kNN(j); ties -> smaller index), the
 *             synthetic large-graph generator.  Same weights and normalisation.
 *   workspace device scratch of wg_build_graph_workspace_bytes(S, k) bytes.
 * ---------------------------------------------------------------------------------- */
size_t wg_build_graph_workspace_bytes(int S, int k);
int wg_build_graph_f64(const double* xy, double* adj_f64, float* adj_f32, int S, int k,
                       void* workspace, size_t workspace_bytes, int device, void* stream);

/* The same kNN graph (k > 0) straight into CSR, without any S x S matrix (the form
 * wg_gcn_gru_forward_csr_f32 takes; src/step2_graph_builder.py:24-38 builds the dense matrix):
 *   rowptr  int32 [S + 1] out     colidx  int32 [capacity] out, ascending within a row
 *   vals_f64 / vals_f32 [capacity] out (either may be NULL): bit-identical to the non-zeros of
 *             wg_build_graph_f64's matrix (an exact zero never changes a column sum)
 *   capacity  >= S * (2k + 1) entries (an upper bound of the symmetrised pattern incl. self loops);
 *             the number of stored entries is rowptr[S]. */
size_t wg_build_graph_csr_workspace_bytes(int S, int k);
int wg_build_graph_csr_f64(const double* xy, int S, int k, int32_t* rowptr, int32_t* colidx,
                           double* vals_f64, float* vals_f32, int64_t capacity, void* workspace,
                           size_t workspace_bytes, int device, void* stream);

/* Deterministic synthetic station coordinates (SplitMix64 stream, see DESIGN.md):
 *   latlon [S, 2] fp64 device out, uniform in the shipped stations' bounding box. */
int wg_synthetic_coordinates_f64(double* latlon, int S, uint64_t seed, int device, void* stream);

/* ------------------------------------------------------------------------------------
 * step4 windows — replaces `__create_sequences(data, seq_length)`
 * (src/step4_sequence_preparer.py:7-27) for the numeric block of the pivoted table.
 *   table  [Ttot, S, F] fp32 device: columns 2:15 of the reference's [time, station, 15] table
 *          (feature f = column f + 2; label column 13 = feature 11)
 *   perm   int64 [N] device, window order (the reference shuffles, :23-26); NULL = identity
 *   x      [N, L, S, F]        x[n] = table[perm[n]*L : (perm[n]+1)*L]                  (:13)
 *   y      [N, L, horizons*S]  y[n, l, k*S+s] = table[perm[n]*L + l + 1 + k, s, label_f] (:14-18)
 *   Either of x / y may be NULL.  N*L + horizons <= Ttot is required (the reference would build
 *   ragged label arrays otherwise); wg_num_windows gives the largest such N.
 *
 * De-normalised last-step predictions — replaces `outputs * (wind_max - wind_min) + wind_min`
 * (src/main.py:103) restricted to the last timestep the evaluation reads (main.py:116,131,146):
 *   out [B, T, H] -> pred [B, H], fp32 arithmetic with NumPy's two roundings.
 * ---------------------------------------------------------------------------------- */
/* Pivot of the long table — replaces the per-station stacking loop of `generate_sequences`
 * (src/step4_sequence_preparer.py:36-47):
 *   station int32 [n_rows] device: rank of each row's station name in np.unique order (:38)
 *   values  [n_rows, F] fp32 device: the numeric columns 2:15 of the long table, file order
 *   table   [Ttot, S, F] out: table[t][s] = the t-th row (file order) of station s
 *   counts  int32 [S] out: rows found per station (the reference requires them all equal; rows
 *           beyond Ttot are not stored). */
int wg_pivot_table_f32(const int32_t* station, const float* values, float* table, int32_t* counts,
                       int64_t n_rows, int S, int F, int64_t Ttot, int device, void* stream);

int64_t wg_num_windows(int64_t Ttot, int L, int horizons);
int wg_make_windows_f32(const float* table, const int64_t* perm, float* x, float* y, int64_t Ttot, int S,
                        int F, int L, int label_f, int horizons, int64_t N, int device, void* stream);
int wg_denorm_last_step_f32(const float* out, float* pred, int64_t B, int T, int H, double vmin,
                            double vmax, int device, void* stream);

/* ------------------------------------------------------------------------------------
 * Training step — replaces the body of the reference's training loop (src/main.py:64-77):
 *   outputs = model(adj_matrix, batch_x)            -> wg_gcn_gru_forward_train_f32
 *   loss = nn.MSELoss()(outputs, batch_y)  (:49,:72) -> wg_mse_loss_grad_f32 (loss and dL/d outputs)
 *   loss.backward()                        (:76)     -> wg_gcn_gru_backward_f32
 *   optimizer.step()  (torch.optim.Adam, :52,:77)    -> wg_adam_step_f32
 * FP32 throughout, dense adjacency, F_in / F_hid / F_out <= 16, H <= 106 (the limit the
 * planner enforces: W_hh and the recurrent state resident in shared
 * memory; the shipped models).  B * T may be at most 2,097,024 rows (16,383 tiles of 128): the
 * backward re-lays the input-gate gradients in one pass, and the planner rejects larger batches.
 *
 * The forward is the inference path's three kernels; the recurrence additionally saves the gate
 * values [r | z | n | W_hn h + b_hn] per (sequence, step).  `workspace` (sized by
 * wg_gcn_gru_train_workspace_bytes for the same dims, 256-byte aligned) carries the saved state
 * from the forward to the backward call and must not be touched in between.
 *
 * Backward: `out` is the forward's result, `d_out` [B, T, H] the gradient w.r.t. every hidden
 * state.  `grads` receives (overwrites) ONE flat fp32 buffer of wg_gcn_gru_param_count floats in
 * state_dict order  conv1.weight | conv1.bias | conv2.weight | conv2.bias | gru.weight_ih_l0 |
 * gru.weight_hh_l0 | gru.bias_ih_l0 | gru.bias_hh_l0  — one bucket, so that a data-parallel job
 * all-reduces it with a single collective.  No gradient is produced for x or adj (data).
 * All reductions run in a fixed order: the gradients are bit-reproducible run to run.
 * ---------------------------------------------------------------------------------- */
size_t wg_gcn_gru_param_count(int S, int F_in, int F_hid, int F_out, int H);
size_t wg_gcn_gru_train_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H);
int wg_gcn_gru_forward_train_f32(const float* adj, const float* x, const float* w1, const float* b1,
                                 const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                                 const float* b_ih, const float* b_hh, float* out, int64_t B, int T, int S,
                                 int F_in, int F_hid, int F_out, int H, void* workspace, size_t workspace_bytes,
                                 int device, void* stream);
int wg_gcn_gru_backward_f32(const float* adj, const float* x, const float* w1, const float* b1, const float* w2,
                            const float* b2, const float* w_ih, const float* w_hh, const float* out,
                            const float* d_out, float* grads, int64_t B, int T, int S, int F_in, int F_hid,
                            int F_out, int H, void* workspace, size_t workspace_bytes, int device, void* stream);

/* Mean-squared-error loss over n elements and its gradient: *loss = mean((out - y)^2) (device
 * scalar), d_out = 2 (out - y) / n (may be NULL).  workspace: wg_mse_workspace_bytes() bytes. */
size_t wg_mse_workspace_bytes(void);
int wg_mse_loss_grad_f32(const float* out, const float* y, int64_t n, float* d_out, float* loss, void* workspace,
                         size_t workspace_bytes, int device, void* stream);

/* One torch.optim.Adam step (no weight decay / amsgrad) over flat buffers of n floats; `step` is
 * the 1-based step count, `grad_scale` multiplies the gradient first (1 / world size after a
 * sum all-reduce). */
int wg_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                     double beta1, double beta2, double eps, int64_t step, double grad_scale, int device,
                     void* stream);

/* ------------------------------------------------------------------------------------
 * Measurement helper: sustained FP32 FFMA throughput of this device in TFLOP/s (2 flops per
 * FFMA), measured with CUDA events over `iters` launches of a register-resident FFMA loop.
 * Used by bench.py as the FP32 roofline denominator.  Returns < 0 on error.
 * ---------------------------------------------------------------------------------- */
double wg_measure_ffma_tflops(int device, int iters);

#ifdef __cplusplus
}
#endif
#endif /* WINDGNN_B200_H */
