/* mogstn.h -- C ABI of libmogstn.so: the B200 (sm_100a) implementation of the MOG-ASR hot path.
 *
 * The reference (taufikxu/MOG-ASR) is pure Python on TensorFlow 1.12 and has no FFI of its own; the
 * entry points below are what a binding for its hot path would need, one per reference interface:
 *
 *   mog_stn_forward            <- transformer(U, theta, out_size)          air/transformer.py:18,173-175
 *                                 batch_transformer(U, thetas, out_size)   air/transformer.py:178-195 (u_batch_div = T)
 *   mog_stn_backward           <- TF autodiff of that graph                air/air_number_bbox_location.py:1098
 *   mog_stn_corners            <- the clipped corner indices x0,x1,y0,y1   air/transformer.py:79-87 (parity probe)
 *   mog_stn_write_composite_*  <- write call site + canvas compositing     air/air_number_bbox_location.py:592-600,:718-727
 *   mog_asr_reg_*              <- ASR regularisers                         air/air_number_bbox_location.py:645-681,:970-1069
 *   mog_bce_recon_*            <- reconstruction cross-entropy             air/air_number_bbox_location.py:945-968
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer to fp32 (or int32 where stated), dense row-major, owned by the
 *     caller.  The library allocates nothing, keeps no state, never synchronises: each call enqueues
 *     its kernels on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream) and returns.
 *     All calls are CUDA-graph capturable and re-entrant.
 *   - Layout is the reference's NHWC: U[B][Hs][Ws][C], out[B][Ho][Wo][C], theta[B][6] (= [B][2][3]).
 *   - Return value: 0 on success; a negative mog_status on bad arguments; a positive cudaError_t value
 *     if a launch failed.  Nothing is thrown across the ABI.  mog_last_error_string() describes the
 *     last failure on the calling thread.
 *   - There is no CPU fallback anywhere in this library.
 *   - Non-finite theta (e.g. 1/s = inf when a sigmoid scale underflows to 0, air_number_bbox_location.py:570-578) is
 *     undefined in the reference (int32(floor(NaN)) is platform-defined).  Here a NaN or infinite source coordinate never
 *     indexes out of bounds: the row / column counts as out of range, the forward writes what out-of-range pixels get
 *     (exactly +0 for rows; NaN propagates through the weights of a column) and the backward contributes nothing for it.
 *     The reference would carry NaN into the loss and zero it only at the gradient level (:1105-1108); a caller that
 *     wants that behaviour must test theta for finiteness itself.
 */
#ifndef MOGSTN_H_
#define MOGSTN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOG_ABI_VERSION 1

#if defined(__GNUC__)
#define MOG_API __attribute__((visibility("default")))
#else
#define MOG_API
#endif

typedef enum {
    MOG_OK = 0,
    MOG_ERR_NULL = -1,        /* a required pointer is NULL */
    MOG_ERR_DIM = -2,         /* non-positive or inconsistent dimension */
    MOG_ERR_OVERFLOW = -3,    /* an element count does not fit the index type used (reference: silent int32 wrap) */
    MOG_ERR_UNSUPPORTED = -4  /* shape outside what the kernels are built for (see message) */
} mog_status;

MOG_API int mog_version(void);
/* Copies the calling thread's last error message (NUL terminated) into buf; returns its full length. */
MOG_API int mog_last_error_string(char* buf, size_t n);

/* out[b] = bilinear_sample(U[b / u_batch_div]; theta[b])       (transformer.py:56-171)
 * B counts thetas/outputs; U holds B / u_batch_div images (u_batch_div >= 1 must divide B). */
MOG_API int mog_stn_forward(const float* U, const float* theta, float* out, int64_t B, int Hs, int Ws, int C, int Ho,
                    int Wo, int u_batch_div, void* stream);

/* corners: int32 [4][B*Ho*Wo] in the order x0, x1, y0, y1 after clipping (transformer.py:79-87). */
MOG_API int mog_stn_corners(const float* theta, int32_t* corners, int64_t B, int Hs, int Ws, int Ho, int Wo,
                    void* stream);

/* Gradients of sum(gout * out).  dU (nullable) is [B / u_batch_div][Hs][Ws][C] and is fully overwritten
 * (no pre-zeroing needed); dtheta (nullable) is [B][6] and fully overwritten. */
MOG_API int mog_stn_backward(const float* U, const float* theta, const float* gout, float* dU, float* dtheta,
                     int64_t B, int Hs, int Ws, int C, int Ho, int Wo, int u_batch_div, void* stream);

/* Host-buffer form of forward + backward in one call (what one `sess.run([out, grads], feed_dict)` of
 * the reference does, train_air_pr.py:294-295): U_h, theta_h, gout_h, out_h, dU_h (nullable), dtheta_h
 * (nullable) are HOST pointers (pinned memory for full PCIe rate); the batch is cut into chunks that are
 * copied in, sampled, differentiated and copied out on `nstreams` CUDA streams so H2D, kernels and D2H
 * overlap.  workspace_d is caller-owned device scratch of at least mog_stn_host_workspace_bytes(...)
 * bytes.  Unlike the device entry points this one waits for its streams before returning. */
MOG_API int mog_stn_fwd_bwd_host(const float* U_h, const float* theta_h, const float* gout_h, float* out_h, float* dU_h,
                         float* dtheta_h, int64_t B, int Hs, int Ws, int C, int Ho, int Wo, int64_t chunk,
                         void* workspace_d, size_t workspace_bytes, void* const* streams, int nstreams);
/* Scratch needed by mog_stn_fwd_bwd_host for a given chunk size and stream count (returns 0 on bad args). */
MOG_API size_t mog_stn_host_workspace_bytes(int64_t chunk, int Hs, int Ws, int C, int Ho, int Wo, int nstreams);

/* batch_transformer form of the same (air/transformer.py:178-195): U_h [B][Hs][Ws][C] holds B source images, every one
 * of them sampled with T transforms: thetas_h [B][T][6], gout_h / out_h [B][T][Ho][Wo][C] (the reference's output order,
 * index b*T + t), dtheta_h [B][T][6] (nullable), dU_h [B][Hs][Ws][C] (nullable) = the gradient summed over the T
 * transforms.  A source image crosses the bus once for its T transforms, dU once (or never: the AIR read site asks for
 * dtheta only).  gout_h may be NULL when no gradient is requested.  chunk counts source images. */
MOG_API int mog_stn_batch_fwd_bwd_host(const float* U_h, const float* thetas_h, const float* gout_h, float* out_h, float* dU_h,
                               float* dtheta_h, int64_t B, int T, int Hs, int Ws, int C, int Ho, int Wo, int64_t chunk,
                               void* workspace_d, size_t workspace_bytes, void* const* streams, int nstreams);
MOG_API size_t mog_stn_batch_host_workspace_bytes(int64_t chunk, int T, int Hs, int Ws, int C, int Ho, int Wo, int nstreams);

/* canvas_out[b] = canvas_in[b] + (stop_sum[b] < threshold ? z_pres[b] * sample(U[b]; theta[b]) : 0)
 * U is the [B][Hw][Ww] window (C = 1), canvases are [B][Hc][Wc]; canvas_out may alias canvas_in (the
 * in-place form touches only pixels that change).  stop_sum NULL = every image active. */
MOG_API int mog_stn_write_composite_forward(const float* U, const float* theta, const float* z_pres,
                                    const float* stop_sum, float threshold, const float* canvas_in,
                                    float* canvas_out, int64_t B, int Hw, int Ww, int Hc, int Wc, void* stream);

/* Given gcanvas = d loss / d canvas_out: dU [B][Hw][Ww], dtheta [B][6], dz [B] (each nullable, each fully
 * overwritten).  d loss / d canvas_in is gcanvas itself and is not written. */
MOG_API int mog_stn_write_composite_backward(const float* U, const float* theta, const float* z_pres,
                                     const float* stop_sum, float threshold, const float* gcanvas, float* dU,
                                     float* dtheta, float* dz, int64_t B, int Hw, int Ww, int Hc, int Wc,
                                     void* stream);

/* The two sampler calls of an AIR step with theta built in the kernel from the model's (s, x, y) -- SURVEY 8(f)2: "pass 3
 * floats, return ds, dx, dy directly".  shift [B][2] = (x, y) (tanh output, :435-436), scale [B] = s (sigmoid output,
 * :458-459); read: theta = [[s,0,x],[0,s,y]] (air_number_bbox_location.py:511-531), write: theta = [[1/s,0,-x/s],[0,1/s,-y/s]]
 * (:563-584), evaluated with the same fp32 expressions as mog_air_thetas_forward, so outputs equal those of the theta-taking
 * entry points bit for bit.  C = 1.  The backward writes d_shift [B][2] and d_scale [B] (fully overwritten); g_shift_in /
 * g_scale_in (nullable) are added to them -- the gradient that reached the same (s, x, y) through the step's other sampler
 * call -- so no accumulation kernel is needed.  dU / dz nullable as in the theta-taking forms. */
MOG_API int mog_stn_read_sxy_forward(const float* U, const float* shift, const float* scale, float* out, int64_t B, int Hs,
                             int Ws, int Ho, int Wo, void* stream);
MOG_API int mog_stn_read_sxy_backward(const float* U, const float* shift, const float* scale, const float* gout,
                              const float* g_shift_in, const float* g_scale_in, float* dU, float* d_shift,
                              float* d_scale, int64_t B, int Hs, int Ws, int Ho, int Wo, void* stream);
MOG_API int mog_stn_write_composite_sxy_forward(const float* U, const float* shift, const float* scale, const float* z_pres,
                                        const float* stop_sum, float threshold, const float* canvas_in,
                                        float* canvas_out, int64_t B, int Hw, int Ww, int Hc, int Wc, void* stream);
MOG_API int mog_stn_write_composite_sxy_backward(const float* U, const float* shift, const float* scale, const float* z_pres,
                                         const float* stop_sum, float threshold, const float* gcanvas,
                                         const float* g_shift_in, const float* g_scale_in, float* dU, float* d_shift,
                                         float* d_scale, float* dz, int64_t B, int Hw, int Ww, int Hc, int Wc,
                                         void* stream);

/* The write call site of the AIR loop on HOST buffers (air_number_bbox_location.py:592-600 and :718-727): T windows per
 * image are written onto ONE canvas per image, canvas[b] = sum_t z[t][b] * sample(W[t][b]; theta[t][b]) (accumulated in
 * step order, exactly as T calls of mog_stn_write_composite_forward on a zero canvas), and gcanvas_h = d loss / d canvas
 * is differentiated back to every step's window, theta and z_pres.  Step-major arrays (the model's stacks): W_h
 * [T][B][Hw][Ww], thetas_h [T][B][6], z_h [T][B]; canvas_h / gcanvas_h [B][Hc][Wc]; dW_h, dtheta_h, dz_h (each nullable)
 * like W_h, thetas_h, z_h.  gcanvas_h may be NULL when no gradient is requested.  The canvas crosses the bus once per
 * image instead of once per glimpse.  chunk counts images; waits for its streams before returning. */
MOG_API int mog_stn_write_composite_host(const float* W_h, const float* thetas_h, const float* z_h, const float* gcanvas_h,
                                 float* canvas_h, float* dW_h, float* dtheta_h, float* dz_h, int64_t B, int T, int Hw,
                                 int Ww, int Hc, int Wc, int64_t chunk, void* workspace_d, size_t workspace_bytes,
                                 void* const* streams, int nstreams);
MOG_API size_t mog_stn_write_composite_host_workspace_bytes(int64_t chunk, int T, int Hw, int Ww, int Hc, int Wc, int nstreams);

/* ---- ASR regularisers (one fused per-image kernel) ------------------------------------------------ */
#define MOG_ASR_MAX_STEPS 16
#define MOG_ASR_MAX_COUNTS 8
#define MOG_ASR_NUM_COMPONENTS 6 /* pr_num, num_min, area, out, size, overlap  (the reference's log_variables) */

typedef struct {
    float canvas_size;                  /* cs */
    int max_steps;                      /* reference max_steps (columns of the objective) */
    int num_counts;                     /* K = len(-dn) */
    int counts[MOG_ASR_MAX_COUNTS];     /* c_k */
    float gamma_num, gamma_margin, gamma_elem, gamma_bbox, gamma_size, gamma_area; /* -gn -gm -gne -gb -gs -ga */
    float size_min, size_max;           /* constrains_area_minmax */
} mog_asr_config;

/* psum[t] += sum_b sigmoid(log_odds[b][t]); caller zeroes psum[T] first (and all-reduces it across ranks
 * for global-batch semantics, air_number_bbox_location.py:982). */
MOG_API int mog_asr_reg_colsum(const float* log_odds, float* psum, int64_t B, int T, void* stream);

/* per_image[b] = pr_loss[b] + L_elem[b]; components [B][6] nullable; margin[1] = L_margin computed from
 * psum * inv_global_batch.  log_odds [B][T], shifts [B][T][2], scales [B][T]. */
MOG_API int mog_asr_reg_forward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                        float inv_global_batch, int64_t B, int T, const mog_asr_config* cfg, float* per_image,
                        float* components, float* margin, void* stream);

/* Gradients of sum_b g_per_image[b]*per_image[b] + g_margin[0]*margin. */
MOG_API int mog_asr_reg_backward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                         float inv_global_batch, const float* g_per_image, const float* g_margin, int64_t B,
                         int T, const mog_asr_config* cfg, float* d_log_odds, float* d_shifts, float* d_scales,
                         void* stream);

/* The same regularisers over the steps the reference loop executes (air_number_bbox_location.py:386-390 stops as soon as
 * no image of the batch is active), for a step that always runs T iterations but must train the reference's objective.
 * psum has 2T floats: psum[0:T) as above, psum[T:2T) the number of active images after each step over the GLOBAL batch
 * (the caller zeroes all 2T floats, and all-reduces them in one exchange across ranks).
 *   colsum_steps: also adds sum_b active[t][b] != 0 into psum[T + t]; active is the [T][B] byte stack of the loop.
 *   Executed steps Te = 1 + (first t in [0, T-2] with psum[T + t] == 0), or T if there is none.  Only "count > 0" is
 *   used, so the rounding of large counts cannot change Te.
 *   forward_steps / backward_steps: every sum, mean and the margin run over t < Te (the area mean divides by Te); the
 *   arrays keep row stride T.  The backward writes exact zeros into d_log_odds, d_shifts and d_scales at t >= Te (all
 *   three stay fully overwritten).  steps_out[1] (int32, nullable) receives Te.  psum is required whatever gamma_margin
 *   is.  With B = 0 the forward still writes margin and steps_out (a rank may hold no images while others do). */
MOG_API int mog_asr_reg_colsum_steps(const float* log_odds, const unsigned char* active, float* psum, int64_t B, int T,
                             void* stream);
MOG_API int mog_asr_reg_forward_steps(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                              float inv_global_batch, int64_t B, int T, const mog_asr_config* cfg, float* per_image,
                              float* components, float* margin, int32_t* steps_out, void* stream);
MOG_API int mog_asr_reg_backward_steps(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                               float inv_global_batch, const float* g_per_image, const float* g_margin, int64_t B,
                               int T, const mog_asr_config* cfg, float* d_log_odds, float* d_shifts, float* d_scales,
                               void* stream);

/* ---- reconstruction loss (the canvas epilogue right after the hot path) ------------------------------
 * air/air_number_bbox_location.py:945-968: r = clip(canvas, 0, 1);
 * loss[b] = -sum_p images*log(r + 1e-10) + (1 - images)*log(1 - r + 1e-10);  mse[b] = sum_p (images - r)^2 (nullable).
 * canvas, images: [B][P].  Backward: dcanvas[b][p] = g_loss[b] * d loss[b] / d canvas[b][p] (fully overwritten). */
MOG_API int mog_bce_recon_forward(const float* canvas, const float* images, float* loss, float* mse, int64_t B, int P,
                          void* stream);
MOG_API int mog_bce_recon_backward(const float* canvas, const float* images, const float* g_loss, float* dcanvas,
                           int64_t B, int P, void* stream);

/* ---- per-step elementwise math of the AIR loop body, fused ([B]-wide, latency-bound) ---------------
 * gauss_sample: latent = mean + eps*sqrt(exp(logvar)); squashed = act(latent), act 0 none / 1 tanh / 2 sigmoid
 *   (_sample_from_mvn :180-184 with :433-436, :456-459; air/vae.py:28-31).  n = number of elements.
 *   backward: g_latent / g_squashed nullable; d_mean, d_logvar fully overwritten.
 * thetas: shift[B][2], scale[B] -> theta_r = [[s,0,x],[0,s,y]] (:511-531), theta_w = [[1/s,0,-x/s],[0,1/s,-y/s]] (:563-584).
 * zpres: Concrete sample (air/concrete.py:20-27), z_pres = sigmoid(y) (:631), stop_out = stop_in + 1 - z_pres (:712),
 *   active_prev / active = stop < threshold before / after the update (1 byte each). */
MOG_API int mog_air_gauss_sample_forward(const float* mean, const float* logvar, const float* eps, float* latent,
                                 float* squashed, int64_t n, int act, void* stream);
MOG_API int mog_air_gauss_sample_backward(const float* logvar, const float* eps, const float* squashed, const float* g_latent,
                                  const float* g_squashed, float* d_mean, float* d_logvar, int64_t n, int act,
                                  void* stream);
MOG_API int mog_air_thetas_forward(const float* shift, const float* scale, float* theta_r, float* theta_w, int64_t B,
                           void* stream);
MOG_API int mog_air_thetas_backward(const float* shift, const float* scale, const float* g_theta_r, const float* g_theta_w,
                            float* d_shift, float* d_scale, int64_t B, void* stream);
MOG_API int mog_air_zpres_forward(const float* log_odds, const float* u, const float* stop_in, float temperature,
                          float threshold, float* y_pre, float* z_pres, float* stop_out, unsigned char* active_prev,
                          unsigned char* active, int64_t B, void* stream);
MOG_API int mog_air_zpres_backward(const float* z_pres, const float* g_y, const float* g_z, float temperature,
                           float* d_log_odds, int64_t B, void* stream);

/* LSTM cell pointwise part (tf.nn.rnn_cell.LSTMCell, air_number_bbox_location.py:865-872): gates [B][4H] in the order
 * i, j, f, o; c' = sigmoid(f + 1)*c + sigmoid(i)*tanh(j); h' = sigmoid(o)*tanh(c').  gates2 (nullable) is added to gates
 * first (the step-invariant part of the cell input, computed once per training step); d_gates is the gradient w.r.t. the
 * sum, i.e. w.r.t. both.  backward: g_h / g_c nullable. */
MOG_API int mog_air_lstm_pointwise_forward(const float* gates, const float* gates2, const float* c_prev, float* c_new, float* h_new,
                                   int64_t B, int H, void* stream);
MOG_API int mog_air_lstm_pointwise_backward(const float* gates, const float* gates2, const float* c_prev, const float* c_new,
                                    const float* g_h, const float* g_c, float* d_gates, float* d_c_prev, int64_t B, int H,
                                    void* stream);

/* The four KL terms of the ELBO for all executed steps at once (air_number_bbox_location.py:690-787, masked and summed
 * as at :930-935).  Inputs are [T][B][..] stacks: y_pre / prior_lo / post_lo [T][B] (Concrete KL, air/concrete.py:30-64,
 * equal temperatures), active_prev / active [T][B] bytes (stopping_sum < threshold before / after the step's update),
 * sc_mean / sc_lv [T][B] (fixed scale prior), sh_* and g_sh_* [T][B][2] (learned shift prior), v_mean / v_lv [T][B][L].
 * kl[b] = sum_t active_prev*z_pres_kl + active*(scale_kl + shift_kl + vae_kl); components [B][4] (nullable) holds the four
 * per-image sums the reference logs.  Backward: every d_* is fully overwritten with g_kl[b] * d kl[b] / d input. */
MOG_API int mog_air_kl_forward(const float* y_pre, const float* prior_lo, const float* post_lo, const unsigned char* active_prev,
                       const unsigned char* active, const float* sc_mean, const float* sc_lv, const float* sh_mean,
                       const float* sh_lv, const float* g_sh_mean, const float* g_sh_lv, const float* v_mean,
                       const float* v_lv, int64_t B, int T, int L, float temperature, float scale_prior_mean,
                       float scale_prior_var, float vae_prior_mean, float vae_prior_var, float* kl, float* components,
                       void* stream);
MOG_API int mog_air_kl_backward(const float* y_pre, const float* prior_lo, const float* post_lo, const unsigned char* active_prev,
                        const unsigned char* active, const float* sc_mean, const float* sc_lv, const float* sh_mean,
                        const float* sh_lv, const float* g_sh_mean, const float* g_sh_lv, const float* v_mean,
                        const float* v_lv, int64_t B, int T, int L, float temperature, float scale_prior_mean,
                        float scale_prior_var, float vae_prior_mean, float vae_prior_var, const float* g_kl,
                        float* d_y_pre, float* d_prior_lo, float* d_post_lo, float* d_sc_mean, float* d_sc_lv,
                        float* d_sh_mean, float* d_sh_lv, float* d_g_sh_mean, float* d_g_sh_lv, float* d_v_mean,
                        float* d_v_lv, void* stream);

/* ---- detection metrics of the evaluation pass ------------------------------------------------------------
 * air/evaluation_detection.py:29-98 for a whole batch in one launch.  gt_pos / gt_size: [B][G][2] int32 (x, y) and (w, h)
 * of each ground-truth box, the first gt_num[b] valid; inf_shifts [B][T][2], inf_scales [B][T] float64 (the model's
 * fp32 outputs widened, as numpy does), the first inf_num[b] valid; G, T <= MOG_DET_MAX_BOXES; counts are clamped to
 * G / T.  Outputs per image: precision, recall [B][11] (thresholds 0.5 + 0.05 i, strict >), gt_max_iou,
 * detected_max_iou, global_iou [B] (matched IoU sum / max(#gt, #inferred)); the reference returns their batch means. */
#define MOG_DET_MAX_BOXES 8
MOG_API int mog_detection_eval(const int* gt_pos, const int* gt_size, const int* gt_num, const double* inf_shifts,
                       const double* inf_scales, const int* inf_num, int64_t B, int G, int T, double csize,
                       double* precision, double* recall, double* gt_max_iou, double* detected_max_iou,
                       double* global_iou, void* stream);

/* ---- synthetic dataset: object placement (the step before the hot path) ------------------------------------
 * multi_mnist.py:110-221 / multi_dsprites.py:92-302 for a whole batch in one launch: per canvas a count from
 * counts[0..num_counts) (host array), per object a sprite id in [0, num_sprites), a square size in [size_min, size_max]
 * pixels (one per canvas when share_size) and a position inside the margins found by <= 100 rejection draws against
 * the objects already placed; mode 0 = the reference's bounding_boxes_overlap as written (x-intervals only), mode 1 =
 * true box intersection (the pixel-overlap rule is mog_synth_place_pixels below).  Draws are a counter-based hash of
 * (seed, first_canvas + b, ...): reproducible, independent of B.  Outputs: num [B], pos / size [B][max_objects][2] (x, y) / (w, h), sprite [B][max_objects] (int32; unused = 0). */
#define MOG_SYNTH_MAX_OBJECTS 8
#define MOG_SYNTH_MAX_COUNTS 8
#define MOG_SYNTH_MAX_RESTARTS 32
MOG_API int mog_synth_place(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                    int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                    int num_sprites, int* num, int* pos, int* size, int* sprite, void* stream);

/* The same placement with the reference's pixel-overlap rule (multi_mnist.py:53-57,:180-182; its default Multi-MNIST):
 * a candidate is rejected when any canvas pixel where its pasted value is >= 0.05 (the feeder's drop threshold,
 * :153-154) lies within Chebyshev distance `gap` of such a pixel of an object already placed; boxes may overlap, pixels
 * may not (gap = 0: no shared pixel).  The reference's add_buffer is not available, so the exact shape of its buffer is
 * UNPINNED; `gap` is this library's dilation.  Draws, attempts and restarts are those of mog_synth_place (with counts
 * (1,) the two give the same placement).  "Pasted value" is the sampler's write-direction forward of the sprite onto
 * the canvas with theta [[box_scale[w], 0, box_offset[x][w]], [0, box_scale[w], box_offset[y][w]]], evaluated with the
 * forward kernel's arithmetic: sprites [num_sprites][sprite_side][sprite_side] (device fp32), box_scale [size_max + 1]
 * and box_offset [canvas][size_max + 1] (device fp32) the entries t00 and t02 of the caller's paste theta for each
 * (position, size), so that the test is exact for what the caller then pastes.  canvas <= MOG_SYNTH_PIXEL_MAX_CANVAS
 * (else MOG_ERR_UNSUPPORTED).  One warp per canvas.  Outputs as mog_synth_place. */
#define MOG_SYNTH_PIXEL_MAX_CANVAS 128
MOG_API int mog_synth_place_pixels(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                           int num_counts, int size_min, int size_max, int gap, int margin, int share_size,
                           const float* sprites, int num_sprites, int sprite_side, const float* box_scale,
                           const float* box_offset, int* num, int* pos, int* size, int* sprite, void* stream);

/* Rotated objects labelled with their tight boxes (the reference rotates each object and re-crops it to its tight box,
 * multi_mnist.py:144-163), placed under any of the three rules: mode 0 = bounding_boxes_overlap as written, 1 = box
 * intersection, 2 = the pixel-overlap rule of mog_synth_place_pixels.  Count, size, sprite and position draws are those
 * of mog_synth_place; every object also draws an angle index k = draw_int(draw32(seed, canvas, restart, object, 0, 6),
 * 0, num_angles) (redrawn on every restart, like the size) into rot [num_angles][2], a HOST table of (cos, sin) pairs
 * computed by the caller in fp64 (unit vectors to 1e-9, 1 <= num_angles <= MOG_SYNTH_MAX_ANGLES; no trigonometric
 * function is evaluated here).  An object of size w fits the square of side e = min(canvas, ceil(w (|cos| + |sin|)))
 * (fp64), whose position (x, y) is drawn inside the margins (span canvas - e - 2 margin + 1) and about whose centre it
 * is rotated.  Its paste theta, normative, evaluated in fp64 without FMA and rounded to fp32 once per entry, with
 * sc = (w - 1) / (canvas - 1), cx = -1 + (2x + e - 1) / (canvas - 1), cy = -1 + (2y + e - 1) / (canvas - 1):
 *   t00 = cos / sc        t01 = sin / sc        t02 = -(cos cx + sin cy) / sc
 *   t10 = (0 - sin) / sc  t11 = cos / sc        t12 = -(cos cy - sin cx) / sc
 * For (cos, sin) = (1, +0), e = w and theta is box_theta's bit for bit, signed zeros included.
 * A candidate's "pixels" are those where the write-direction forward of its sprite with that theta (mog_stn_forward's
 * arithmetic) is >= 0.05.  The kernel evaluates them over the e-square widened by one pixel; no pixel outside reaches
 * 0.05 for sprite values in [0, 1] and sprite_side < 1000 (the argument is at the kernel).  Their row / column extents
 * are the tight box, tested by the box rules of modes 0 and 1 (widened by `gap`); mode 2 tests the pixels themselves.
 * An object whose mask is empty (a blank sprite) clashes with nothing and is labelled with its e-square.
 * canvas in [2, MOG_SYNTH_PIXEL_MAX_CANVAS] (above: MOG_ERR_UNSUPPORTED), size_min >= 2.  One warp per canvas.
 * Outputs: num, sprite as mog_synth_place; pos / size [B][max_objects][2] the tight box (x, y) / (w, h), not square in
 * general; theta [B][max_objects][6] (device fp32) the paste theta of every placed object (unused slots 0). */
#define MOG_SYNTH_MAX_ANGLES 64
MOG_API int mog_synth_place_rotated(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                            int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                            const float* sprites, int num_sprites, int sprite_side, const double* rot, int num_angles,
                            int* num, int* pos, int* size, int* sprite, float* theta, void* stream);

/* The three placements with the batch's first canvas index read from DEVICE memory: first_canvas points to one int64
 * (>= 0; canvas b of the batch is *first_canvas + b) that the kernel reads when it runs, so that a captured CUDA graph
 * can advance the index between replays (a by-value index would repeat the captured batch).  Every other argument,
 * check and draw is that of the host-index entry point of the same name without _dev, and so is the output for the same
 * index; first_canvas NULL with B > 0 is MOG_ERR_NULL.  A negative index is not checked on the host. */
MOG_API int mog_synth_place_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                        const int* counts, int num_counts, int size_min, int size_max, int gap, int margin, int mode,
                        int share_size, int num_sprites, int* num, int* pos, int* size, int* sprite, void* stream);
MOG_API int mog_synth_place_pixels_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                               const int* counts, int num_counts, int size_min, int size_max, int gap, int margin,
                               int share_size, const float* sprites, int num_sprites, int sprite_side,
                               const float* box_scale, const float* box_offset, int* num, int* pos, int* size, int* sprite,
                               void* stream);
MOG_API int mog_synth_place_rotated_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                                const int* counts, int num_counts, int size_min, int size_max, int gap, int margin, int mode,
                                int share_size, const float* sprites, int num_sprites, int sprite_side, const double* rot,
                                int num_angles, int* num, int* pos, int* size, int* sprite, float* theta, void* stream);

/* ---- two-layer (mean, log-variance) heads of the loop body, fused after the first GEMM ---------------------------------
 * air_number_bbox_location.py:424-460, :472-481.  pre1 [B][2h] = x [W1m | W1v] (first-layer GEMM without bias, computed by
 * the caller); weights in the nn.Linear layout: w1m / w1v [h][K+S] (only the S skip columns at K.. are read), b1* [h],
 * w2m / w2v [O][h+S], b2* [O]; skip [B][S] (S = 0: none), eps [B][O]; act as for gauss_sample.  hidden in {16,32,64,128}.
 * forward: mean, logvar, latent [B][O] (+ squashed when act != 0).
 * backward: g_* nullable gradients of the four outputs; dpre1 [B][2h] and dskip [B][S] are fully overwritten; the
 * second-layer parameter gradients gw2m / gw2v [O][h+S], gb2m / gb2v [O] are ACCUMULATED (atomics) into the given buffers. */
#define MOG_HEAD_MAX_SKIP 2
#define MOG_HEAD_MAX_OUT 2
MOG_API int mog_air_head_forward(const float* pre1, const float* skip, const float* eps, const float* w1m, const float* b1m,
                         const float* w1v, const float* b1v, const float* w2m, const float* b2m, const float* w2v,
                         const float* b2v, int64_t B, int hidden, int K, int S, int O, int act, float* mean, float* logvar,
                         float* latent, float* squashed, void* stream);
MOG_API int mog_air_head_backward(const float* pre1, const float* skip, const float* eps, const float* w1m, const float* b1m,
                          const float* w1v, const float* b1v, const float* w2m, const float* w2v, const float* logvar,
                          const float* squashed, const float* g_mean, const float* g_logvar, const float* g_latent,
                          const float* g_squashed, int64_t B, int hidden, int K, int S, int O, int act, float* dpre1,
                          float* dskip, float* gw2m, float* gb2m, float* gw2v, float* gb2v, void* stream);

/* ---- epilogues of dense layers whose GEMM is the library's -----------------------------------------------------------
 * bias_act: out[b][n] = act(pre[b][n] + bias[n]), act 0 none / 1 relu / 2 softplus / 3 sigmoid (vae.py:16-19,:34-41;
 *   :609-623); out may alias pre.  backward: dpre = g * act'(.) from the saved output y (n = B*N elements; dpre may alias g).
 * bias_gauss: pre [B][2L] = x [Wmean | Wlogvar] -> mean, logvar (biases added) and latent = mean + eps*sqrt(exp(logvar))
 *   (vae.py:21-31); backward: g_* nullable, dpre [B][2L] fully overwritten. */
MOG_API int mog_air_bias_act_forward(const float* pre, const float* bias, float* out, int64_t B, int N, int act, void* stream);
MOG_API int mog_air_bias_act_backward(const float* y, const float* g, float* dpre, int64_t n, int act, void* stream);
MOG_API int mog_air_bias_gauss_forward(const float* pre, const float* bias_mean, const float* bias_logvar, const float* eps,
                               float* mean, float* logvar, float* latent, int64_t B, int L, void* stream);
MOG_API int mog_air_bias_gauss_backward(const float* logvar, const float* eps, const float* g_mean, const float* g_logvar,
                                const float* g_latent, float* dpre, int64_t B, int L, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOGSTN_H_ */
