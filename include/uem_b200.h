/*
 * uem_b200.h -- C-ABI of libuem_b200.so: hand-written sm_100a kernels for UemDA's
 * uncertain-example pseudo-label mining path.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - maps are contiguous NCHW (class/feature planes of H*W pixels, pixel stride 1);
 *   - labels, pseudo-labels and superpixel ids are int64 (the reference's dtypes,
 *     uemda/datasets/basedata.py:77-79,87), probabilities/logits/features are fp32;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - every function returns 0 on success; on failure it returns non-zero and
 *     uem_last_error() describes why (thread-local, valid until the next call);
 *   - no function allocates device memory, synchronises the device or copies to the host:
 *     workspaces are caller-provided (sizes via the *_ws_bytes helpers);
 *   - class count c is limited to UEM_MAX_CLASSES (ISPRS = 6, LoveDA = 7).
 *
 * Each entry point cites the reference interface it replaces (file:line in StuLiu/UemDA).
 */
#ifndef UEM_B200_H
#define UEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define UEM_API __attribute__((visibility("default")))
#else
#define UEM_API
#endif

#define UEM_MAX_CLASSES 8
#define UEM_ABI_VERSION 1

/* label_refine view bits (alignment.py:215 'p', :225 'l', :238 's'; 'all' = all three) */
#define UEM_VIEW_PROTO 1
#define UEM_VIEW_PRED 2
#define UEM_VIEW_SUP 4
#define UEM_VIEW_REGIONS_READY 8 /* uem_mine_refine_select_f32 only: uem_mine_region_phase_f32 already ran on this ws */
#define UEM_VIEW_SIMI_READY 16   /* uem_mine_refine_select_f32 only: uem_mine_proto_phase_f32 already ran on this ws */

/* region reduce ops (torch_scatter.scatter reduce=..., alignment.py:187,245) */
#define UEM_REDUCE_SUM 0
#define UEM_REDUCE_MAX 1
#define UEM_REDUCE_MEAN 2

UEM_API const char* uem_last_error(void);
UEM_API int uem_version(void);
/* number of CUDA kernels this library has launched in this process (monotonic) */
UEM_API int64_t uem_kernel_launches(void);
/* measurement hook: the next uem_label_refine_f32 / uem_mine_refine_select_f32 call on this thread records
 * the two cudaEvent_t (passed as void*) immediately before / after its fused refine kernel */
UEM_API int uem_profile_refine_events(void* start_event, void* stop_event);
/* binds the calling thread to a CUDA device (the library links cudart statically) */
UEM_API int uem_set_device(int device);

/* ---- a1-a4: fused logits pass -------------------------------------------------------
 * soft = mean_heads softmax(bilinear_up(x_head, align_corners=True) / temp)  [train_align_uem.py:158-160,
 * Encoder.py:153-155, alignment.py:311-314]; conf/argmax = max / first-index argmax over classes
 * [pseudo_generation.py:47,148]; entropy = sum_c -p log p [balance.py:372].
 * x1,x2: (b,c,h,w) (x2 may be NULL); outputs (any may be NULL): soft (b,c,H,W), conf (b,H,W),
 * entropy (b,H,W), argmax (b,H,W) int64. */
UEM_API int uem_softmax_conf_entropy_argmax_f32(const float* x1, const float* x2, int b, int c, int h, int w,
                                        int H, int W, float temp, float* soft, float* conf,
                                        float* entropy, int64_t* argmax, void* stream);

/* ---- a2+a3: entropy of a probability map + UVEM weight ---------------------------------
 * balance.py:368-373,396-423.  soft (b,c,HW) -> entropy (b*HW), weight (b*HW) (either may be NULL).
 * coef_left/right are the reference's Python-double coefficients -1/m^2 and -1/(t-m)^2 rounded to
 * fp32 by the caller; inv_gamma = fp32(1/gamma). */
UEM_API int uem_entropy_uvem_weight_f32(const float* soft, int b, int c, int64_t hw, float m, float t,
                                float inv_gamma, float coef_left, float coef_right,
                                float* entropy, float* weight, void* stream);
/* UVEMLoss.get_weight on an arbitrary uncertainty vector, balance.py:396-423 */
UEM_API int uem_uvem_weight_f32(const float* u, int64_t n, float m, float t, float inv_gamma,
                        float coef_left, float coef_right, float* weight, void* stream);
/* detached per-pixel factors of UVEMLoss/UPSLoss.forward, balance.py:372-382 (uvem) / :331-342 (ups):
 * entropy u of soft, gate = (u > t) as uint8, weight = get_weight(u) (1.0 if use_weight==0),
 * valid_cnt[0] += #( u <= t && target != ignore ).  target int64 (b*HW). valid_cnt must be zeroed. */
UEM_API int uem_uvem_terms_f32(const float* soft, const int64_t* target, int b, int c, int64_t hw, float m,
                       float t, float inv_gamma, float coef_left, float coef_right, int use_weight,
                       int64_t ignore_label, float* weight, uint8_t* gate, int64_t* valid_cnt,
                       void* stream);

/* ---- a5: class-wise thresholded pseudo labels ------------------------------------------
 * pseudo_generation.py:59-93 (variant 0) and :24-56 (variant 1).
 * uem_class_max_f32: per-(b,c) max / min over HW pixels of mask (b,c,HW) -> cmax,cmin (b*c);
 *   has_nan[0] set non-zero if any NaN was seen.  ws: uem_class_max_ws_bytes(b,c,hw) bytes. */
UEM_API int64_t uem_class_max_ws_bytes(int b, int c, int64_t hw);
UEM_API int uem_class_max_f32(const float* mask, int b, int c, int64_t hw, float* cmax, float* cmin,
                      int32_t* has_nan, void* ws, void* stream);
/* thr[b,c] = fmaxf(cmax*cutoff_top, cutoff_low) in fp32; strict '>' ; kept iff exactly one class wins */
UEM_API int uem_pseudo_select_f32(const float* mask, const float* cmax, int b, int c, int64_t hw,
                          float cutoff_top, float cutoff_low, int64_t ignore_label, int variant,
                          int64_t* out, void* stream);

/* Class statistics table raised atomically by uem_label_refine_f32: (b, c+2) uint32 =
 * [c order-preserving encodings of the per-class maxima | encoding of -(image minimum) | bad flag (NaN/inf seen)].
 * The caller zeroes it (uem_class_stats_bytes bytes) before the refine call; 0 = untouched slot.
 * uem_select_entropy_stats_f32: a5 (variant 0) fed by that table (no second pass for the class max), plus,
 * optionally, a2 + a3 of the same map in the same pass: entropy (b*hw) and UVEM weight (b*hw).
 * uvem_host: NULL or HOST pointer to {m, t, 1/gamma, coef_left, coef_right}.
 * uem_class_stats_decode_f32: table -> cmax (b*c) and image_min (b) as plain floats (NaN if the bad flag is set),
 * for the reference's range assert (pseudo_generation.py:71). */
UEM_API int64_t uem_class_stats_bytes(int b, int c);
/* tuning switches (an unknown name is refused with an error):
 * "{refine,region,proto}_ctas_per_sm": cap on resident CTAs per SM (0 = occupancy limit; pipelined hosts cap the region-max kernel).
 * L2 eviction-priority hints (results never change): "l2_stream" (default 1) = maps a step touches exactly once (feature maps,
 * full-resolution labels, the selection's outputs and its read of the refined map) are evict_first; "l2_last_use" (default 1) =
 * the refine kernel's reads of soft / ids on the fused chain are evict_first; "l2_region" = 0 | 1 (evict_first, default) | 2
 * (evict_last) for the region-max kernel's reads of soft / ids on the fused chain; "l2_keep" = 0 (default) | 2 (evict_last) for
 * the refine kernel's stores of the refined map, which the selection reads next. */
UEM_API int uem_set_option(const char* name, int value);
UEM_API int uem_select_entropy_stats_f32(const float* mask, const uint32_t* class_stats, int b, int c, int64_t hw,
                                 float cutoff_top, float cutoff_low, int64_t ignore_label, int64_t* out,
                                 const float* uvem_host, float* entropy, float* weight, void* stream);
UEM_API int uem_class_stats_decode_f32(const uint32_t* class_stats, int b, int c, float* cmax, float* image_min,
                               void* stream);

/* ---- a6s/a7 seam: torch_scatter.scatter over superpixel ids -----------------------------
 * alignment.py:187 (sum, int64) and :245 (max, f32).  src element (bi,n,ci) lives at
 * src[bi*src_sb + n*src_sn + ci*src_sc] (element strides: (b,N,c) contiguous = {N*c,c,1};
 * an NCHW map viewed as (b,N,c) = {c*N,1,N}).  index (b,N) int64 in [0,R).  out (b,R,c) dense,
 * untouched slots 0.  ws: uem_region_reduce_ws_bytes(b,R,c). */
UEM_API int uem_i64_minmax(const int64_t* x, int64_t n, int64_t* out_min_max /*[2]*/, void* stream);
UEM_API int64_t uem_region_reduce_ws_bytes(int b, int64_t R, int c);
UEM_API int uem_region_reduce_f32(const float* src, int64_t src_sb, int64_t src_sn, int64_t src_sc,
                          const int64_t* index, int b, int64_t N, int c, int64_t R, int op,
                          float* out, void* ws, void* stream);
UEM_API int uem_region_reduce_i64(const int64_t* src, int64_t src_sb, int64_t src_sn, int64_t src_sc,
                          const int64_t* index, int b, int64_t N, int c, int64_t R, int op,
                          int64_t* out, void* ws, void* stream);

/* ---- a7: Aligner.superpixel_expand, alignment.py:175-192 -------------------------------
 * hard (b,N) int64 in [-1,c) (ignore_label dropped), sup (b,N) int64 in [0,R) -> out (b,N) int64:
 * majority class of the pixel's region (first index on ties), -1 if the region has no labelled pixel.
 * ws: uem_superpixel_expand_ws_bytes(b,R,c). */
UEM_API int64_t uem_superpixel_expand_ws_bytes(int b, int64_t R, int c);
UEM_API int uem_superpixel_expand_i64(const int64_t* hard, const int64_t* sup, int b, int64_t N, int c,
                              int64_t R, int64_t ignore_label, int64_t* out, void* ws, void* stream);

/* ---- a8: DownscaleLabel.forward, alignment.py:484-509 ----------------------------------
 * label (b,H,W) int64 -> out (b,H/s,W/s) int64.  status[0] |= 1 if a label outside
 * {ignore} U [0,n_classes) was seen (the reference's one_hot raises). */
UEM_API int uem_downscale_label_i64(const int64_t* label, int b, int H, int W, int scale, int n_classes,
                            int64_t ignore_label, float min_ratio, int64_t* out, int32_t* status,
                            void* stream);

/* ---- a9: Aligner._pearson_dist, alignment.py:424-451 -----------------------------------
 * nchw: feat (b,k,hw) planar, protos (m,k) row-major -> out (b,m,hw) planar:
 *   out = dist, or 1/dist if reciprocal!=0 (alignment.py:216).  m <= UEM_MAX_CLASSES.
 * rows: feat1 (n,k), feat2 (m,k) row-major -> out (n,m) row-major, any m.
 * ws: uem_pearson_nchw_ws_bytes(b,hw,m,k) for the nchw form, uem_pearson_ws_bytes(m,k) for the rows form. */
UEM_API int64_t uem_pearson_ws_bytes(int m, int k);
UEM_API int64_t uem_pearson_nchw_ws_bytes(int b, int64_t hw, int m, int k);
UEM_API int uem_pearson_dist_nchw_f32(const float* feat, int b, int k, int64_t hw, const float* protos, int m,
                              float eps, int reciprocal, float* out, void* ws, void* stream);
UEM_API int uem_pearson_dist_rows_f32(const float* feat1, int64_t n, int k, const float* feat2, int m,
                              float eps, float* out, void* ws, void* stream);

/* ---- a6: Aligner.label_refine, alignment.py:194-293 ------------------------------------
 * views: bitmask of UEM_VIEW_*.  simi (b,c,h,w): 1/pearson distance at feature resolution (PROTO view);
 * pred1/pred2 (b,c,h,w) logits (pred2 may be NULL) (PRED view); sup (b,H,W) int64 + region_max
 * (b,R,c) from uem_region_reduce_f32(MAX) + ignored_id (device pointer to the batch-global max id,
 * alignment.py:241) (SUP view).  soft (b,c,H,W) -> out (b,c,H,W).
 * class_stats (optional, may be NULL): the (b, c+2) statistics table of `out` described above, zeroed by the
 * caller, consumed by uem_select_entropy_stats_f32.
 * ws: uem_label_refine_ws_bytes(b,c,R,W) bytes (per-region weights of the SUP view + column tables; may be NULL
 * without that view). */
UEM_API int64_t uem_label_refine_ws_bytes(int b, int c, int64_t R, int W);
UEM_API int uem_label_refine_f32(int views, const float* simi, const float* pred1, const float* pred2, int h,
                         int w, const int64_t* sup, const float* region_max, int64_t R,
                         const int64_t* ignored_id, const float* soft, int b, int c, int H, int W,
                         float temp, float* out, uint32_t* class_stats, void* ws, void* stream);

/* ---- fused chain: label_refine -> pseudo_selection in one call, no host sync -----------------
 * tools/train_ssl_uem.py:209-214 (vis_corrected_pseudo_labels.py:185-189).  feat (b,k,h,w), protos (c,k),
 * pred1/pred2 (b,c,h,w), sup (b,H,W) with ids in [0,R) (R = capacity of the region table, >= max id+1),
 * ignored_id: device pointer to the batch-global max id or NULL (then computed from sup, alignment.py:241),
 * soft (b,c,H,W) -> refined (b,c,H,W), hard (b,H,W) int64 (NULL = skip the selection); with hard, optionally the
 * entropy (b,H,W) and UVEM weight (b,H,W) of the refined map (balance.py:372,396-423; uvem_host as above).
 * ws: uem_mine_ws_bytes(...) bytes, ZERO-INITIALISED by the caller before its first use (every call leaves it clean
 * for the next one, so a persistent workspace needs no per-call memset; after a failed call zero it again; a
 * workspace may be shared by calls with different views / feature shapes as long as b, c and R stay the same);
 * ws[0..3] int32 status word: bit 2 = superpixel id outside [0,R);
 * the class statistics table of `refined` is left at byte offset uem_mine_ws_stats_offset(...) of ws. */
UEM_API int64_t uem_mine_ws_bytes(int b, int c, int H, int W, int h, int w, int k, int64_t R);
UEM_API int64_t uem_mine_ws_stats_offset(int b, int c, int H, int W, int h, int w, int k, int64_t R);
/* Multi-GPU form (SURVEY 8e): the region half of the chain on its own.  It needs nothing global, so it can run one step
 * ahead of the exchange; it leaves the per-region weights in ws and the rank-LOCAL max superpixel id (int64) at byte
 * offset uem_mine_ws_maxid_offset(...).  uem_mine_refine_select_f32(views | UEM_VIEW_REGIONS_READY, ..., ignored_id =
 * the batch-global max id) then skips the region pass. */
UEM_API int64_t uem_mine_ws_maxid_offset(int b, int c, int H, int W, int h, int w, int k, int64_t R);
UEM_API int uem_mine_region_phase_f32(const int64_t* sup, int64_t R, const float* soft, int b, int c, int H, int W, int h,
                              int w, int k, float temp, void* ws, void* stream);
/* Same pass, and the last CTA of its region-max kernel also carries the id part of the step's exchange (see
 * uem_xchg_send_f32 with parts = 2 below: same slot, same sequence number; the sums follow with parts = 5 or inside
 * uem_xchg_exchange_fold_ema_f32): this rank's max id is stored into slot `slot` of every rank's region and, when
 * global_id_out is given, the batch-global id (alignment.py:241) is left there once all ranks' ids of this step have
 * arrived (bounded poll).  peer_regions / rank / world / depth as for uem_xchg_send_f32; the slot geometry uses this call's c, k. */
UEM_API int uem_mine_region_phase_xchg_f32(const int64_t* sup, int64_t R, const float* soft, int b, int c, int H, int W, int h,
                                   int w, int k, float temp, void* ws, const void* const* peer_regions, int rank, int world,
                                   int depth, int slot, int64_t* global_id_out, void* stream);
/* The prototype half on its own: 1/Pearson distance of feat (b,k,h,w) to protos (c,k) (alignment.py:215-217) into the
 * similarity slot of ws.  It only depends on the prototype bank, so in a pipelined loop it runs as soon as the EMA of the
 * previous step is done, next to that step's refine / selection kernels; uem_mine_refine_select_f32(views |
 * UEM_VIEW_SIMI_READY, ...) then skips it (feat / protos may be NULL there). */
UEM_API int uem_mine_proto_phase_f32(const float* feat, int k, const float* protos, int b, int c, int H, int W, int h, int w,
                             int64_t R, float eps, void* ws, void* stream);
UEM_API int uem_mine_refine_select_f32(int views, const float* feat, int k, const float* protos,
                               const float* pred1, const float* pred2, int h, int w, const int64_t* sup,
                               int64_t R, const int64_t* ignored_id, const float* soft, int b, int c, int H,
                               int W, float temp, float eps, float cutoff_top, float cutoff_low,
                               int64_t ignore_label, float* refined, int64_t* hard, const float* uvem_host,
                               float* entropy, float* weight, void* ws, void* stream);

/* ---- a13: Aligner.get_prototype_weight_4pixel, alignment.py:295-309 --------------------- */
UEM_API int uem_proto_weight_4pixel_f32(const float* simi, int h, int w, const int64_t* hard, int b, int c,
                                int H, int W, int64_t ignore_label, float eps, float* out, void* stream);

/* ---- a10-a12: prototypes ----------------------------------------------------------------
 * accumulate: feat (b,k,hw) planar, label (b,hw) int64 in {ignore} U [0,c) ->
 *   sums (c,k) fp32 and counts (c) int64 (OVERWRITTEN, deterministic order).  alignment.py:341-348,109-119.
 * accumulate_soft: soft (b,c,H,W) bilinearly down-sampled (align_corners) to (h,w) as weights ->
 *   sums (c,k) (alignment.py:98-104, before the /n mean).
 * finalize: local = sums/(cnt+eps), classes with cnt<1 keep proto_old (counts==NULL: local = sums/mean_n,
 *   the torch.mean of alignment.py:104); proto_new = (1-decay)*local +
 *   decay*proto_old with one_minus_decay/decay pre-rounded to fp32 by the caller (alignment.py:347-353,463-466).
 * ws: uem_proto_accum_ws_bytes(b,c,k). */
UEM_API int64_t uem_proto_accum_ws_bytes(int b, int c, int k);
UEM_API int uem_proto_accum_nchw_f32(const float* feat, int b, int k, int64_t hw, const int64_t* label, int c,
                             int64_t ignore_label, float* sums, int64_t* counts, void* ws, void* stream);
/* sums == counts == NULL: leave the per-image partial sums in ws for uem_proto_fold_finalize_ema_f32, which folds them
 * (image order), applies the keep-old rule and the EMA in one launch (proto_new may alias proto_old). */
UEM_API int uem_proto_fold_finalize_ema_f32(const void* ws, int b, int c, int k, const float* proto_old, float eps,
                                    float one_minus_decay, float decay, float* proto_new, void* stream);
UEM_API int64_t uem_proto_accum_soft_ws_bytes(int b, int c, int k, int h, int w);
UEM_API int uem_proto_accum_soft_f32(const float* feat, int b, int k, int h, int w, const float* soft, int c,
                             int H, int W, float* sums, void* ws, void* stream);
UEM_API int uem_proto_finalize_ema_f32(const float* sums, const int64_t* counts, int64_t mean_n,
                               const float* proto_old, int c, int k, float eps, float one_minus_decay,
                               float decay, float* local_out, float* proto_new, void* stream);

/* ---- a14/a15: histograms ------------------------------------------------------------------
 * class_hist: hist[0..c) = #label==ci, hist[c] = #label!=ignore (balance.py:45-52); hist must be zeroed.
 * class_weight_lookup: out[i] = table[label[i]] or 0 for ignore (balance.py:29-32).
 * hist_f32: torch.histc semantics (balance.py:193): bins over [lo,hi], x==hi in last bin, outside dropped;
 *   hist must be zeroed. */
UEM_API int uem_class_hist_i64(const int64_t* label, int64_t n, int c, int64_t ignore_label, int64_t* hist,
                       void* stream);
UEM_API int uem_class_weight_lookup_f32(const int64_t* label, int64_t n, int c, int64_t ignore_label,
                                const float* table, float* out, void* stream);
UEM_API int uem_hist_f32(const float* x, int64_t n, int bins, float lo, float hi, int64_t* hist, void* stream);
/* torch.bucketize(x, boundaries) (right=False; balance.py:194,263): inds[i] = number of boundaries < x[i]; boundaries
 * (device, ascending, nb <= 1024).  NaN -> nb, like torch. */
UEM_API int uem_bucketize_f32(const float* x, int64_t n, const float* boundaries, int nb, int64_t* inds, void* stream);

/* ---- offline pseudo-label regeneration (next row, SURVEY 8f-1) ------------------------------
 * pseudo_generation.py:150-151, vis_corrected_pseudo_labels.py:191: the map written to disk is
 * uint8(label + 1), i.e. ignore (-1) -> 0, class j -> j+1 (numpy astype semantics: modulo 256). */
UEM_API int uem_label_plus1_u8_i64(const int64_t* label, int64_t n, uint8_t* out, void* stream);

/* ---- PrototypeContrastiveLoss, forward + backward (next row, SURVEY 8f-2) ---------------------
 * uemda/loss.py:10-47 (tools/train_align_uem.py:176-177): loss = mean over non-ignored pixels of
 * CrossEntropy(normalize(f) normalize(P)^T / T, label).  feat (b,k,hw) planar NCHW read in place (hw % 4 == 0,
 * k >= 32), protos (c,k), labels (b,hw) int64.
 * forward : loss[0] (NaN if no pixel is valid, like the reference) and coef (b, c+1, hw): the per-pixel backward
 *           coefficients a_j = (softmax_j - onehot_j) / (Nv T ||f||), beta = sum_j a_j (f.P^_j) / ||f||^2.
 * backward: grad_feat (b,k,hw) = grad_out[0] * (sum_j a_j P^_j[k] - beta f[k]); grad_out: device scalar or NULL (= 1).
 * ws: uem_pcl_ws_bytes(b,k,hw), the same buffer for both calls (it keeps the normalised prototypes). */
UEM_API int64_t uem_pcl_ws_bytes(int b, int k, int64_t hw);
UEM_API int uem_pcl_forward_f32(const float* feat, int b, int k, int64_t hw, const float* protos, int c,
                        const int64_t* labels, int64_t ignore_label, float temperature, float* loss,
                        float* coef, void* ws, void* stream);
UEM_API int uem_pcl_backward_f32(const float* feat, int b, int k, int64_t hw, int c, const float* coef,
                         const float* grad_out, float* grad_feat, const void* ws, void* stream);

/* ---- multi-GPU exchange helpers (SURVEY 8e) -----------------------------------------------------
 * The rank-local statistics of a step travel as one fp64 vector [c*k prototype sums | c counts | max superpixel id]
 * (every part exact in fp64); uem_fold_gathered_f64 folds the all-gathered (world, c*k+c+1) matrix in rank order, so
 * every rank gets bit-identical sums (alignment.py:347-353) and the batch-global max id (alignment.py:241). */
UEM_API int uem_pack_local_f64(const float* sums, const int64_t* counts, const int64_t* max_id, int c, int k, double* out,
                       void* stream);
/* same, straight from the per-image partials uem_proto_accum_nchw_f32 leaves in its ws when sums == NULL (folded in
 * image order with the same fp32 additions as the separate fold) */
UEM_API int uem_pack_local_partials_f64(const void* ws, int b, int c, int k, const int64_t* max_id, double* out, void* stream);
UEM_API int uem_fold_gathered_f64(const double* gathered, int world, int c, int k, float* sums, int64_t* counts,
                          int64_t* max_id, void* stream);

/* ---- f4: IAST class-wise percentile thresholds + sliding-window accumulation (uemda/utils/tools.py) -----------------
 * ias_thresh (:323-333) / generate_pseudo (:347-371): probs (b,c,hw) planar fp32 (the model output the reference calls
 * `logits`).  conf_hist: per class, the EXACT histogram of float16(max prob) over the pixels whose argmax is that class, on
 * the 65536 half bit patterns ordered like the numbers (hist: uem_iast_hist_bytes(c) bytes, zeroed by the call).
 * thresholds: per class np.percentile(linear) of [previous threshold] + samples at qfrac_host[c] = q/100 (host doubles:
 * q = 100*(1 - alpha*w**gamma) is Python arithmetic), written as float32 to tmp_out (optional), then
 * cls_thresh <- beta*cls_thresh + float32(1-beta)*tmp, values >= 1 -> 0.999 (cls_thresh: device double (c), in/out).
 * labels: out (b,hw) uint8 = argmax + 1, or 0 where the winning probability < cls_thresh[argmax].
 * window_accumulate / window_average: pre_slide (:84-97): full[:, :, y1:y2, x1:x2] += tile[:, :, :y2-y1, :x2-x1],
 * count += 1 (count may be NULL), then full /= count.  views_mean: tta_predict's mean over n stacked views (:149-150). */
UEM_API int64_t uem_iast_hist_bytes(int c);
UEM_API int uem_iast_conf_hist_f32(const float* probs, int b, int c, int64_t hw, uint32_t* hist, void* stream);
UEM_API int uem_iast_thresholds_f64(const uint32_t* hist, int c, const double* qfrac_host, double beta, float one_minus_beta,
                            double* cls_thresh, float* tmp_out, int64_t* count_out, void* stream);
UEM_API int uem_iast_labels_u8(const float* probs, int b, int c, int64_t hw, const double* cls_thresh, uint8_t* out,
                       void* stream);
UEM_API int uem_window_accumulate_f32(float* full, float* count, const float* tile, int b, int c, int H, int W, int th, int tw,
                              int y1, int x1, int y2, int x2, void* stream);
UEM_API int uem_window_average_f32(float* full, const float* count, int b, int c, int64_t hw, void* stream);
UEM_API int uem_views_mean_f32(const float* views, int n, int64_t numel, float* out, void* stream);

/* ---- device-side exchange over peer-mapped memory (SURVEY 8e; csrc/uem_exchange.cu) -------------------------------
 * The same statistics as above, but stored by a kernel straight into every peer's symmetric region over NVLink, with
 * release/acquire flags instead of a host-issued collective, so a whole sharded step is capturable as CUDA graphs with no
 * NCCL call between them.  Per-rank vector: [c*k prototype sums f32 | c counts i64 | c+1 class histogram i64 (balance.py:
 * 45-52; zeros when hist == NULL) | rank-local max superpixel id i64 (alignment.py:241)].
 * region: uem_xchg_region_bytes(world, depth, c, k) bytes per rank, ZEROED before the first use (then a barrier across
 *   ranks), mapped into every peer (torch symmetric memory or uem_peer_*); peer_regions: HOST array of `world` device
 *   pointers, entry r = rank r's region as mapped in THIS process (entry `rank` = the local region).
 * depth <= 4 slots are used round-robin by the caller (slot = step % depth); world <= 16.
 * send: folds the per-image partials uem_proto_accum_nchw_f32 left in partials_ws (sums == NULL form) in image order and
 *   stores the vector into slot [slot][rank] of every peer; waits (bounded) for the peers' acknowledgement of the
 *   previous use of that slot first.  global_id_out (optional): the same launch then also polls the other ranks' max ids of
 *   this step and writes the batch-global max id there (what wait_maxid would return), saving that launch.
 *   parts: bit 0 = sums + counts + histogram, bit 1 = max id, bit 2 = this is the step's last send into the slot (advances
 *   the sequence number); 7 = everything in one launch.  A step may send the id early (parts = 2, partials_ws NULL: the id
 *   is known after the region pass) and the sums later (parts = 5): every word carries the step's sequence number itself.
 * wait_maxid: blocks the stream (bounded spin in a one-warp kernel) until every rank's vector of this slot has arrived;
 *   writes the batch-global max id.  fold_finalize_ema: (after wait_maxid on the same stream) folds the ranks in rank
 *   order -> keep-old rule -> EMA (alignment.py:347-353,463-466; proto_new may alias proto_old; NULL = no EMA), optional
 *   folded sums (c,k) / counts (c) / histogram (c+1) outputs; acknowledges the slot to every peer.
 * Every payload word travels as one 8-byte {word, sequence number} store (no fences or flags on the data path); the
 * consumers poll the words they read.
 * uem_xchg_status: synchronises the stream and returns the region's status word: bit 8 = a poll timed out (2 s: a peer
 *   is gone, or the calls are not issued in lockstep on every rank). */
UEM_API int64_t uem_xchg_region_bytes(int world, int depth, int c, int k);
UEM_API int uem_xchg_send_f32(const void* partials_ws, int b, int c, int k, const int64_t* max_id, const int64_t* hist,
                      const void* const* peer_regions, int rank, int world, int depth, int slot, int64_t* global_id_out,
                      int parts, void* stream);
UEM_API int uem_xchg_wait_maxid(void* region, int world, int depth, int slot, int c, int k, int64_t* max_id_out, void* stream);
UEM_API int uem_xchg_fold_finalize_ema_f32(const void* const* peer_regions, int rank, int world, int depth, int slot, int c,
                                   int k, const float* proto_old, float eps, float one_minus_decay, float decay,
                                   float* proto_new, float* sums_out, int64_t* counts_out, int64_t* hist_out, void* stream);
/* send (sums part) + fold_finalize_ema in ONE launch: every thread carries its element of the (c,k) bank from this rank's
 * per-image partials through the LL stores into every rank's slot, the poll of every rank's words and the rank-ordered
 * fold to the EMA-updated prototype (the max id of the step has been sent before with parts = 2).  Not for emulated ranks
 * on one device: every rank's launch must be able to run while the others' are running. */
UEM_API int uem_xchg_exchange_fold_ema_f32(const void* partials_ws, int b, int c, int k, const int64_t* hist,
                                   const void* const* peer_regions, int rank, int world, int depth, int slot,
                                   const float* proto_old, float eps, float one_minus_decay, float decay, float* proto_new,
                                   float* sums_out, int64_t* counts_out, int64_t* hist_out, void* stream);
UEM_API int uem_xchg_status(const void* region, int* status_out, void* stream);
/* cudaIpc plumbing for the region when torch symmetric memory is unavailable: alloc (cudaMalloc + zero) returns the local
 * pointer and a 64-byte handle to ship to the peers (any host channel), open maps a peer's handle. */
UEM_API int uem_peer_alloc(int64_t bytes, void** ptr, void* handle64);
UEM_API int uem_peer_open(const void* handle64, void** ptr);
UEM_API int uem_peer_close(void* ptr);
UEM_API int uem_peer_free(void* ptr);

/* ---- UVEM / UPS target loss fused end to end, forward + backward (next row, SURVEY 8f-3) ----------
 * uemda/gast/balance.py:437-457 (loss_calc_uvem: every head's logits up-sampled bilinearly, align_corners=True, to the
 * label size; loss averaged over heads), :356-394 (UVEMLoss.forward), :321-342 (UPSLoss.forward).
 * x1 [, x2] (b,c,h,w) low-resolution logits of the heads (x2 may be NULL), target (b,H,W) int64, coef (b*H*W) fp32: the
 * detached per-pixel factor weight x gate x class weight (0 for ignored / gated pixels; from uem_uvem_terms_f32).
 * forward : sums[m] += sum_px coef * CrossEntropy(upsample(x_m))[px, target]   (fp64, zeroed by the caller); the loss
 *           is (sums[0] [+ sums[1]]) / (valid + 1e-7) / heads.
 * backward: g_m (b,c,h,w) = scale[0] * d sums[m] / d x_m, every element written, deterministic (a gather per low-res
 *           cell, no atomics); scale: device scalar = grad_out / (valid + 1e-7) / heads.  ws (required, not NULL):
 *           uem_uvem_loss_backward_ws_bytes bytes of scratch for the per-block partials (every pixel's softmax is evaluated
 *           once, then a fixed-order gather per cell). */
UEM_API int uem_uvem_loss_forward_f32(const float* x1, const float* x2, int b, int c, int h, int w, int H, int W,
                              const int64_t* target, const float* coef, double* sums, void* stream);
UEM_API int64_t uem_uvem_loss_backward_ws_bytes(int b, int c, int h, int w, int heads);
UEM_API int uem_uvem_loss_backward_f32(const float* x1, const float* x2, int b, int c, int h, int w, int H, int W,
                               const int64_t* target, const float* coef, const float* scale, float* g1, float* g2,
                               void* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UEM_B200_H */
