/* cia.h -- C-ABI of libcia.so, the sm_100a implementation of the per-cell
 * screening hot path of Kmatsuo57/cell-image-analysis.
 *
 * The reference has no FFI: its seams are the Python methods
 *   ProductionMutantScreening.extract_quality_cells   improved_detection.py:48-115
 *   ProductionMutantScreening.compute_anomaly_scores  improved_detection.py:117-153
 * (training twins CAE_improved_modeltrain.py:39-111, 328-339, 398-402).  Each entry
 * point below names the reference lines it replaces.  INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative CIA_E_* code on failure and
 *     never throws or prints; cia_last_error() gives the message for the handle;
 *   - image / label / crop / score buffers are raw DEVICE pointers unless the name
 *     ends in _host; artifact tensors passed to cia_load_* are HOST pointers and
 *     are copied -- the library keeps no reference to caller memory;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work unless
 *     stated otherwise ("synchronises");
 *   - counts that are data dependent live in device memory (`*_dev`); a host
 *     capacity bounds every output buffer and overflow is reported through
 *     cia_check_status(), never by writing out of bounds.
 */
#ifndef CIA_H
#define CIA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CIA_OK            0
#define CIA_E_CUDA       -1   /* a CUDA runtime call failed                         */
#define CIA_E_ARG        -2   /* bad argument                                       */
#define CIA_E_STATE      -3   /* artifacts not loaded / wrong topology              */
#define CIA_E_CAPACITY   -4   /* an output capacity was exceeded on the device      */
#define CIA_E_LABEL      -5   /* a label outside [0, max_label] was seen            */
#define CIA_E_UNSUPPORTED -6  /* bbox too large for the crop kernel's scratch, etc. */

#define CIA_CROP 64                 /* det:99  resize target                         */
#define CIA_FEATURES 2048           /* 8*8*32, det:131 HWC flatten                   */

typedef struct cia_ctx* cia_handle;

/* One labelled region, as skimage.measure.regionprops exposes it (det:67, 73, 80):
 * half-open bbox and pixel count, plus the exact integer raw moments (image
 * coordinates) the eccentricity of det:84 is derived from.  A zeroed record is an
 * absent label.  Slot i of a field's table is label i+1. */
typedef struct cia_region {
    uint32_t area;                  /* prop.area                                     */
    int32_t  minr, minc, maxr, maxc;/* prop.bbox (half open)                         */
    int32_t  flags;                 /* bit0: passed all gates of det:76-95           */
    uint64_t m10, m01, m20, m02, m11; /* sum r, sum c, sum r^2, sum c^2, sum r*c     */
} cia_region;                        /* 64 bytes                                      */

/* One cell that passed the gates, in reference order: fields in call order, labels
 * ascending (det:72).  The stats are the cell_stats dict of det:103-109; its solidity entry
 * comes from cia_solidity (it needs the label field, which the fused path does not keep). */
typedef struct cia_cell {
    int32_t field;                  /* index of the field inside the call            */
    int32_t label;
    int32_t minr, minc, maxr, maxc;
    int32_t area;
    int32_t pad_;
    double  eccentricity;
    double  mean_intensity;
    double  std_intensity;
} cia_cell;                          /* 56 bytes                                      */

/* Literals of det:76-99 / train:66-93 (defaults via cia_default_params). */
typedef struct cia_params {
    int32_t border_margin;          /* 10                                            */
    int32_t area_min, area_max;     /* 200, 8000                                     */
    double  ecc_max;                /* 0.95                                          */
    double  mean_min, std_min;      /* 0.5, 0.1                                      */
    double  clip_limit;             /* 0.02                                          */
    double  intensity_inv;          /* 1/65535: img_as_float's factor inside equalize_adapthist
                                     * (det:98) for 16-bit fields; 1/255 when an 8-bit field was
                                     * widened to uint16 by the caller                              */
} cia_params;

/* Per-cell scores, the arrays of the dict at det:144-153 (signs as libsvm returns
 * them: decision > 0 <=> inlier; the Python layer negates like det:149-150). */
typedef struct cia_scores {
    float*  mse;                    /* [n]  det:126                                  */
    float*  mae;                    /* [n]  det:127                                  */
    double* dec_conservative;       /* [n]  det:141                                  */
    double* dec_moderate;           /* [n]  det:142                                  */
    int8_t* pred_conservative;      /* [n]  det:138  (+1 / -1)                       */
    int8_t* pred_moderate;          /* [n]  det:139                                  */
} cia_scores;

/* ---- lifecycle ---------------------------------------------------------- */
int  cia_version(void);
int  cia_create(int device, cia_handle* out);
int  cia_destroy(cia_handle h);
const char* cia_last_error(cia_handle h);
void cia_default_params(cia_params* p);
/* Reads back the device status word (synchronises `stream`): 0 or a CIA_E_* code
 * raised by a kernel since the last check (capacity / label / unsupported: a crop kernel bbox too large,
 * or a tensor-core autoencoder activation outside the fp16 range). */
int  cia_check_status(cia_handle h, void* stream);
/* Tuning knobs of the handle (no reference counterpart; defaults reproduce the documented
 * behaviour).  Unknown names / out-of-range values give CIA_E_ARG.
 *   "cae_pass_cells"  cells per pass of the tensor-core autoencoder over its seven layers
 *                     (default 18944 = 128 per SM; 303 KB of fp16 activations per cell);
 *                     results do not depend on it (tests/test_gpu_multipass.py)
 *   "cae_l1_debias", "cae_l2_debias", "cae_l3_debias"
 *                     compensation of tcgen05's round-toward-zero accumulation in the
 *                     split-precision encoder layers, in units of 2^-24 relative
 *                     (defaults 0.5 / 2.4 / 1.2, 0 = off; DESIGN.md section 5)
 *   "svm_kernel"      1 (default): tcgen05 GEMM-form RBF decision (csrc/score_tc.cu; |d dec| <= ~2e-5 vs
 *                     libsvm at 20 000 SVs, DESIGN.md section 4.1); 0: the fp64 DMMA kernel (equal to
 *                     libsvm to 1e-9).  Models the tensor-core kernel does not serve (more than 256
 *                     dimensions, negative dual coefficients) take the fp64 kernel by themselves.
 *   "pca_kernel"      1 (default): tcgen05 RobustScaler + PCA projection; 0: the fp64 DMMA kernel
 *   "svm_refine"      1 (default): decisions within the tensor-core kernel's error of zero are
 *                     recomputed in fp64 (sign rule svm.cpp:2841 evaluated on exact values); 0: off
 *   "seg_conv_tma"    segmentation (csrc/segment.cu): 1 (default) the Cin = 32 direct layers and the heads run the
 *                     TMA-fed warp-specialised kernels; 0: the staged kernel everywhere (same arithmetic)
 *   "seg_conv_ws"     1 (default): the software-producer warp-specialised kernel for the layers where it measured
 *                     faster; 2: for every layer the TMA kernel does not take; 0: off
 *   "seg_pool_out"    1 (default): a TMA-fed layer whose output the next layer max-pools writes the pooled copy itself
 *                     (and only that, where nothing else reads the full-resolution map); 0: the consumer pools (bit-identical)
 * A `precision` 0 call (cia_screen_fields*, cia_cae_forward) is the exact anchor end to end and uses the
 * fp64 scoring kernels whatever these options say. */
int  cia_set_option(cia_handle h, const char* name, double value);

/* ---- artifacts (replaces load_trained_models, det:23-41) ----------------- */
/* which = 0: best_autoencoder.keras (7 Conv2D, 6 BatchNormalization);
 * which = 1: encoder.keras (3 + 3) when its weights differ from the autoencoder's
 *            encoder half (det:29-30, 130); never loading it makes the feature tap of
 *            the autoencoder pass serve det:130.
 * kernels[i]: float32 HWIO (3,3,Cin,Cout) as Keras stores them; bn[4*i+{0,1,2,3}] =
 * gamma, beta, moving_mean, moving_variance of BatchNormalization i. */
int cia_load_cae(cia_handle h, int which, int n_conv,
                 const float* const* kernels, const float* const* biases,
                 const float* const* bn, float bn_eps);
/* RobustScaler (det:134) + PCA (det:135).  All vectors as float64; f32_flow=1 mirrors
 * scikit-learn's dtype flow for float32-fitted artifacts (every intermediate rounded
 * to float32), 0 the float64-components flow.  pca_offset = mean_ @ components_.T
 * evaluated by the caller exactly as sklearn does. */
int cia_load_scaler_pca(cia_handle h, int n_features, int n_components,
                        const double* center /* or NULL */, const double* scale /* or NULL */,
                        int center_is_f32, const double* components /* [C,F] */,
                        const double* pca_offset /* [C] */, int f32_flow);
/* OneClassSVM, RBF kernel (det:138-142).  which: 0 conservative, 1 moderate.
 * rho = -intercept_[0]. */
int cia_load_svm(cia_handle h, int which, int n_sv, int dim,
                 const double* support_vectors /* [n_sv, dim] */,
                 const double* dual_coef /* [n_sv] */, double gamma, double rho);

/* ---- stage entry points -------------------------------------------------- */
/* regionprops bbox/area/moments (det:67).  labels: int32 [n_fields, H, W];
 * regions: [n_fields, max_label], zeroed by the call. */
int cia_label_scan(cia_handle h, const int32_t* labels, int n_fields, int H, int W,
                   int max_label, cia_region* regions, void* stream);
/* Quality gates of det:76-95 and compaction in reference order.
 * images: uint16 [n_fields, H, W].  cells: capacity cells_cap; n_cells_dev: int32
 * total; field_counts_dev: int32 [n_fields] or NULL. */
int cia_filter(cia_handle h, const uint16_t* images, int n_fields, int H, int W,
               int max_label, cia_region* regions, const cia_params* params,
               cia_cell* cells, int cells_cap, int32_t* n_cells_dev,
               int32_t* field_counts_dev, void* stream);
/* prop.solidity of det:106 / train:101 for the cells that passed the gates: area over the pixel count
 * of skimage's convex_hull_image of the region mask (edge-midpoint offsets, border included).
 * labels: int32 [n_fields, H, W] as given to cia_label_scan; solidity: float64 [n_cells]. */
int cia_solidity(cia_handle h, const int32_t* labels, int H, int W, const cia_cell* cells,
                 int n_cells, const int32_t* n_cells_dev, double* solidity, void* stream);
/* det:88 crop + det:98 equalize_adapthist + det:99 resize + det:122 float32 cast.
 * n_cells: host upper bound; n_cells_dev (may be NULL) the device count.
 * crops32: float32 [n,64,64]; crops64 (may be NULL): float64 [n,64,64]. */
int cia_crop_resize(cia_handle h, const uint16_t* images, int H, int W,
                    const cia_cell* cells, int n_cells, const int32_t* n_cells_dev,
                    const cia_params* params, float* crops32, double* crops64,
                    void* stream);
/* Test tap: same as cia_crop_resize, additionally writing the uint16 CLAHE levels (the
 * bit-exact integer core of det:98, before the final [0,1] rescale) of cell i as h*w
 * values at levels_out + level_offsets[i] (device pointers). */
int cia_debug_clahe_levels(cia_handle h, const uint16_t* images, int H, int W,
                           const cia_cell* cells, int n_cells, const cia_params* params,
                           float* crops32, uint16_t* levels_out,
                           const int64_t* level_offsets, void* stream);
/* autoencoder.predict + MSE/MAE (det:125-127) and encoder.predict + flatten
 * (det:130-131).  features (may be NULL): float32 [n, 2048] HWC order.
 * precision: 0 = fp32 CUDA-core path, 1 = tcgen05 tensor-core path (split-precision encoder, features
 * from it), 2 = tensor-core autoencoder for MSE/MAE with the fp32 encoder for the features, 3 = as 1 with
 * the third encoder layer in exact fp32 (an A/B mode).
 * Precisions 1-3 store every activation as fp16.  An activation outside the fp16 range (|x| > 65504, e.g.
 * a BatchNorm with a large gamma over a small moving variance) or a NaN raises CIA_E_UNSUPPORTED on the
 * status word (cia_check_status); the scores of that call are then not valid.  Precision 0 has no such
 * limit.  n_cells_dev (may be NULL): device int32 count <= n_cells; cells from it on get mse = mae = 0. */
int cia_cae_forward(cia_handle h, const float* crops32, int n_cells,
                    const int32_t* n_cells_dev, float* mse, float* mae,
                    float* features, int precision, void* stream);
/* scaler.transform -> pca.transform -> both detectors' decision_function / predict
 * (det:134-142).  pca_out (may be NULL): float64 [n, n_components]. */
int cia_svm_decision(cia_handle h, const float* features, int n_cells,
                     const int32_t* n_cells_dev, double* dec_cons, double* dec_mod,
                     int8_t* pred_cons, int8_t* pred_mod, double* pca_out, void* stream);
/* Per-strain accumulators behind det:151-152, 202-211: acc[s] = {n, n_cons_anom,
 * n_mod_anom, sum mse, sum mse^2, sum mae, sum mae^2, 0} (float64 [S,8], added to).
 * field_strain: int32 [n_fields] strain id of each field of the call. */
int cia_strain_accumulate(cia_handle h, const cia_cell* cells, int n_cells,
                          const int32_t* n_cells_dev, const cia_scores* scores,
                          const int32_t* field_strain, double* acc, int n_strains,
                          void* stream);

/* ---- fits of create_anomaly_detector (CAE_improved_modeltrain.py:404-423) ---- */
/* RobustScaler().fit(features) (train:408): center_ = np.nanmedian(X, axis=0) (float32 [F]) and
 * scale_ = q75 - q25 of np.nanpercentile(X, (25, 75)) (float64 [F]) with _handle_zeros_in_scale, from exact
 * column sorts and numpy's "linear" interpolation.  features: float32 [n, F].  scaled (may be NULL): float32 [n, F],
 * RobustScaler.transform of the same rows (train:408 fit_transform).  NaN is not supported: a NaN in features is
 * reported as CIA_E_ARG by cia_check_status (np.nanmedian would skip it; the encoder never produces one). */
int cia_fit_robust_scaler(cia_handle h, const float* features, int n, int n_features, float* center, double* scale,
                          float* scaled, void* stream);
/* The covariance PCA(n_components).fit diagonalises (train:412-414; sklearn's covariance_eigh, in fp64):
 * mean float64 [F] of x float32 [n, F] and cov float64 [F, F] = X_c^T X_c / (n - 1), X_c = x - mean.  n >= 2. */
int cia_fit_pca_gram(cia_handle h, const float* x, int n, int n_features, double* mean, double* cov, void* stream);
/* OneClassSVM(kernel="rbf", nu, gamma, tol, max_iter).fit(x) (train:420-423): libsvm's solve_one_class and
 * Solver::Solve (svm.cpp) iteration for iteration, without shrinking, in one cooperative kernel.  x: float64
 * [l, dim], dim <= 512 (CIA_E_UNSUPPORTED above); gamma the numeric value (sklearn's _gamma); max_iter -1 = none.
 * alpha: float64 [l] the dual solution (support vectors: alpha != 0); result: float64 [4] = rho, obj, n_iter,
 * status (1 when max_iter stopped the solver).  No host synchronisation. */
int cia_ocsvm_fit(cia_handle h, const double* x, int l, int dim, double nu, double gamma, double tol, int max_iter,
                  double* alpha, double* result, void* stream);

/* ---- fused path ----------------------------------------------------------- */
/* The whole hot path for a batch of device-resident fields, with no host
 * synchronisation: scan -> gates -> crop/CLAHE/resize -> CAE -> scaler/PCA/SVM ->
 * strain accumulate.  Optional outputs may be NULL (crops32, features, acc). */
int cia_screen_fields(cia_handle h, const uint16_t* images, const int32_t* labels,
                      int n_fields, int H, int W, int max_label,
                      const cia_params* params, int precision,
                      cia_cell* cells, int cells_cap, int32_t* n_cells_dev,
                      int32_t* field_counts_dev, const cia_scores* scores,
                      float* crops32, float* features,
                      const int32_t* field_strain, double* acc, int n_strains,
                      void* stream);
/* Same, from HOST buffers (pinned or pageable): copies the fields in, runs the
 * path, copies cells + scores out and synchronises.  All outputs are host
 * pointers; returns the number of cells through *n_cells_host. */
int cia_screen_fields_host(cia_handle h, const uint16_t* images_host,
                           const int32_t* labels_host, int n_fields, int H, int W,
                           int max_label, const cia_params* params, int precision,
                           cia_cell* cells_host, int cells_cap, int32_t* n_cells_host,
                           int32_t* field_counts_host, const cia_scores* scores_host,
                           void* stream);

/* Run-length transport of label fields (host -> device).  The int32 label image the
 * reference passes to regionprops (improved_detection.py:66-70) is 16.8 MB per 2048 x 2048
 * field and its PCIe copy, not a kernel, bounds the end-to-end rate; label images are
 * piecewise constant along rows, so the host encodes runs, only those cross the bus, and
 * cia_rle_expand rebuilds the dense field in HBM bit for bit.
 *   cia_rle_slot_words   words per field slot that always suffice for <= 1 run per 8 pixels
 *   cia_rle_encode_fields host-only (no handle, no GPU): encodes n_fields fields with
 *                        n_threads host threads (<= 0: CIA_HOST_THREADS or all cores) into
 *                        slots_host + f * slot_words; field_words[f] = words used;
 *                        *max_label = largest label seen (may be NULL).  CIA_E_CAPACITY if a
 *                        field does not fit its slot (send that batch as raw int32 instead).
 *   cia_rle_upload       one async copy per field of exactly the words used
 *   cia_rle_expand       device slots -> dense int32 labels [n_fields, H, W]
 *   cia_label_scan_rle   cia_label_scan computed from the runs themselves: bbox / area / raw
 *                        moments are sums over pixels with closed forms over a run, so the
 *                        region table (bit-identical to cia_label_scan of the expanded field)
 *                        needs neither the dense field in HBM nor its 4 B/pixel read
 *   cia_screen_fields_rle cia_screen_fields with the label fields given as device slots */
size_t cia_rle_slot_words(int H, int W);
int cia_rle_encode_fields(const int32_t* labels_host, int n_fields, int H, int W,
                          uint32_t* slots_host, size_t slot_words, uint32_t* field_words,
                          int32_t* max_label, int n_threads);
/* Host-only probe: streaming-read bandwidth (GB/s) of `bytes` at `buf` with n_threads threads
 * (<= 0: CIA_HOST_THREADS or all cores), `reps` passes -- the memory side of cia_rle_encode_fields. */
double cia_host_read_probe(const void* buf, size_t bytes, int n_threads, int reps);
int cia_rle_upload(cia_handle h, const uint32_t* slots_host, int n_fields, size_t slot_words,
                   const uint32_t* field_words, uint32_t* slots_dev, void* stream);
int cia_rle_expand(cia_handle h, const uint32_t* slots_dev, int n_fields, size_t slot_words,
                   int H, int W, int32_t* labels_dev, void* stream);
/* ---- patch transport of the image (no reference counterpart: the implicit hand-over of `green_channel`,
 * det:57-59, to the crop of det:88) ----
 * The device reads the image only inside the bounding boxes of labelled regions, so only those rectangles
 * cross PCIe (~1.2 of 8.4 MB per 2048^2 field with ~500 cells):
 *   cia_rle_encode_pack_fields  cia_rle_encode_fields, and the thread that encoded a field also packs the bbox
 *                        rectangles of its labels 1..label_cap (label ascending, rows contiguous) into
 *                        patches_host[f * patch_cap_px ..]; patch_px[f] = pixels used, 0xFFFFFFFF if they do
 *                        not fit (copy that chunk's images densely instead)
 *   cia_patch_upload     one async copy per field of exactly the pixels used
 *   cia_screen_fields_rle_patches  cia_screen_fields_rle whose `images` is a dense [n_fields, H, W] device
 *                        SCRATCH buffer: after the region scan the rectangles are written to their bbox
 *                        positions (pixels outside every bbox stay undefined; the path never reads them) */
int cia_rle_encode_pack_fields(const int32_t* labels_host, const uint16_t* images_host, int n_fields, int H, int W,
                               uint32_t* slots_host, size_t slot_words, uint32_t* field_words, int32_t* max_label,
                               int label_cap, uint16_t* patches_host, size_t patch_cap_px, uint32_t* patch_px,
                               int n_threads);
int cia_patch_upload(cia_handle h, const uint16_t* patches_host, int n_fields, size_t patch_cap_px,
                     const uint32_t* patch_px, uint16_t* patches_dev, void* stream);
int cia_screen_fields_rle_patches(cia_handle h, uint16_t* images, const uint16_t* patches, size_t patch_cap_px,
                                  const uint32_t* rle_slots, size_t slot_words, int n_fields, int H, int W,
                                  int max_label, const cia_params* params, int precision, cia_cell* cells,
                                  int cells_cap, int32_t* n_cells_dev, int32_t* field_counts_dev,
                                  const cia_scores* scores, float* crops32, float* features,
                                  const int32_t* field_strain, double* acc, int n_strains, void* stream);
int cia_label_scan_rle(cia_handle h, const uint32_t* rle_slots, size_t slot_words, int n_fields,
                       int H, int W, int max_label, cia_region* regions, void* stream);
int cia_screen_fields_rle(cia_handle h, const uint16_t* images, const uint32_t* rle_slots,
                          size_t slot_words, int n_fields, int H, int W, int max_label,
                          const cia_params* params, int precision,
                          cia_cell* cells, int cells_cap, int32_t* n_cells_dev,
                          int32_t* field_counts_dev, const cia_scores* scores,
                          float* crops32, float* features,
                          const int32_t* field_strain, double* acc, int n_strains,
                          void* stream);

/* Host-only strip / tile decompressors of the TIFF reader that stands in for tiff.imread
 * (improved_detection.py:51; SURVEY 8f row N1): TIFF-LZW, PackBits and Zstandard (RFC 8878 frames, the
 * decoder cia_tiff_decode_fields runs; dictionaries are refused, content sizes and checksums are verified; a few
 * non-conforming streams libzstd accepts are refused, see csrc/tiff_decode.h).  Return the bytes written to dst
 * (at most cap) or -1 on a corrupt stream. */
long long cia_tiff_lzw_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap);
long long cia_tiff_packbits_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap);
long long cia_tiff_zstd_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap);

/* One compressed strip or tile of a field (tiff_min.page_layout parses it from the file's directory). */
typedef struct cia_tiff_segment {
    uint64_t src_off, src_len;      /* its compressed bytes: src[src_off, src_off + src_len)             */
    uint64_t dst_off;               /* decoded into scratch[dst_off, dst_off + rows * cols * samples * bytes) */
    int32_t  field;                 /* [0, n_fields)                                                     */
    int32_t  compression;           /* 1, 5 (LZW), 8 or 32946 (Deflate), 32773 (PackBits), 50000 or 34926 (Zstandard) */
    int32_t  predictor;             /* 1, or 2 (horizontal differencing, per sample, wrapping)           */
    int32_t  bytes_per_sample;      /* 1 (widened to uint16) or 2                                        */
    int32_t  big_endian;            /* 16-bit samples are stored big endian                              */
    int32_t  samples;               /* interleaved samples per pixel in the segment (planar files: 1)    */
    int32_t  y0, x0, rows, cols;    /* its rectangle in the field; pixels past H / W (tile edges) are dropped */
    int32_t  seg_sample, img_sample;/* sample written to seg_out / img_out, -1: none                     */
} cia_tiff_segment;                  /* 72 bytes                                                          */

/* Decodes the strips / tiles of n_fields TIFF fields in one launch (one warp per segment, csrc/tiff_dev.cu) into
 * uint16 [n_fields][H][W] planes: seg_out (may be NULL) takes the segmentation channel, img_out the analysis
 * channel of cia_screen_images (det:54-59).  src, segs, scratch, the planes and field_status are DEVICE pointers.
 * field_status int32 [n_fields] is zeroed, then bit 0 marks a corrupt stream, bit 1 a segment that decoded short
 * and bit 2 a descriptor outside src / scratch, with rows or cols outside [1, 2^20], samples outside [1, 16] or
 * another field outside its range; a field with a nonzero status is unusable and the other fields are unaffected.
 * A descriptor whose `field` is outside [0, n_fields) is skipped: there is no field to flag, so the caller must
 * give every field its segments (tiff_device.pack_fields does).  Reads stay inside each segment's bytes, writes inside its rectangle of its own
 * field.  Deflate streams are accepted and refused exactly as Python's zlib.decompress does; Zstandard streams
 * exactly as cia_tiff_zstd_decode does. */
int cia_tiff_decode_fields(cia_handle h, const uint8_t* src, size_t src_bytes, const cia_tiff_segment* segs,
                           int n_segs, int n_fields, int H, int W, uint8_t* scratch, size_t scratch_bytes,
                           uint16_t* seg_out, uint16_t* img_out, int32_t* field_status, void* stream);

/* Stage timing of the fused path with CUDA events recorded in-stream (no host sync is
 * added to the timed region): after cia_profile_begin(h, R) the next R calls of
 * cia_screen_fields bracket scan / gates / crop / CAE / SVM / accumulate with events;
 * cia_profile_end sums the elapsed milliseconds per stage over the recorded calls
 * (synchronises on the last event of each). */
int cia_profile_begin(cia_handle h, int max_records);
int cia_profile_end(cia_handle h, double* stage_ms /* [6] */, int* n_records);
/* Per-layer split of the CAE stage of the same recorded calls (tensor-core precisions; up to 8
 * passes of each call): elapsed milliseconds of the seven conv layers L1..L7, summed over the
 * records.  Call it BEFORE cia_profile_end (which closes the recording). */
int cia_profile_layers(cia_handle h, double* layer_ms /* [7] */);

/* Test tap: copy `bytes` at `offset` of internal workspace `ws_id` to host (synchronises).
 * ws_id 5 holds the tensor-core path's fp16 activations (layout in cae_tc.cu). */
int cia_debug_copy_workspace(cia_handle h, int ws_id, size_t offset, void* dst_host, size_t bytes);

/* ---------------------------------------------------------------------------------------------
 * Segmentation (SURVEY 8f row N2): the producer of the int32 label field.  Replaces
 *   normalized_seg = normalize(seg_channel)                              improved_detection.py:62
 *   labels, details = self.stardist_model.predict_instances(normalized_seg)   improved_detection.py:63
 * (model construction improved_detection.py:44; the training twin CAE_improved_modeltrain.py:54-55).
 * csbdeep / stardist are third-party packages absent from the reference tree; oracle/stardist.py and
 * oracle/stardist_post.c restate them ("parity unpinned").  All image / map pointers are DEVICE
 * pointers; weights, ray tables and the config are host pointers read during the call.
 * ------------------------------------------------------------------------------------------- */
typedef struct cia_seg_config {   /* the fields of a StarDist2D config.json the network depends on */
    int32_t n_channel_in;          /* 1 */
    int32_t grid;                  /* 1, 2 or 4 (square grids) */
    int32_t n_rays;                /* 32 */
    int32_t unet_n_depth;
    int32_t unet_n_filter_base;    /* multiple of 32 */
    int32_t unet_n_conv_per_depth;
    int32_t net_conv_after_unet;   /* channels of the `features` layer, multiple of 32 */
    int32_t reserved;
} cia_seg_config;

/* StarDist2D.__init__ / _build (improved_detection.py:44): upload the 3x3 convolutions of the network in the
 * order the model applies them (grid blocks, down levels, middle, up levels, `features`), then the 1x1 heads
 * `prob` and `dist`: kernels[l] is HWIO float32 with shapes[4*l..4*l+3] = {kh, kw, cin, cout}.  ray_sin / ray_cos:
 * float64 [n_rays] = sin / cos of np.linspace(0, 2 pi, n_rays, endpoint=False) (stardist ray_angles), passed in so
 * that the polygon vertices equal the host library's bit for bit.  CIA_E_UNSUPPORTED / CIA_E_ARG (with
 * cia_last_error) when the layers do not fit the configuration. */
int cia_seg_load(cia_handle h, const cia_seg_config* cfg, int n_layers, const float* const* kernels,
                 const float* const* biases, const int64_t* shapes, const double* ray_sin, const double* ray_cos);
/* csbdeep.utils.normalize(x, pmin, pmax) of a uint16 field (improved_detection.py:62; defaults 3 / 99.8):
 * np.percentile's linear interpolation from the exact histogram, then (x - mi) / (ma - mi + 1e-20) in float32.
 * out: float32 [H][W]; mi_ma (may be NULL): float32 [2] on the device. */
int cia_seg_normalize(cia_handle h, const uint16_t* image, int H, int W, double pmin, double pmax, float* out,
                      float* mi_ma, void* stream);
/* The network of predict_instances (improved_detection.py:63): normalized float32 field [H][W] -> prob
 * float32 [H/grid][W/grid] and dist float32 [H/grid][W/grid][n_rays] (dist = max(1e-3, dist) as StarDist2D.predict).
 * prob / dist may be NULL: the maps stay inside the handle for cia_seg_instances.  H, W must be multiples of
 * grid * 2^depth (StarDist reflect-pads other sizes: CIA_E_UNSUPPORTED here). */
int cia_seg_predict(cia_handle h, const float* image, int H, int W, float* prob, float* dist, void* stream);
/* _instances_from_prediction: candidates prob > prob_thresh outside the 2-pixel border, sorted by
 * probability, greedy polygon NMS (intersection / smaller area > nms_thresh suppresses), polygons_to_label.
 * prob / dist NULL = the maps of the last cia_seg_predict.  labels: int32 [H][W]; n_instances (may be NULL): device int32. */
int cia_seg_instances(cia_handle h, const float* prob, const float* dist, int Hg, int Wg, int grid, int H, int W,
                      double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_instances, void* stream);
/* `details` of the last cia_seg_instances for the first `cap` kept polygons, in label order:
 * points int32 [cap][2] (y, x), prob float32 [cap], coord float32 [cap][2][n_rays]. */
int cia_seg_details(cia_handle h, int cap, int32_t* points, float* prob, float* coord, void* stream);
/* ---- F equally sized fields per call (the calls above are the F = 1 case of the same kernels) ----
 * Every stage runs all F fields in one launch sequence: the number of launches does not depend on F, and per
 * field the arithmetic (and its order) is that of the one-field call, so the outputs equal it bit for bit.
 * Fields of different sizes go to separate calls.  Device memory held by the handle per field (grow-only):
 *   normalisation   4.2 MB (per-field histograms; its own workspace, not shared with the screen)
 *   U-Net           sum over the plan's buffers of C * (Hp/2^s) * (Wp/2^s) * 2 bytes + prob / dist maps:
 *                   1.4 GB for a 2048 x 2048 field with 2D_versatile_fluo
 *   instances       352 bytes per map pixel of Hp/grid x Wp/grid (0.37 GB for a 2048 x 2048 field, grid 2)
 *   cia_screen_images  additionally Hp * Wp * 4 (normalized field) and, when labels_out is NULL, H * W * 4
 *
 * cia_seg_normalize_fields  csbdeep normalize of each field by ITS OWN percentiles (images uint16 [F][H][W]),
 *                    written reflect-padded to out float32 [F][Hp][Wp], Hp / Wp the next multiples of
 *                    grid * 2^depth of the loaded model (np.pad(mode='reflect') of the normalized field, what
 *                    StarDist pads with).  CIA_E_STATE without a loaded model.
 * cia_seg_predict_fields   the network on images float32 [F][Hp][Wp] (Hp, Wp multiples of grid * 2^depth):
 *                    prob float32 [F][Hp/g][Wp/g], dist float32 [F][Hp/g][Wp/g][n_rays]; either may be NULL (the
 *                    maps stay in the handle for cia_seg_instances_fields).
 * cia_seg_instances_fields _instances_from_prediction per field on maps [F][Hgp][Wgp] (padded: candidates only
 *                    inside each field's ceil(H/grid) x ceil(W/grid) part, the 2-pixel border measured from
 *                    that edge); prob / dist NULL = the maps of the last predict call.  labels int32 [F][H][W]
 *                    numbered per field (1..n_instances[f]); n_instances device int32 [F] (may be NULL).
 * cia_screen_images  det:51-153 for F fields given nothing but images: the three calls above (pmin 3, pmax 99.8)
 *                    on seg_images, then the cia_screen_fields path on `images` with those labels, with no host
 *                    synchronisation.  seg_images may equal images (single-channel fields, det:57-59).
 *                    max_label bounds the instances of one field: a field with more is reported as CIA_E_LABEL by
 *                    cia_check_status, nothing is written out of bounds.  labels_out (may be NULL): int32 [F][H][W]. */
int cia_seg_normalize_fields(cia_handle h, const uint16_t* images, int n_fields, int H, int W, double pmin, double pmax,
                             float* out, void* stream);
int cia_seg_predict_fields(cia_handle h, const float* images, int n_fields, int Hp, int Wp, float* prob, float* dist,
                           void* stream);
int cia_seg_instances_fields(cia_handle h, const float* prob, const float* dist, int n_fields, int Hgp, int Wgp, int grid,
                             int H, int W, double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_instances,
                             void* stream);
int cia_screen_images(cia_handle h, const uint16_t* seg_images, const uint16_t* images, int n_fields, int H, int W,
                      double prob_thresh, double nms_thresh, int max_label, const cia_params* params, int precision,
                      cia_cell* cells, int cells_cap, int32_t* n_cells_dev, int32_t* field_counts_dev,
                      const cia_scores* scores, float* crops32, float* features, const int32_t* field_strain,
                      double* acc, int n_strains, int32_t* n_instances_dev, int32_t* labels_out, void* stream);
/* Test taps: the plan entry of a layer (info[6] = mode {-1 first, 0 direct, 1 pooled, 2 up ++ skip}, c0, c1, cout,
 * log2 of the resolution divisor, number of 3x3 layers) and one layer run on caller-provided fp16 chunk-planar
 * activations [C/8][H][W][8] (layer -2 = the heads). */
int cia_seg_layer_info(cia_handle h, int layer, int32_t* info);
int cia_seg_debug_layer(cia_handle h, int layer, const void* src0, const void* src1, const float* image, int Ho, int Wo,
                        void* out, float* prob, float* dist, void* stream);

/* Number of kernels this library has launched on the handle (bench's gpu_launches). */
int64_t cia_launch_count(cia_handle h);

#ifdef __cplusplus
}
#endif
#endif /* CIA_H */
