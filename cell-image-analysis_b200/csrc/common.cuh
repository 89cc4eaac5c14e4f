// common.cuh -- context, workspace and small device helpers shared by libcia's
// translation units.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <set>
#include <string>
#include <vector>

#include "../../include/cia.h"

#define CIA_NUM_SMS_DEFAULT 148

// CAE topology of CAE_improved_modeltrain.py:188-216
#define CAE_NCONV 7
static const int kCaeCin[CAE_NCONV]  = {1, 32, 64, 32, 32, 64, 32};
static const int kCaeCout[CAE_NCONV] = {32, 64, 32, 32, 64, 32, 1};

struct CaeWeights {
    bool loaded = false;
    int n_conv = 0;
    float* kernel[CAE_NCONV] = {};   // HWIO fp32 (tap, ci, co)
    float* bias[CAE_NCONV] = {};
    float* bn_scale[CAE_NCONV] = {}; // gamma / sqrt(var + eps)            (fp32, folded like tf.nn.batch_normalization)
    float* bn_shift[CAE_NCONV] = {}; // beta - mean * scale
    // tensor-core operand images (built at load time, see cae_tc.cu): per layer the fp16
    // hi / lo parts of the power-of-two scaled weights in UMMA K-major core-matrix order
    void* tc_w[CAE_NCONV][2] = {};
    void* tc_w7 = nullptr;           // layer 7 as one tap with the (phase, neighbour) pairs on N (final_tapsum_kernel)
    float tc_inv_scale[CAE_NCONV] = {};
    bool tc_ready = false;
};

struct SvmModel {
    bool loaded = false;
    int n_sv = 0, dim = 0;
    double* sv_t = nullptr;   // [dim, n_sv_pad] transposed for coalesced reads
    double* coef = nullptr;   // [n_sv_pad] (zero padded)
    double* sv_pad = nullptr; // [n_sv_pad, dim_pad] row-major, zero padded (GEMM-form kernel)
    double* gsn = nullptr;    // [n_sv_pad] -gamma * ||s_i||^2
    int n_sv_pad = 0, dim_pad = 0;
    double gamma = 0, rho = 0;
    // tensor-core operand images (score_tc.cu): fp16 hi / lo parts of the 2^tc_es scaled support vectors as
    // [SV tile of 128][dim / 8][128][8], and per SV log2(e) * -gamma||s||^2 + log2(coef)
    void* tc_hi = nullptr;
    void* tc_lo = nullptr;
    float* tc_gcol = nullptr;
    int tc_es = 0, tc_svt = 0, tc_fx = 40;   // tc_fx: the row sums are 64-bit fixed point with 2^-tc_fx resolution
    bool tc_ok = false;
};

struct ScalerPca {
    bool loaded = false;
    int F = 0, C = 0;
    int center_is_f32 = 1, f32_flow = 1, has_center = 0, has_scale = 0;
    double* center = nullptr;   // [F]
    double* scale = nullptr;    // [F]
    double* rscale = nullptr;   // [F] 1 / scale, correctly rounded on the host (division by FMA correction)
    bool rscale_ok = false;     // every scale and reciprocal is a normal number
    double* comp_pad = nullptr; // [F rounded up to 32, CP] zero-padded copy for the cp.async-fed DMMA kernel
    int CP = 0;                 // C rounded up to a multiple of 104
    double* offset = nullptr;   // [C]
    // tensor-core operand image of the components (score_tc.cu): fp16 hi | lo of the 2^tc_ew scaled rows
    void* tc_img = nullptr;
    void* tc_par = nullptr;     // per feature {center, RN(1/scale), scale hi, scale lo} as fp32 (the kernel's fp32-only scaler)
    int tc_ew = 0;
    bool tc_ok = false;
};

struct Workspace {
    void* p = nullptr;
    size_t cap = 0;
};

struct SegModel;   // segment.cu

struct cia_ctx {
    int device = 0;
    SegModel* seg = nullptr;              // StarDist2D network + post-processing state (cia_seg_load)
    int num_sms = CIA_NUM_SMS_DEFAULT;
    int max_smem_optin = 227 * 1024;
    std::string err;
    CaeWeights cae[2];
    ScalerPca sp;
    SvmModel svm[2];
    int32_t* status_dev = nullptr;        // device status word (CIA_E_* raised by kernels)
    int32_t* status_host = nullptr;       // pinned
    int64_t launches = 0;
    std::set<const void*> attr_done;       // kernels whose opt-in smem attribute is set on THIS device
    // grow-only workspaces
    Workspace ws_flags, ws_act, ws_crop_scratch, ws_pipe, ws_feat, ws_misc, ws_stage, ws_svm;
    Workspace ws_fit;                      // fit.cu: sort buffers, covariance partials, SMO state
    Workspace ws_seg_norm;                 // segment.cu: per-field histograms and percentiles of the normalisation
    cudaEvent_t ev = nullptr;
    // side stream: the exact-fp32 encoder pass (FMA pipe) overlaps the tensor-core autoencoder
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // stage profiler: ring of CUDA events recorded in-stream by the fused path
    std::vector<cudaEvent_t> prof_ev;     // [records][CIA_PROF_MARKS]
    std::vector<cudaEvent_t> prof_layer_ev;   // [records][CIA_LAYER_PASSES][CIA_LAYER_MARKS]: CAE layer boundaries
    std::vector<int> prof_layer_passes;       // [records] passes recorded
    int layer_passes = 0;
    cudaEvent_t* layer_ev = nullptr;      // the current call's layer marks (null: not profiling)
    bool prof_layers_valid = false;
    int prof_records = 0, prof_used = 0;
    // cia_set_option: cells per pass of the tensor-core autoencoder (303 KB of activations per cell)
    // and the truncation compensation of its accumulating layers in units of 2^-24 (cae_tc.cu)
    int cae_pass_cells = 18944;
    float cae_debias[3] = {0.5f, 2.4f, 1.2f};   // L1, L2, L3
    // cia_set_option "svm_kernel": 1 = tcgen05 GEMM form (score_tc.cu), 0 = fp64 DMMA anchor (score.cu)
    int svm_kernel = 1;
    int pca_kernel = 1;        // "pca_kernel": 1 = tcgen05 projection (score_tc.cu), 0 = fp64 DMMA anchor
    int seg_pool_out = 1;      // "seg_pool_out": TMA-fed layers also write the max-pooled copy the next layer reads (0: it pools itself)
    int seg_conv_ws = 1;       // "seg_conv_ws": warp-specialised software-producer kernel for the other layers (0: staged kernel)
    int seg_conv_tma = 1;      // "seg_conv_tma": segment.cu's TMA-fed convolution kernel for Cin = 32 direct layers (0: staged kernel)
    int svm_refine = 1;        // "svm_refine": decisions within the tensor-core kernel's error of 0 are recomputed in fp64
};
#define CIA_LAYER_MARKS 8  // before L1, after L1 .. L7
#define CIA_LAYER_PASSES 8 // passes of one call that carry marks (cells_cap <= 8 x 18944)
#define CIA_PROF_MARKS 7   // before scan, after scan, gates, crop, cae, svm, accumulate

#define CIA_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) {                                                    \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);            \
            return CIA_E_CUDA;                                                      \
        }                                                                           \
    } while (0)

#define CIA_LAUNCH_CHECK()                                                          \
    do {                                                                            \
        h->launches++;                                                              \
        cudaError_t e_ = cudaGetLastError();                                        \
        if (e_ != cudaSuccess) {                                                    \
            h->err = std::string("kernel launch: ") + cudaGetErrorString(e_);       \
            return CIA_E_CUDA;                                                      \
        }                                                                           \
    } while (0)

static inline int ws_reserve(cia_ctx* h, Workspace& w, size_t bytes) {
    if (bytes <= w.cap) return CIA_OK;
    if (w.p) {
        CIA_CUDA(cudaDeviceSynchronize());
        CIA_CUDA(cudaFree(w.p));
        w.p = nullptr; w.cap = 0;
    }
    size_t want = bytes + bytes / 4 + 256;
    CIA_CUDA(cudaMalloc(&w.p, want));
    w.cap = want;
    return CIA_OK;
}

// function attributes are per device: remember them per handle, not in a process-wide static
static inline bool first_use(cia_ctx* h, const void* fn) { return h->attr_done.insert(fn).second; }

// ---- device helpers -------------------------------------------------------
__device__ __forceinline__ int dev_count(int n, const int32_t* n_dev) {
    if (n_dev == nullptr) return n;
    int m = *n_dev;
    return m < n ? m : n;
}

__device__ __forceinline__ void raise_status(int32_t* status, int code) {
    if (status) atomicMin(status, code);   // codes are negative; keep the first/lowest
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// stage-level forward declarations (one per .cu)
int k_label_scan_rle(cia_ctx* h, const uint32_t* slots, size_t slot_words, int n_fields, int H, int W,
                     int max_label, cia_region* regions, cudaStream_t s);
int k_patch_scatter(cia_ctx* h, const uint16_t* patches, size_t cap_px, const cia_region* regions, int n_fields,
                    int max_label, int H, int W, uint16_t* images, cudaStream_t s);
int k_label_scan(cia_ctx* h, const int32_t* labels, int n_fields, int H, int W, int max_label,
                 cia_region* regions, cudaStream_t s);
int k_filter(cia_ctx* h, const uint16_t* images, int n_fields, int H, int W, int max_label,
             cia_region* regions, const cia_params* p, cia_cell* cells, int cells_cap,
             int32_t* n_cells_dev, int32_t* field_counts_dev, cudaStream_t s);
int k_solidity(cia_ctx* h, const int32_t* labels, int H, int W, const cia_cell* cells, int n_cells,
               const int32_t* n_dev, double* out, cudaStream_t s);
int k_crop_resize(cia_ctx* h, const uint16_t* images, int H, int W, const cia_cell* cells,
                  int n_cells, const int32_t* n_cells_dev, const cia_params* p, float* crops32,
                  double* crops64, cudaStream_t s, uint16_t* levels_out = nullptr,
                  const int64_t* level_offsets = nullptr);
int k_cae_forward_fp32(cia_ctx* h, const float* crops, int n, const int32_t* n_dev, float* mse,
                       float* mae, float* features, cudaStream_t s);
int k_cae_forward_tc(cia_ctx* h, const float* crops, int n, const int32_t* n_dev, float* mse,
                     float* mae, float* features, int mode, cudaStream_t s);
int k_encoder_fp32(cia_ctx* h, const CaeWeights& w, const float* crops, int n, const int32_t* n_dev,
                   float* features, cudaStream_t s);
int k_conv3_fp32(cia_ctx* h, const CaeWeights& w, const float* a2, int n, const int32_t* n_dev,
                 float* features, int cell0, int chunk, cudaStream_t s);
int k_cae_tc_prepare(cia_ctx* h, int which);
int k_svm_decision(cia_ctx* h, const float* features, int n, const int32_t* n_dev,
                   double* dec_cons, double* dec_mod, int8_t* pred_cons, int8_t* pred_mod,
                   double* pca_out, cudaStream_t s);
int k_pca_tc_prepare(cia_ctx* h, ScalerPca& sp, const double* components);
int k_pca_tc(cia_ctx* h, const float* features, int n, const int32_t* n_dev, double* z, bool* done, cudaStream_t s);
int k_svm_tc_prepare(cia_ctx* h, SvmModel& m, const double* sv, const double* coef);
int k_svm_tc(cia_ctx* h, const SvmModel& m, const double* z, int n, const int32_t* n_dev, double* dec,
             int8_t* pred, bool* done, cudaStream_t s);
void k_seg_free(cia_ctx* h);
int k_seg_load(cia_ctx* h, const cia_seg_config* cfg, int n_layers, const float* const* kernels,
               const float* const* biases, const int64_t* shapes, const double* ray_sin, const double* ray_cos);
// segmentation of n_fields equally sized fields per call (the single-field entry points are n_fields = 1)
int k_seg_normalize(cia_ctx* h, const uint16_t* img, int n_fields, int H, int W, int Hp, int Wp, double pmin, double pmax,
                    float* out, float* mi_ma_out, cudaStream_t s);
int k_seg_predict(cia_ctx* h, const float* img, int n_fields, int H, int W, float* prob_out, float* dist_out, cudaStream_t s);
int k_seg_instances(cia_ctx* h, const float* prob, const float* dist, int n_fields, int Hgp, int Wgp, int hg, int wg,
                    int grid, int H, int W, double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_inst_dev,
                    cudaStream_t s);
int k_seg_div(cia_ctx* h);
int k_seg_grid(cia_ctx* h);
int k_seg_screen_buffers(cia_ctx* h, size_t norm_bytes, size_t label_bytes, float** norm, int32_t** labels);
int k_seg_details(cia_ctx* h, int cap, int32_t* points, float* prob, float* coord, cudaStream_t s);
int k_seg_layer_info(cia_ctx* h, int layer, int* info);
int k_seg_debug_layer(cia_ctx* h, int layer, const void* src0, const void* src1, const float* img, int Ho, int Wo,
                      void* out, float* prob, float* dist, cudaStream_t s);
int k_fit_robust_scaler(cia_ctx* h, const float* x, int n, int F, float* center, double* scale, float* scaled,
                        cudaStream_t s);
int k_fit_pca_gram(cia_ctx* h, const float* x, int n, int F, double* mean, double* cov, cudaStream_t s);
int k_ocsvm_fit(cia_ctx* h, const double* X, int l, int d, double nu, double gamma, double tol, int max_iter,
                double* alpha, double* result, cudaStream_t s);
int k_strain_accumulate(cia_ctx* h, const cia_cell* cells, int n, const int32_t* n_dev,
                        const cia_scores* sc, const int32_t* field_strain, double* acc,
                        int n_strains, cudaStream_t s);
