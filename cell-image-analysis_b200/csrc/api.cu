// api.cu -- the extern "C" boundary of libcia.so (include/cia.h): handle lifecycle,
// artifact upload, stage wrappers and the fused screening path.
#include "common.cuh"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#define CIA_VERSION 100

static int bad_handle() { return CIA_E_ARG; }

template <typename T>
static int upload(cia_ctx* h, T** dst, const T* src, size_t n) {
    cudaFree(*dst); *dst = nullptr;
    CIA_CUDA(cudaMalloc((void**)dst, n * sizeof(T)));
    CIA_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return CIA_OK;
}

extern "C" {

int cia_version(void) { return CIA_VERSION; }

void cia_default_params(cia_params* p) {
    if (!p) return;
    p->border_margin = 10;      // det:76
    p->area_min = 200;          // det:80
    p->area_max = 8000;
    p->ecc_max = 0.95;          // det:84
    p->mean_min = 0.5;          // det:94
    p->std_min = 0.1;
    p->clip_limit = 0.02;       // det:98
    p->intensity_inv = 1.0 / 65535.0;   // img_as_float of a uint16 image (inside det:98)
}

int cia_create(int device, cia_handle* out) {
    if (!out) return CIA_E_ARG;
    *out = nullptr;
    cia_ctx* h = new (std::nothrow) cia_ctx();
    if (!h) return CIA_E_ARG;
    h->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { delete h; return CIA_E_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) { h->num_sms = prop.multiProcessorCount; h->max_smem_optin = (int)prop.sharedMemPerBlockOptin; }
    if (cudaMalloc(&h->status_dev, sizeof(int32_t)) != cudaSuccess ||
        cudaMemset(h->status_dev, 0, sizeof(int32_t)) != cudaSuccess ||
        cudaMallocHost(&h->status_host, sizeof(int32_t)) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return CIA_E_CUDA;
    }
    *out = h;
    return CIA_OK;
}

int cia_set_option(cia_handle h, const char* name, double value) {
    if (!h) return bad_handle();
    if (!name) { h->err = "cia_set_option: null name"; return CIA_E_ARG; }
    const std::string n(name);
    if (n == "cae_pass_cells") {
        if (!(value >= 1 && value <= 1 << 20)) { h->err = "cia_set_option: cae_pass_cells must be in [1, 2^20]"; return CIA_E_ARG; }
        h->cae_pass_cells = (int)value;
    } else if (n == "cae_l1_debias" || n == "cae_l2_debias" || n == "cae_l3_debias") {
        if (!(value >= 0 && value <= 64)) { h->err = "cia_set_option: debias must be in [0, 64] (units of 2^-24)"; return CIA_E_ARG; }
        h->cae_debias[n[5] - '1'] = (float)value;
    } else if (n == "svm_kernel") {
        if (value != 0 && value != 1) { h->err = "cia_set_option: svm_kernel is 0 (fp64 DMMA) or 1 (tcgen05)"; return CIA_E_ARG; }
        h->svm_kernel = (int)value;
    } else if (n == "pca_kernel") {
        if (value != 0 && value != 1) { h->err = "cia_set_option: pca_kernel is 0 (fp64 DMMA) or 1 (tcgen05)"; return CIA_E_ARG; }
        h->pca_kernel = (int)value;
    } else if (n == "svm_refine") {
        h->svm_refine = value != 0;
    } else if (n == "seg_conv_tma") {
        // segmentation: 1 = single-chunk direct layers run the TMA-fed warp-specialised kernel, 0 = the staged kernel everywhere
        h->seg_conv_tma = value != 0;
    } else if (n == "seg_pool_out") {
        h->seg_pool_out = value != 0;
    } else if (n == "seg_conv_ws") {
        // segmentation: the warp-specialised software-producer kernel: 1 = for the layers where it measured faster, 2 = every
        // layer the TMA kernel does not take, 0 = the staged kernel
        if (value != 0 && value != 1 && value != 2) { h->err = "cia_set_option: seg_conv_ws is 0 (off), 1 (where it pays) or 2 (every layer)"; return CIA_E_ARG; }
        h->seg_conv_ws = (int)value;
    } else {
        h->err = "cia_set_option: unknown option '" + n + "'";
        return CIA_E_ARG;
    }
    return CIA_OK;
}

static void free_cae(CaeWeights& w) {
    for (int i = 0; i < CAE_NCONV; ++i) {
        cudaFree(w.kernel[i]); cudaFree(w.bias[i]); cudaFree(w.bn_scale[i]); cudaFree(w.bn_shift[i]);
        w.kernel[i] = w.bias[i] = w.bn_scale[i] = w.bn_shift[i] = nullptr;
    }
    for (int i = 0; i < CAE_NCONV; ++i)
        for (int j = 0; j < 2; ++j) { cudaFree(w.tc_w[i][j]); w.tc_w[i][j] = nullptr; }
    cudaFree(w.tc_w7); w.tc_w7 = nullptr;
    w.tc_ready = false;
    w.loaded = false;
}

int cia_destroy(cia_handle h) {
    if (!h) return bad_handle();
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    free_cae(h->cae[0]); free_cae(h->cae[1]);
    k_seg_free(h);
    cudaFree(h->sp.center); cudaFree(h->sp.scale); cudaFree(h->sp.rscale); cudaFree(h->sp.comp_pad); cudaFree(h->sp.offset); cudaFree(h->sp.tc_img); cudaFree(h->sp.tc_par);
    for (int i = 0; i < 2; ++i) { cudaFree(h->svm[i].sv_t); cudaFree(h->svm[i].coef); cudaFree(h->svm[i].sv_pad); cudaFree(h->svm[i].gsn);
                                  cudaFree(h->svm[i].tc_hi); cudaFree(h->svm[i].tc_lo); cudaFree(h->svm[i].tc_gcol); }
    Workspace* ws[] = {&h->ws_flags, &h->ws_act, &h->ws_crop_scratch, &h->ws_pipe, &h->ws_feat,
                       &h->ws_misc, &h->ws_stage, &h->ws_svm, &h->ws_fit, &h->ws_seg_norm};
    for (Workspace* w : ws) cudaFree(w->p);
    cudaFree(h->status_dev);
    cudaFreeHost(h->status_host);
    if (h->ev) cudaEventDestroy(h->ev);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->side) cudaStreamDestroy(h->side);
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->prof_layer_ev) cudaEventDestroy(e);
    delete h;
    return CIA_OK;
}

const char* cia_last_error(cia_handle h) { return h ? h->err.c_str() : "null handle"; }

int64_t cia_launch_count(cia_handle h) { return h ? h->launches : 0; }

int cia_debug_copy_workspace(cia_handle h, int ws_id, size_t offset, void* dst_host, size_t bytes) {
    if (!h) return bad_handle();
    Workspace* ws[] = {&h->ws_flags, &h->ws_act, &h->ws_crop_scratch, &h->ws_pipe, &h->ws_feat,
                       &h->ws_misc, &h->ws_stage, &h->ws_svm, &h->ws_fit};
    if (ws_id < 0 || ws_id >= (int)(sizeof(ws) / sizeof(ws[0])) || !dst_host || offset + bytes > ws[ws_id]->cap) {
        h->err = "cia_debug_copy_workspace: bad argument";
        return CIA_E_ARG;
    }
    CIA_CUDA(cudaDeviceSynchronize());
    CIA_CUDA(cudaMemcpy(dst_host, (const char*)ws[ws_id]->p + offset, bytes, cudaMemcpyDeviceToHost));
    return CIA_OK;
}

int cia_check_status(cia_handle h, void* stream) {
    if (!h) return bad_handle();
    cudaStream_t s = (cudaStream_t)stream;
    CIA_CUDA(cudaMemcpyAsync(h->status_host, h->status_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CIA_CUDA(cudaMemsetAsync(h->status_dev, 0, sizeof(int32_t), s));
    CIA_CUDA(cudaStreamSynchronize(s));
    const int code = *h->status_host;
    if (code == CIA_E_CAPACITY) h->err = "device: output capacity exceeded (cells_cap too small)";
    else if (code == CIA_E_LABEL) h->err = "device: label outside [0, max_label]";
    else if (code == CIA_E_UNSUPPORTED) h->err = "device: bbox side > 1024 not supported by the crop kernel, or a tensor-core "
                                                 "autoencoder activation outside the fp16 range (use precision 0)";
    else if (code == CIA_E_ARG) h->err = "device: NaN in the features given to cia_fit_robust_scaler";
    else if (code != 0) h->err = "device: unknown status";
    return code;
}

// ---- artifacts --------------------------------------------------------------

int cia_load_cae(cia_handle h, int which, int n_conv, const float* const* kernels,
                 const float* const* biases, const float* const* bn, float bn_eps) {
    if (!h) return bad_handle();
    if (which < 0 || which > 1 || !kernels || !biases || !bn) { h->err = "cia_load_cae: bad argument"; return CIA_E_ARG; }
    if ((which == 0 && n_conv != 7) || (which == 1 && n_conv != 3)) {
        h->err = "cia_load_cae: topology is not CAE_improved_modeltrain.py:188-216 (7 convs) / its encoder (3)";
        return CIA_E_STATE;
    }
    CIA_CUDA(cudaSetDevice(h->device));
    CaeWeights& w = h->cae[which];
    free_cae(w);
    int rc;
    for (int i = 0; i < n_conv; ++i) {
        const int cin = kCaeCin[i], cout = kCaeCout[i];
        if ((rc = upload(h, &w.kernel[i], kernels[i], (size_t)9 * cin * cout))) return rc;
        if ((rc = upload(h, &w.bias[i], biases[i], (size_t)cout))) return rc;
        if (i < 6) {
            // tf.nn.batch_normalization inference: inv = gamma * rsqrt(var + eps);
            // y = x * inv + (beta - mean * inv), all float32
            std::vector<float> sc(cout), sh(cout);
            const float *g = bn[4 * i], *b = bn[4 * i + 1], *m = bn[4 * i + 2], *v = bn[4 * i + 3];
            for (int c = 0; c < cout; ++c) {
                const float inv = g[c] / std::sqrt(v[c] + bn_eps);
                sc[c] = inv;
                const float mi = m[c] * inv;
                sh[c] = b[c] - mi;
            }
            if ((rc = upload(h, &w.bn_scale[i], sc.data(), (size_t)cout))) return rc;
            if ((rc = upload(h, &w.bn_shift[i], sh.data(), (size_t)cout))) return rc;
        }
    }
    w.n_conv = n_conv;
    w.loaded = true;
    return k_cae_tc_prepare(h, which);
}

int cia_load_scaler_pca(cia_handle h, int F, int C, const double* center, const double* scale,
                        int center_is_f32, const double* components, const double* pca_offset,
                        int f32_flow) {
    if (!h) return bad_handle();
    if (F <= 0 || C <= 0 || !components || !pca_offset) { h->err = "cia_load_scaler_pca: bad argument"; return CIA_E_ARG; }
    CIA_CUDA(cudaSetDevice(h->device));
    ScalerPca& sp = h->sp;
    sp.loaded = false;
    int rc;
    sp.has_center = center != nullptr; sp.has_scale = scale != nullptr;
    if (center && (rc = upload(h, &sp.center, center, (size_t)F))) return rc;
    if (scale && (rc = upload(h, &sp.scale, scale, (size_t)F))) return rc;
    if (scale) {
        std::vector<double> rs((size_t)F);
        sp.rscale_ok = true;
        for (int f = 0; f < F; ++f) {
            rs[f] = 1.0 / scale[f];
            if (!std::isnormal(scale[f]) || !std::isnormal(rs[f])) sp.rscale_ok = false;
        }
        if ((rc = upload(h, &sp.rscale, rs.data(), rs.size()))) return rc;
    }
    std::vector<double> t((size_t)F * C);
    for (int c = 0; c < C; ++c)
        for (int f = 0; f < F; ++f) t[(size_t)f * C + c] = components[(size_t)c * F + f];
    {
        const int FP = (F + 31) / 32 * 32, CP = (C + 103) / 104 * 104;
        std::vector<double> tp((size_t)FP * CP, 0.0);
        for (int f = 0; f < F; ++f)
            for (int c = 0; c < C; ++c) tp[(size_t)f * CP + c] = t[(size_t)f * C + c];
        if ((rc = upload(h, &sp.comp_pad, tp.data(), tp.size()))) return rc;
        sp.CP = CP;
    }
    if ((rc = upload(h, &sp.offset, pca_offset, (size_t)C))) return rc;
    sp.F = F; sp.C = C; sp.center_is_f32 = center_is_f32; sp.f32_flow = f32_flow;
    if ((rc = k_pca_tc_prepare(h, sp, components))) return rc;
    sp.loaded = true;
    return CIA_OK;
}

int cia_load_svm(cia_handle h, int which, int n_sv, int dim, const double* sv, const double* coef,
                 double gamma, double rho) {
    if (!h) return bad_handle();
    if (which < 0 || which > 1 || n_sv <= 0 || dim <= 0 || !sv || !coef) { h->err = "cia_load_svm: bad argument"; return CIA_E_ARG; }
    CIA_CUDA(cudaSetDevice(h->device));
    SvmModel& m = h->svm[which];
    m.loaded = false;
    const int pad = (n_sv + 255) / 256 * 256;
    const int dpad = (dim + 15) / 16 * 16;
    std::vector<double> t((size_t)dim * pad, 0.0), a((size_t)pad, 0.0);
    std::vector<double> r((size_t)pad * dpad, 0.0), g((size_t)pad, 0.0);   // row-major copy + -gamma*||s||^2
    for (int i = 0; i < n_sv; ++i) {
        a[i] = coef[i];
        double ss = 0.0;
        for (int d = 0; d < dim; ++d) {
            const double v = sv[(size_t)i * dim + d];
            t[(size_t)d * pad + i] = v;
            r[(size_t)i * dpad + d] = v;
            ss += v * v;
        }
        g[i] = -gamma * ss;
    }
    int rc;
    if ((rc = upload(h, &m.sv_t, t.data(), t.size()))) return rc;
    if ((rc = upload(h, &m.coef, a.data(), a.size()))) return rc;
    if ((rc = upload(h, &m.sv_pad, r.data(), r.size()))) return rc;
    if ((rc = upload(h, &m.gsn, g.data(), g.size()))) return rc;
    m.n_sv = n_sv; m.n_sv_pad = pad; m.dim = dim; m.dim_pad = dpad; m.gamma = gamma; m.rho = rho;
    if ((rc = k_svm_tc_prepare(h, m, sv, coef))) return rc;
    m.loaded = true;
    return CIA_OK;
}

// ---- segmentation (segment.cu; improved_detection.py:44, 62-63) ----------------
int cia_seg_load(cia_handle h, const cia_seg_config* cfg, int n_layers, const float* const* kernels,
                 const float* const* biases, const int64_t* shapes, const double* ray_sin, const double* ray_cos) {
    if (!h) return bad_handle();
    if (!cfg || !kernels || !biases || !shapes || !ray_sin || !ray_cos || n_layers < 3) { h->err = "cia_seg_load: bad argument"; return CIA_E_ARG; }
    for (int l = 0; l < n_layers; ++l)
        if (!kernels[l] || !biases[l]) { h->err = "cia_seg_load: null layer"; return CIA_E_ARG; }
    cudaSetDevice(h->device);
    return k_seg_load(h, cfg, n_layers, kernels, biases, shapes, ray_sin, ray_cos);
}
int cia_seg_normalize(cia_handle h, const uint16_t* image, int H, int W, double pmin, double pmax, float* out,
                      float* mi_ma, void* stream) {
    if (!h) return bad_handle();
    if (!image || !out || H <= 0 || W <= 0 || !(pmin >= 0 && pmin <= pmax && pmax <= 100)) { h->err = "cia_seg_normalize: bad argument"; return CIA_E_ARG; }
    return k_seg_normalize(h, image, 1, H, W, H, W, pmin, pmax, out, mi_ma, (cudaStream_t)stream);
}
int cia_seg_predict(cia_handle h, const float* image, int H, int W, float* prob, float* dist, void* stream) {
    if (!h) return bad_handle();
    if (!image) { h->err = "cia_seg_predict: null image"; return CIA_E_ARG; }
    return k_seg_predict(h, image, 1, H, W, prob, dist, (cudaStream_t)stream);
}
int cia_seg_instances(cia_handle h, const float* prob, const float* dist, int Hg, int Wg, int grid, int H, int W,
                      double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_instances, void* stream) {
    if (!h) return bad_handle();
    if (!labels || Hg <= 0 || Wg <= 0 || grid <= 0 || H <= 0 || W <= 0) { h->err = "cia_seg_instances: bad argument"; return CIA_E_ARG; }
    return k_seg_instances(h, prob, dist, 1, Hg, Wg, Hg, Wg, grid, H, W, prob_thresh, nms_thresh, labels, n_instances,
                           (cudaStream_t)stream);
}

// ---- segmentation of F equally sized fields per call -------------------------------
static int seg_padded(cia_handle h, const char* who, int n_fields, int H, int W, int* Hp, int* Wp) {
    const int div = k_seg_div(h);
    if (!div) { h->err = std::string(who) + ": segmentation model not loaded (cia_seg_load)"; return CIA_E_STATE; }
    if (n_fields < 1 || n_fields > 65535 || H <= 0 || W <= 0) { h->err = std::string(who) + ": bad argument"; return CIA_E_ARG; }
    *Hp = (H + div - 1) / div * div;
    *Wp = (W + div - 1) / div * div;
    return CIA_OK;
}
int cia_seg_normalize_fields(cia_handle h, const uint16_t* images, int n_fields, int H, int W, double pmin, double pmax,
                             float* out, void* stream) {
    if (!h) return bad_handle();
    int Hp, Wp, rc;
    if ((rc = seg_padded(h, "cia_seg_normalize_fields", n_fields, H, W, &Hp, &Wp))) return rc;
    if (!images || !out || !(pmin >= 0 && pmin <= pmax && pmax <= 100)) { h->err = "cia_seg_normalize_fields: bad argument"; return CIA_E_ARG; }
    return k_seg_normalize(h, images, n_fields, H, W, Hp, Wp, pmin, pmax, out, nullptr, (cudaStream_t)stream);
}
int cia_seg_predict_fields(cia_handle h, const float* images, int n_fields, int Hp, int Wp, float* prob, float* dist,
                           void* stream) {
    if (!h) return bad_handle();
    if (!images || n_fields < 1) { h->err = "cia_seg_predict_fields: bad argument"; return CIA_E_ARG; }
    return k_seg_predict(h, images, n_fields, Hp, Wp, prob, dist, (cudaStream_t)stream);
}
int cia_seg_instances_fields(cia_handle h, const float* prob, const float* dist, int n_fields, int Hgp, int Wgp, int grid,
                             int H, int W, double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_instances,
                             void* stream) {
    if (!h) return bad_handle();
    if (!labels || n_fields < 1 || Hgp <= 0 || Wgp <= 0 || grid <= 0 || H <= 0 || W <= 0) {
        h->err = "cia_seg_instances_fields: bad argument";
        return CIA_E_ARG;
    }
    return k_seg_instances(h, prob, dist, n_fields, Hgp, Wgp, (H + grid - 1) / grid, (W + grid - 1) / grid, grid, H, W,
                           prob_thresh, nms_thresh, labels, n_instances, (cudaStream_t)stream);
}
int cia_seg_details(cia_handle h, int cap, int32_t* points, float* prob, float* coord, void* stream) {
    if (!h) return bad_handle();
    if (cap > 0 && (!points || !prob || !coord)) { h->err = "cia_seg_details: null pointer"; return CIA_E_ARG; }
    return k_seg_details(h, cap, points, prob, coord, (cudaStream_t)stream);
}
int cia_seg_layer_info(cia_handle h, int layer, int32_t* info) {
    if (!h) return bad_handle();
    if (!info) { h->err = "cia_seg_layer_info: null pointer"; return CIA_E_ARG; }
    return k_seg_layer_info(h, layer, info);
}
int cia_seg_debug_layer(cia_handle h, int layer, const void* src0, const void* src1, const float* image, int Ho, int Wo,
                        void* out, float* prob, float* dist, void* stream) {
    if (!h) return bad_handle();
    return k_seg_debug_layer(h, layer, src0, src1, image, Ho, Wo, out, prob, dist, (cudaStream_t)stream);
}

// ---- stage wrappers ----------------------------------------------------------
int cia_label_scan(cia_handle h, const int32_t* labels, int n_fields, int H, int W, int max_label,
                   cia_region* regions, void* stream) {
    if (!h) return bad_handle();
    if (!labels || !regions) { h->err = "cia_label_scan: null pointer"; return CIA_E_ARG; }
    return k_label_scan(h, labels, n_fields, H, W, max_label, regions, (cudaStream_t)stream);
}

int cia_filter(cia_handle h, const uint16_t* images, int n_fields, int H, int W, int max_label,
               cia_region* regions, const cia_params* params, cia_cell* cells, int cells_cap,
               int32_t* n_cells_dev, int32_t* field_counts_dev, void* stream) {
    if (!h) return bad_handle();
    if (!images || !regions || !params || !cells || !n_cells_dev) { h->err = "cia_filter: null pointer"; return CIA_E_ARG; }
    return k_filter(h, images, n_fields, H, W, max_label, regions, params, cells, cells_cap,
                    n_cells_dev, field_counts_dev, (cudaStream_t)stream);
}

int cia_solidity(cia_handle h, const int32_t* labels, int H, int W, const cia_cell* cells, int n_cells,
                 const int32_t* n_cells_dev, double* solidity, void* stream) {
    if (!h) return bad_handle();
    if (!labels || !cells || !solidity) { h->err = "cia_solidity: null pointer"; return CIA_E_ARG; }
    return k_solidity(h, labels, H, W, cells, n_cells, n_cells_dev, solidity, (cudaStream_t)stream);
}

int cia_crop_resize(cia_handle h, const uint16_t* images, int H, int W, const cia_cell* cells,
                    int n_cells, const int32_t* n_cells_dev, const cia_params* params,
                    float* crops32, double* crops64, void* stream) {
    if (!h) return bad_handle();
    if (!images || !cells || !params || !crops32) { h->err = "cia_crop_resize: null pointer"; return CIA_E_ARG; }
    return k_crop_resize(h, images, H, W, cells, n_cells, n_cells_dev, params, crops32, crops64,
                         (cudaStream_t)stream);
}

int cia_debug_clahe_levels(cia_handle h, const uint16_t* images, int H, int W, const cia_cell* cells,
                           int n_cells, const cia_params* params, float* crops32,
                           uint16_t* levels_out, const int64_t* level_offsets, void* stream) {
    if (!h) return bad_handle();
    if (!images || !cells || !params || !crops32 || !levels_out || !level_offsets) { h->err = "cia_debug_clahe_levels: null pointer"; return CIA_E_ARG; }
    return k_crop_resize(h, images, H, W, cells, n_cells, nullptr, params, crops32, nullptr,
                         (cudaStream_t)stream, levels_out, level_offsets);
}

int cia_cae_forward(cia_handle h, const float* crops32, int n_cells, const int32_t* n_cells_dev,
                    float* mse, float* mae, float* features, int precision, void* stream) {
    if (!h) return bad_handle();
    if (!crops32 || !mse || !mae) { h->err = "cia_cae_forward: null pointer"; return CIA_E_ARG; }
    if (precision == 0)
        return k_cae_forward_fp32(h, crops32, n_cells, n_cells_dev, mse, mae, features, (cudaStream_t)stream);
    if (precision >= 1 && precision <= 3)
        return k_cae_forward_tc(h, crops32, n_cells, n_cells_dev, mse, mae, features, precision, (cudaStream_t)stream);
    h->err = "cia_cae_forward: precision must be 0 (fp32), 1 (tensor core), 2 (tensor core + fp32 encoder) or 3 (tensor core + fp32 third layer)";
    return CIA_E_ARG;
}

int cia_svm_decision(cia_handle h, const float* features, int n_cells, const int32_t* n_cells_dev,
                     double* dec_cons, double* dec_mod, int8_t* pred_cons, int8_t* pred_mod,
                     double* pca_out, void* stream) {
    if (!h) return bad_handle();
    if (!features || !dec_cons || !dec_mod || !pred_cons || !pred_mod) { h->err = "cia_svm_decision: null pointer"; return CIA_E_ARG; }
    return k_svm_decision(h, features, n_cells, n_cells_dev, dec_cons, dec_mod, pred_cons, pred_mod,
                          pca_out, (cudaStream_t)stream);
}

int cia_strain_accumulate(cia_handle h, const cia_cell* cells, int n_cells,
                          const int32_t* n_cells_dev, const cia_scores* scores,
                          const int32_t* field_strain, double* acc, int n_strains, void* stream) {
    if (!h) return bad_handle();
    if (!cells || !scores || !acc || n_strains <= 0) { h->err = "cia_strain_accumulate: bad argument"; return CIA_E_ARG; }
    return k_strain_accumulate(h, cells, n_cells, n_cells_dev, scores, field_strain, acc, n_strains,
                               (cudaStream_t)stream);
}

// ---- fits of create_anomaly_detector (fit.cu; CAE_improved_modeltrain.py:404-423) ----
int cia_fit_robust_scaler(cia_handle h, const float* features, int n, int n_features, float* center, double* scale,
                          float* scaled, void* stream) {
    if (!h) return bad_handle();
    if (!features || !center || !scale || n < 1 || n_features < 1) { h->err = "cia_fit_robust_scaler: bad argument"; return CIA_E_ARG; }
    return k_fit_robust_scaler(h, features, n, n_features, center, scale, scaled, (cudaStream_t)stream);
}

int cia_fit_pca_gram(cia_handle h, const float* x, int n, int n_features, double* mean, double* cov, void* stream) {
    if (!h) return bad_handle();
    if (!x || !mean || !cov || n < 2 || n_features < 1) { h->err = "cia_fit_pca_gram: bad argument"; return CIA_E_ARG; }
    return k_fit_pca_gram(h, x, n, n_features, mean, cov, (cudaStream_t)stream);
}

int cia_ocsvm_fit(cia_handle h, const double* x, int l, int dim, double nu, double gamma, double tol, int max_iter,
                  double* alpha, double* result, void* stream) {
    if (!h) return bad_handle();
    if (!x || !alpha || !result || l < 1 || dim < 1 || !(nu > 0 && nu <= 1) || !(gamma > 0) || !(tol > 0) || max_iter < -1) {
        h->err = "cia_ocsvm_fit: bad argument";
        return CIA_E_ARG;
    }
    return k_ocsvm_fit(h, x, l, dim, nu, gamma, tol, max_iter, alpha, result, (cudaStream_t)stream);
}

// ---- fused path ---------------------------------------------------------------
}  // extern "C"

// labels (dense int32) or rle_slots (run-length transport format) -- exactly one is given
static int screen_fields_impl(cia_handle h, const uint16_t* images, const int32_t* labels,
                              const uint32_t* rle_slots, size_t slot_words, int n_fields,
                      int H, int W, int max_label, const cia_params* params, int precision,
                      cia_cell* cells, int cells_cap, int32_t* n_cells_dev,
                      int32_t* field_counts_dev, const cia_scores* scores, float* crops32,
                      float* features, const int32_t* field_strain, double* acc, int n_strains,
                      void* stream, const uint16_t* patches = nullptr, size_t patch_cap_px = 0) {
    if (!h) return bad_handle();
    if (!images || (!labels && !rle_slots) || !params || !cells || !n_cells_dev || !scores) {
        h->err = "cia_screen_fields: null pointer";
        return CIA_E_ARG;
    }
    if (cells_cap <= 0) { h->err = "cia_screen_fields: cells_cap must be > 0"; return CIA_E_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    // internal buffers: region tables, crops, features
    const size_t n_slots = (size_t)n_fields * max_label;
    const size_t reg_bytes = n_slots * sizeof(cia_region);
    const size_t crop_bytes = crops32 ? 0 : (size_t)cells_cap * 4096 * sizeof(float);
    const size_t feat_bytes = features ? 0 : (size_t)cells_cap * CIA_FEATURES * sizeof(float);
    if ((rc = ws_reserve(h, h->ws_pipe, reg_bytes + crop_bytes + feat_bytes + 512))) return rc;
    unsigned char* p = (unsigned char*)h->ws_pipe.p;
    cia_region* regions = (cia_region*)p; p += (reg_bytes + 255) & ~(size_t)255;
    float* crops = crops32 ? crops32 : (float*)p; p += (crop_bytes + 255) & ~(size_t)255;
    float* feats = features ? features : (float*)p;

    cudaEvent_t* pe = nullptr;
    if (h->prof_records > 0 && h->prof_used < h->prof_records)
        pe = &h->prof_ev[(size_t)(h->prof_used++) * CIA_PROF_MARKS];
#define CIA_MARK(i) do { if (pe) CIA_CUDA(cudaEventRecord(pe[i], s)); } while (0)
    CIA_MARK(0);
    if (labels) rc = k_label_scan(h, labels, n_fields, H, W, max_label, regions, s);
    else rc = k_label_scan_rle(h, rle_slots, slot_words, n_fields, H, W, max_label, regions, s);
    if (rc) return rc;
    // patch transport: the bbox rectangles of the regions just found go back to their places in the dense image
    if (patches && (rc = k_patch_scatter(h, patches, patch_cap_px, regions, n_fields, max_label, H, W,
                                         const_cast<uint16_t*>(images), s))) return rc;
    CIA_MARK(1);
    if ((rc = k_filter(h, images, n_fields, H, W, max_label, regions, params, cells, cells_cap,
                       n_cells_dev, field_counts_dev, s))) return rc;
    CIA_MARK(2);
    if ((rc = k_crop_resize(h, images, H, W, cells, cells_cap, n_cells_dev, params, crops, nullptr, s))) return rc;
    CIA_MARK(3);
    if (precision == 0) rc = k_cae_forward_fp32(h, crops, cells_cap, n_cells_dev, scores->mse, scores->mae, feats, s);
    else {
        h->layer_ev = pe ? &h->prof_layer_ev[(size_t)(h->prof_used - 1) * CIA_LAYER_PASSES * CIA_LAYER_MARKS] : nullptr;
        h->layer_passes = 0;
        rc = k_cae_forward_tc(h, crops, cells_cap, n_cells_dev, scores->mse, scores->mae, feats, precision, s);
        if (pe) h->prof_layer_passes[(size_t)(h->prof_used - 1)] = h->layer_passes;
        h->layer_ev = nullptr;
        h->prof_layers_valid = pe != nullptr;
    }
    if (rc) return rc;
    CIA_MARK(4);
    {
        // precision 0 is the exact anchor end to end: fp32 CUDA-core autoencoder AND the fp64 DMMA scoring kernels
        const int sk = h->svm_kernel, pk = h->pca_kernel;
        if (precision == 0) h->svm_kernel = h->pca_kernel = 0;
        rc = k_svm_decision(h, feats, cells_cap, n_cells_dev, scores->dec_conservative, scores->dec_moderate,
                            scores->pred_conservative, scores->pred_moderate, nullptr, s);
        h->svm_kernel = sk; h->pca_kernel = pk;
        if (rc) return rc;
    }
    CIA_MARK(5);
    if (acc) {
        if ((rc = k_strain_accumulate(h, cells, cells_cap, n_cells_dev, scores, field_strain, acc, n_strains, s))) return rc;
    }
    CIA_MARK(6);
#undef CIA_MARK
    return CIA_OK;
}

extern "C" {

int cia_screen_fields(cia_handle h, const uint16_t* images, const int32_t* labels, int n_fields,
                      int H, int W, int max_label, const cia_params* params, int precision,
                      cia_cell* cells, int cells_cap, int32_t* n_cells_dev,
                      int32_t* field_counts_dev, const cia_scores* scores, float* crops32,
                      float* features, const int32_t* field_strain, double* acc, int n_strains,
                      void* stream) {
    if (h && !labels) { h->err = "cia_screen_fields: null pointer"; return CIA_E_ARG; }
    return screen_fields_impl(h, images, labels, nullptr, 0, n_fields, H, W, max_label, params, precision,
                              cells, cells_cap, n_cells_dev, field_counts_dev, scores, crops32, features,
                              field_strain, acc, n_strains, stream);
}

int cia_screen_images(cia_handle h, const uint16_t* seg_images, const uint16_t* images, int n_fields, int H, int W,
                      double prob_thresh, double nms_thresh, int max_label, const cia_params* params, int precision,
                      cia_cell* cells, int cells_cap, int32_t* n_cells_dev, int32_t* field_counts_dev,
                      const cia_scores* scores, float* crops32, float* features, const int32_t* field_strain,
                      double* acc, int n_strains, int32_t* n_instances_dev, int32_t* labels_out, void* stream) {
    if (!h) return bad_handle();
    if (!seg_images) { h->err = "cia_screen_images: null pointer"; return CIA_E_ARG; }
    int Hp, Wp, rc;
    if ((rc = seg_padded(h, "cia_screen_images", n_fields, H, W, &Hp, &Wp))) return rc;
    const int grid = k_seg_grid(h);
    cudaStream_t s = (cudaStream_t)stream;
    float* norm = nullptr;
    int32_t* labels = nullptr;
    const size_t label_bytes = labels_out ? 0 : (size_t)n_fields * H * W * sizeof(int32_t);
    if ((rc = k_seg_screen_buffers(h, (size_t)n_fields * Hp * Wp * sizeof(float), label_bytes, &norm, &labels))) return rc;
    if (labels_out) labels = labels_out;
    // det:62 normalize(seg_channel) with csbdeep's defaults, det:63 predict_instances, then det:66-153
    if ((rc = k_seg_normalize(h, seg_images, n_fields, H, W, Hp, Wp, 3.0, 99.8, norm, nullptr, s))) return rc;
    if ((rc = k_seg_predict(h, norm, n_fields, Hp, Wp, nullptr, nullptr, s))) return rc;
    if ((rc = k_seg_instances(h, nullptr, nullptr, n_fields, Hp / grid, Wp / grid, (H + grid - 1) / grid, (W + grid - 1) / grid,
                              grid, H, W, prob_thresh, nms_thresh, labels, n_instances_dev, s))) return rc;
    return screen_fields_impl(h, images, labels, nullptr, 0, n_fields, H, W, max_label, params, precision, cells, cells_cap,
                              n_cells_dev, field_counts_dev, scores, crops32, features, field_strain, acc, n_strains, stream);
}

int cia_screen_fields_rle(cia_handle h, const uint16_t* images, const uint32_t* rle_slots,
                          size_t slot_words, int n_fields, int H, int W, int max_label,
                          const cia_params* params, int precision, cia_cell* cells, int cells_cap,
                          int32_t* n_cells_dev, int32_t* field_counts_dev, const cia_scores* scores,
                          float* crops32, float* features, const int32_t* field_strain, double* acc,
                          int n_strains, void* stream) {
    if (h && !rle_slots) { h->err = "cia_screen_fields_rle: null pointer"; return CIA_E_ARG; }
    return screen_fields_impl(h, images, nullptr, rle_slots, slot_words, n_fields, H, W, max_label, params,
                              precision, cells, cells_cap, n_cells_dev, field_counts_dev, scores, crops32,
                              features, field_strain, acc, n_strains, stream);
}

int cia_screen_fields_rle_patches(cia_handle h, uint16_t* images, const uint16_t* patches, size_t patch_cap_px,
                                  const uint32_t* rle_slots, size_t slot_words, int n_fields, int H, int W,
                                  int max_label, const cia_params* params, int precision, cia_cell* cells,
                                  int cells_cap, int32_t* n_cells_dev, int32_t* field_counts_dev,
                                  const cia_scores* scores, float* crops32, float* features,
                                  const int32_t* field_strain, double* acc, int n_strains, void* stream) {
    if (h && (!rle_slots || !patches || patch_cap_px == 0)) { h->err = "cia_screen_fields_rle_patches: null pointer"; return CIA_E_ARG; }
    return screen_fields_impl(h, images, nullptr, rle_slots, slot_words, n_fields, H, W, max_label, params,
                              precision, cells, cells_cap, n_cells_dev, field_counts_dev, scores, crops32,
                              features, field_strain, acc, n_strains, stream, patches, patch_cap_px);
}

int cia_label_scan_rle(cia_handle h, const uint32_t* rle_slots, size_t slot_words, int n_fields, int H,
                       int W, int max_label, cia_region* regions, void* stream) {
    if (!h) return bad_handle();
    if (!rle_slots || !regions) { h->err = "cia_label_scan_rle: null pointer"; return CIA_E_ARG; }
    return k_label_scan_rle(h, rle_slots, slot_words, n_fields, H, W, max_label, regions, (cudaStream_t)stream);
}

int cia_profile_begin(cia_handle h, int max_records) {
    if (!h) return bad_handle();
    if (max_records < 0) { h->err = "cia_profile_begin: bad argument"; return CIA_E_ARG; }
    CIA_CUDA(cudaSetDevice(h->device));
    const size_t want = (size_t)max_records * CIA_PROF_MARKS;
    while (h->prof_ev.size() < want) {
        cudaEvent_t e;
        CIA_CUDA(cudaEventCreate(&e));
        h->prof_ev.push_back(e);
    }
    h->prof_layer_passes.assign((size_t)max_records, 0);
    while (h->prof_layer_ev.size() < (size_t)max_records * CIA_LAYER_PASSES * CIA_LAYER_MARKS) {
        cudaEvent_t e;
        CIA_CUDA(cudaEventCreate(&e));
        h->prof_layer_ev.push_back(e);
    }
    h->prof_records = max_records;
    h->prof_used = 0;
    h->prof_layers_valid = false;
    return CIA_OK;
}

int cia_profile_layers(cia_handle h, double* layer_ms /* [7] */) {
    if (!h) return bad_handle();
    if (!layer_ms) { h->err = "cia_profile_layers: null pointer"; return CIA_E_ARG; }
    for (int k = 0; k < CIA_LAYER_MARKS - 1; ++k) layer_ms[k] = 0.0;
    if (!h->prof_layers_valid) { h->err = "cia_profile_layers: no tensor-core pass was profiled"; return CIA_E_STATE; }
    for (int r = 0; r < h->prof_used; ++r) {
        for (int p = 0; p < h->prof_layer_passes[(size_t)r]; ++p) {
            cudaEvent_t* le = &h->prof_layer_ev[((size_t)r * CIA_LAYER_PASSES + p) * CIA_LAYER_MARKS];
            CIA_CUDA(cudaEventSynchronize(le[CIA_LAYER_MARKS - 1]));
            for (int k = 0; k < CIA_LAYER_MARKS - 1; ++k) {
                float ms = 0.f;
                CIA_CUDA(cudaEventElapsedTime(&ms, le[k], le[k + 1]));
                layer_ms[k] += ms;
            }
        }
    }
    return CIA_OK;
}

int cia_profile_end(cia_handle h, double* stage_ms /* [6] */, int* n_records) {
    if (!h) return bad_handle();
    if (!stage_ms || !n_records) { h->err = "cia_profile_end: null pointer"; return CIA_E_ARG; }
    for (int k = 0; k < CIA_PROF_MARKS - 1; ++k) stage_ms[k] = 0.0;
    for (int r = 0; r < h->prof_used; ++r) {
        cudaEvent_t* pe = &h->prof_ev[(size_t)r * CIA_PROF_MARKS];
        CIA_CUDA(cudaEventSynchronize(pe[CIA_PROF_MARKS - 1]));
        for (int k = 0; k < CIA_PROF_MARKS - 1; ++k) {
            float ms = 0.f;
            CIA_CUDA(cudaEventElapsedTime(&ms, pe[k], pe[k + 1]));
            stage_ms[k] += ms;
        }
    }
    *n_records = h->prof_used;
    h->prof_records = 0;
    h->prof_used = 0;
    return CIA_OK;
}

int cia_screen_fields_host(cia_handle h, const uint16_t* images_host, const int32_t* labels_host,
                           int n_fields, int H, int W, int max_label, const cia_params* params,
                           int precision, cia_cell* cells_host, int cells_cap,
                           int32_t* n_cells_host, int32_t* field_counts_host,
                           const cia_scores* sh, void* stream) {
    if (!h) return bad_handle();
    if (!images_host || !labels_host || !params || !cells_host || !n_cells_host || !sh) {
        h->err = "cia_screen_fields_host: null pointer";
        return CIA_E_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t px = (size_t)n_fields * H * W;
    const size_t cap = (size_t)cells_cap;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_img = take(px * 2), o_lab = take(px * 4), o_cells = take(cap * sizeof(cia_cell));
    const size_t o_cnt = take(sizeof(int32_t) * (1 + (size_t)n_fields));
    const size_t o_mse = take(cap * 4), o_mae = take(cap * 4), o_dc = take(cap * 8), o_dm = take(cap * 8);
    const size_t o_pc = take(cap), o_pm = take(cap);
    int rc;
    if ((rc = ws_reserve(h, h->ws_stage, off))) return rc;
    unsigned char* b = (unsigned char*)h->ws_stage.p;
    CIA_CUDA(cudaMemcpyAsync(b + o_img, images_host, px * 2, cudaMemcpyHostToDevice, s));
    CIA_CUDA(cudaMemcpyAsync(b + o_lab, labels_host, px * 4, cudaMemcpyHostToDevice, s));
    cia_scores sd;
    sd.mse = (float*)(b + o_mse); sd.mae = (float*)(b + o_mae);
    sd.dec_conservative = (double*)(b + o_dc); sd.dec_moderate = (double*)(b + o_dm);
    sd.pred_conservative = (int8_t*)(b + o_pc); sd.pred_moderate = (int8_t*)(b + o_pm);
    int32_t* cnt = (int32_t*)(b + o_cnt);
    rc = cia_screen_fields(h, (const uint16_t*)(b + o_img), (const int32_t*)(b + o_lab), n_fields, H, W,
                           max_label, params, precision, (cia_cell*)(b + o_cells), cells_cap, cnt,
                           cnt + 1, &sd, nullptr, nullptr, nullptr, nullptr, 0, s);
    if (rc) return rc;
    CIA_CUDA(cudaMemcpyAsync(n_cells_host, cnt, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CIA_CUDA(cudaStreamSynchronize(s));
    int n = *n_cells_host;
    if (n > cells_cap) n = cells_cap;
    if (field_counts_host)
        CIA_CUDA(cudaMemcpyAsync(field_counts_host, cnt + 1, sizeof(int32_t) * n_fields, cudaMemcpyDeviceToHost, s));
    if (n > 0) {
        CIA_CUDA(cudaMemcpyAsync(cells_host, b + o_cells, (size_t)n * sizeof(cia_cell), cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->mse, sd.mse, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->mae, sd.mae, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->dec_conservative, sd.dec_conservative, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->dec_moderate, sd.dec_moderate, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->pred_conservative, sd.pred_conservative, (size_t)n, cudaMemcpyDeviceToHost, s));
        CIA_CUDA(cudaMemcpyAsync(sh->pred_moderate, sd.pred_moderate, (size_t)n, cudaMemcpyDeviceToHost, s));
    }
    return cia_check_status(h, stream);
}

}  // extern "C"
