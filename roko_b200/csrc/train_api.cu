// C ABI of the training path (include/roko_b200.h, "training" section): the train-mode forward of
// reference roko/rnn_model.py:46-59 with its four dropout sites, and the backward autograd would
// run for roko/train.py:46-53, as chains of kernels on the caller's stream.  The caller owns one
// scratch buffer that carries the saved activations from forward to backward.
#include <stdio.h>
#include <stdlib.h>

#include "../../include/roko_b200.h"
#include "model.h"
#include "train.cuh"

using namespace roko;

namespace {

int tfail(int code, const char* fmt, const char* a = "") {
    snprintf(roko_b200_errbuf(), ROKO_ERRBUF, fmt, a);
    return code;
}

#define TCU(call)                                                                                    \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            snprintf(roko_b200_errbuf(), ROKO_ERRBUF, "%s: %s", #call, cudaGetErrorString(e_));                 \
            return ROKO_B200_ECUDA;                                                                  \
        }                                                                                            \
    } while (0)

constexpr int TRAIN_MAX_WINDOWS = 1024;
constexpr size_t ROW_EP = (size_t)EMB * READS;       // per (window, column) row
constexpr size_t ROW_A1 = (size_t)EMB * FC1;
// per (window, column) row, without the materialised masked embedding (only the ROKO_B200_TRAIN_TC <= 4 chains keep one)
constexpr size_t ROW_FLOATS = ROW_A1 + IN0P + GI_N + 3 * (2 * HID * 4) + 3 * OUT_W + 2 * OUT_W
                              + GI_N + OUT_W + OUT_W + IN0P + MASK_WORDS + MASKT_WORDS + READS / 4;

bool keeps_ep(int train_tc) { return train_tc < 5; }
int train_tc_from_env() {                                 // what a model created now would use (api.cu reads the same variable)
    const char* tt = getenv("ROKO_B200_TRAIN_TC");
    return tt ? atoi(tt) : roko_b200_model::TRAIN_TC_DEFAULT;
}
size_t ws_bytes(int n_windows, int train_tc) {
    const size_t n = n_windows < 1 ? 1 : (size_t)n_windows;
    return n * COLS * (ROW_FLOATS + (keeps_ep(train_tc) ? ROW_EP : 0)) * sizeof(float);
}

struct TrainWs {
    float *ep, *a1, *u, *gi, *gates[3], *out[3], *outd[2], *dghp, *dghn, *dh, *din;
    uint32_t* bits;
    uint32_t* bitsT;                 // keep bits per read, [row][200][2]
    uint8_t* xt;                     // validated codes, [row][200]
};

TrainWs carve(void* base, size_t rows) {
    TrainWs w;
    float* p = static_cast<float*>(base);
    w.a1 = p; p += rows * ROW_A1;
    w.u = p; p += rows * IN0P;
    w.gi = p; p += rows * GI_N;
    for (int l = 0; l < 3; ++l) { w.gates[l] = p; p += rows * 2 * HID * 4; }
    for (int l = 0; l < 3; ++l) { w.out[l] = p; p += rows * OUT_W; }
    for (int l = 0; l < 2; ++l) { w.outd[l] = p; p += rows * OUT_W; }
    w.dghp = p; p += rows * GI_N;
    w.dghn = p; p += rows * OUT_W;
    w.dh = p; p += rows * OUT_W;
    w.din = p; p += rows * IN0P;
    w.bits = reinterpret_cast<uint32_t*>(p); p += rows * MASK_WORDS;
    w.bitsT = reinterpret_cast<uint32_t*>(p); p += rows * MASKT_WORDS;
    w.xt = reinterpret_cast<uint8_t*>(p); p += rows * (READS / 4);
    w.ep = p;                                             // last: only there when the chain materialises it (keeps_ep)
    return w;
}

int drop_cfg(float p, unsigned long long seed, DropCfg* d) {
    if (!(p >= 0.f) || p >= 1.f) return tfail(ROKO_B200_EARG, "dropout probability must be in [0, 1)%s");
    d->seed = seed;
    d->thresh = (unsigned int)((double)p * 4294967296.0);
    d->scale = (float)(1.0 / (1.0 - (double)p));
    return ROKO_B200_OK;
}

int check_train(roko_b200_model* m, const void* x, int n, const void* tws, size_t tws_bytes) {
    if (!m) return tfail(ROKO_B200_EARG, "model is NULL%s");
    if (!m->loaded) return tfail(ROKO_B200_ESTATE, "no weights loaded (call roko_b200_model_load)%s");
    if (n < 1 || n > TRAIN_MAX_WINDOWS) return tfail(ROKO_B200_EARG, "training batch must hold 1..1024 windows%s");
    if (!x || !tws) return tfail(ROKO_B200_EARG, "x / workspace is NULL%s");
    if (((uintptr_t)x & 15) || ((uintptr_t)tws & 15)) return tfail(ROKO_B200_EARG, "x / workspace must be 16-byte aligned%s");
    if (tws_bytes < ws_bytes(n, m->train_tc)) return tfail(ROKO_B200_EARG, "training workspace too small%s");
    return ROKO_B200_OK;
}

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

extern "C" {

size_t roko_b200_train_workspace_bytes(int n_windows) { return ws_bytes(n_windows, train_tc_from_env()); }

int roko_b200_train_forward(roko_b200_model* m, const uint8_t* x, int n_windows, float p_drop,
                            unsigned long long seed, float* logits, void* tws, size_t tws_bytes, void* stream) {
    if (int rc = check_train(m, x, n_windows, tws, tws_bytes)) return rc;
    if (!logits) return tfail(ROKO_B200_EARG, "logits is NULL%s");
    DropCfg d;
    if (int rc = drop_cfg(p_drop, seed, &d)) return rc;
    DevGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int rows = n_windows * COLS, rows50 = rows * EMB;
    TrainWs w = carve(tws, rows);
    const float* raw = m->raw_stage;
    const float* pk = m->packed;

    TCU(cudaMemsetAsync(w.u, 0, (size_t)rows * IN0P * sizeof(float), s));      // the 12 pad columns stay zero
    const bool gen_ep = m->train_tc >= 5;                 // ep is rebuilt inside its consumers from (codes, keep bits), never stored
    const EpGen gen{w.xt, w.bits, w.bitsT, raw + RAW_E, d.scale, nullptr};
    TCU(launch_embed_drop(x, raw + RAW_E, gen_ep ? nullptr : w.ep, w.bits, w.xt, gen_ep ? w.bitsT : nullptr, n_windows, d, m->status, s));
    if (m->train_tc) {   // a1 = dropout(relu(ep W1^T + b1))                     rnn_model.py:50-51
        TCU(launch_train_images(raw, m->train_img, s));
        if (gen_ep) TCU(launch_fc1_gen(gen, m->train_img, raw + RAW_B1, w.a1, rows50, d, m->num_sms, s));
        else TCU(launch_fc1_tc(w.ep, m->train_img, raw + RAW_B1, w.a1, rows50, d, m->num_sms, s));
    } else {
        GemmArgs a{};
        a.A = w.ep; a.lda = READS; a.B = raw + RAW_W1; a.ldb = READS; a.C = w.a1; a.ldc = FC1;
        a.M = rows50; a.N = FC1; a.K = READS; a.bias = raw + RAW_B1; a.drop = d;
        TCU(launch_gemm(a, true, true, EPI_FC1, 1, m->num_sms, s));
    }
    TCU(launch_fc2_fwd(w.a1, raw + RAW_W2, raw + RAW_B2, w.u, rows50, d, s));
    const float* in = w.u;
    const size_t dstride = (size_t)(pk_whh(0, 1) - pk_whh(0, 0));
    for (int l = 0; l < LAYERS; ++l) {
        TCU(proj_dispatch(m, in, l, w.gi, rows, m->num_sms, s));       // one stream: the whole chip
        TCU(launch_rec_train(w.gi, pk + pk_whh(l, 0), dstride, pk + pk_bhn(l, 0), w.out[l],
                             reinterpret_cast<float4*>(w.gates[l]), n_windows, m->num_sms, s));
        if (l + 1 < LAYERS) {                                                   // nn.GRU(dropout=...): between layers only
            TCU(launch_drop_apply(w.out[l], w.outd[l], (size_t)rows * OUT_W, DROP_GRU0 + l, d, s));
            in = w.outd[l];
        }
    }
    TCU(launch_head(w.out[LAYERS - 1], pk + PK_W4, pk + PK_B4, logits, nullptr, rows, HEAD_BLOCKS_PER_SM * m->num_sms, s));
    return ROKO_B200_OK;
}

int roko_b200_train_backward(roko_b200_model* m, const uint8_t* x, int n_windows, float p_drop,
                             unsigned long long seed, const float* dlogits, float* grad_raw, void* tws,
                             size_t tws_bytes, void* stream) {
    if (int rc = check_train(m, x, n_windows, tws, tws_bytes)) return rc;
    if (!dlogits || !grad_raw) return tfail(ROKO_B200_EARG, "dlogits / grad_raw is NULL%s");
    DropCfg d;
    if (int rc = drop_cfg(p_drop, seed, &d)) return rc;
    DevGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int rows = n_windows * COLS, rows50 = rows * EMB, sms = m->num_sms;
    TrainWs w = carve(tws, rows);
    const float* raw = m->raw_stage;
    float* dgi = w.gi;                                   // the forward's gi scratch is free by now

    TCU(cudaMemsetAsync(grad_raw, 0, (size_t)RAW_TOTAL * sizeof(float), s));
    {   // fc4: dh = dlogits W4 ; dW4 = dlogits^T h ; db4 = colsum(dlogits)
        GemmArgs a{};
        a.A = dlogits; a.lda = CLASSES; a.B = raw + RAW_W4; a.ldb = OUT_W; a.C = w.dh; a.ldc = OUT_W;
        a.M = rows; a.N = OUT_W; a.K = CLASSES;
        TCU(launch_gemm(a, true, false, EPI_STORE, 1, sms, s));
        GemmArgs b{};
        b.A = dlogits; b.lda = CLASSES; b.B = w.out[LAYERS - 1]; b.ldb = OUT_W; b.C = grad_raw + RAW_W4; b.ldc = OUT_W;
        b.M = CLASSES; b.N = OUT_W; b.K = rows;
        TCU(launch_gemm(b, false, false, EPI_ATOMIC, 0, sms, s));
        TCU(launch_colsum(dlogits, CLASSES, rows, CLASSES, grad_raw + RAW_B4, s));
    }
    for (int l = LAYERS - 1; l >= 0; --l) {
        const int in_w = gru_in(l), in_ld = gru_inp(l);
        const float* in = l == 0 ? w.u : w.outd[l - 1];
        TCU(launch_rec_bwd(w.dh, reinterpret_cast<const float4*>(w.gates[l]), w.out[l], raw + raw_whh(l, 0),
                           (size_t)raw_dir_size(l), dgi, w.dghn, w.dghp, n_windows, sms, s));
        if (m->train_tc >= 6)                             // dW_ih, dW_hh of both directions: one tcgen05 launch per layer
            TCU(launch_gru_dw(l, dgi, in, w.dghp, w.out[l], grad_raw, rows, sms, s));
        for (int dir = 0; dir < 2 && m->train_tc < 6; ++dir) {
            if (m->train_tc == 4) {                       // the same products, one launch each
                TCU(launch_tn_tc(dgi + dir * G3, GI_N, G3, in, in_ld, in_w, grad_raw + raw_wih(l, dir), in_w, rows, sms, s));
                TCU(launch_tn_tc(w.dghp + dir * G3, GI_N, G3, w.out[l] + dir * HID, OUT_W, HID, grad_raw + raw_whh(l, dir), HID,
                                 rows, sms, s));
                continue;
            }
            GemmArgs a{};                                 // dW_ih = dgi_d^T in
            a.A = dgi + dir * G3; a.lda = GI_N; a.B = in; a.ldb = in_ld; a.C = grad_raw + raw_wih(l, dir); a.ldc = in_w;
            a.M = G3; a.N = in_w; a.K = rows;
            TCU(launch_gemm(a, false, false, EPI_ATOMIC, 0, sms, s));
            GemmArgs b{};                                 // dW_hh = dgh_prev_d^T out_d
            b.A = w.dghp + dir * G3; b.lda = GI_N; b.B = w.out[l] + dir * HID; b.ldb = OUT_W;
            b.C = grad_raw + raw_whh(l, dir); b.ldc = HID; b.M = G3; b.N = HID; b.K = rows;
            TCU(launch_gemm(b, false, false, EPI_ATOMIC, 0, sms, s));
        }
        TCU(launch_gru_bias_grad(dgi, w.dghn, rows, grad_raw + raw_bih(l, 0), grad_raw + raw_bhh(l, 0),
                                 grad_raw + raw_bih(l, 1), grad_raw + raw_bhh(l, 1), s));
        if (m->train_tc >= 3) {                           // d(in) = dgi W_ih, both directions in one K = 768 product
            TCU(launch_din_tc(l, dgi, m->train_img, w.din, rows, sms, s));
        } else {
            for (int dir = 0; dir < 2; ++dir) {           // d(in) = dgi_fwd W_ih_fwd + dgi_bwd W_ih_bwd
                GemmArgs a{};
                a.A = dgi + dir * G3; a.lda = GI_N; a.B = m->raw_al + raw_al_off(raw_wih(l, dir)); a.ldb = in_w; a.C = w.din; a.ldc = in_ld;
                a.M = rows; a.N = in_w; a.K = G3;
                TCU(launch_gemm(a, true, false, dir == 0 ? EPI_STORE : EPI_ACC, 1, sms, s));
            }
        }
        if (l > 0)
            TCU(launch_drop_apply(w.din, w.dh, (size_t)rows * OUT_W, DROP_GRU0 + (l - 1), d, s));
    }
    // front end: fc2, fc1, embedding
    TCU(launch_fc2_bwd(w.din, w.u, w.a1, raw + RAW_W2, grad_raw + RAW_W2, grad_raw + RAW_B2, grad_raw + RAW_B1, rows50, d.scale, sms, s));
    {
        const bool gen_ep = m->train_tc >= 5;
        const EpGen gen{w.xt, w.bits, w.bitsT, raw + RAW_E, d.scale, grad_raw + RAW_E};
        if (gen_ep) {                                     // dW1 = dap^T ep, ep rebuilt from (codes, keep bits)
            TCU(launch_dw1_gen(w.a1, gen, grad_raw + RAW_W1, rows50, sms, s));
        } else if (m->train_tc >= 2) {                    // dW1 = dap^T ep
            TCU(launch_dw1_tc(w.a1, w.ep, grad_raw + RAW_W1, rows50, sms, s));
        } else {
            GemmArgs a{};
            a.A = w.a1; a.lda = FC1; a.B = w.ep; a.ldb = READS; a.C = grad_raw + RAW_W1; a.ldc = READS;
            a.M = FC1; a.N = READS; a.K = rows50;
            TCU(launch_gemm(a, false, false, EPI_ATOMIC, 0, sms, s));
        }
        if (gen_ep) {                                     // dE straight from the d(ep) = dap W1 tiles
            TCU(launch_dep_de(w.a1, m->train_img, gen, rows50, sms, s));
            return ROKO_B200_OK;
        }
        if (m->train_tc) {                                // dep = dap W1 (over ep, which nothing reads any more)
            TCU(launch_dep_tc(w.a1, m->train_img, w.ep, rows50, sms, s));
        } else {
            GemmArgs b{};
            b.A = w.a1; b.lda = FC1; b.B = raw + RAW_W1; b.ldb = READS; b.C = w.ep; b.ldc = READS;
            b.M = rows50; b.N = READS; b.K = FC1;
            TCU(launch_gemm(b, true, false, EPI_STORE, 1, sms, s));
        }
        TCU(launch_embed_grad(w.ep, x, w.bits, grad_raw + RAW_E, n_windows, d.scale, sms, s));
    }
    return ROKO_B200_OK;
}

int roko_b200_dropout_mask(float p_drop, unsigned long long seed, int site, size_t n, uint8_t* mask_out,
                           void* stream) {
    if (site < 0 || site >= DROP_SITES || !mask_out) return tfail(ROKO_B200_EARG, "bad site / mask_out%s");
    DropCfg d;
    if (int rc = drop_cfg(p_drop, seed, &d)) return rc;
    TCU(launch_drop_mask((unsigned int)site, n, mask_out, d, static_cast<cudaStream_t>(stream)));
    return ROKO_B200_OK;
}

}  // extern "C"
