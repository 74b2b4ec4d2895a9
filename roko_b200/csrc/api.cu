// C ABI of libroko_b200 (include/roko_b200.h): model lifetime, weight packing, the forward pass
// as a chain of kernels on the caller's stream, and the pipelined host-buffer loop.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/roko_b200.h"
#include "model.h"
#include "train.cuh"

using namespace roko;

namespace {

thread_local char g_err[ROKO_ERRBUF] = "";

int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

#define CU(call)                                                                           \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) return fail(ROKO_B200_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

constexpr size_t WIN_BYTES = (size_t)READS * COLS;                  // 18 000
constexpr size_t WS_WIN_BYTES = WS_PER_WINDOW * sizeof(float) + WIN_BYTES;

// NVTX range around a C-ABI call (visible in nsys / ncu --nvtx; a no-op without an attached tool)
struct Range {
    explicit Range(const char* name) { nvtxRangePushA(name); }
    ~Range() { nvtxRangePop(); }
};

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace


namespace {

struct Taps { float *front, *gru[3]; };

// One chunked pass over n windows; everything is enqueued on `s`.
int run_forward(roko_b200_model* m, const uint8_t* x, int n, float* logits, uint8_t* labels, void* ws,
                size_t ws_bytes, cudaStream_t s, const Taps* taps, size_t per_window_bytes,
                cudaEvent_t* ev = nullptr) {
    const long long cap_ll = (long long)(ws_bytes / per_window_bytes);
    if (cap_ll < 1) return fail(ROKO_B200_EARG, "workspace smaller than one window%s%s");
    int cap = cap_ll > n ? n : (int)cap_ll;
    if (cap > 16384) cap = 16384;               // keeps the kernels' 32-bit element offsets in range
    if (taps && cap < n) return fail(ROKO_B200_EARG, "forward_taps needs the whole batch in the workspace%s%s");
    float* u = static_cast<float*>(ws);
    float* gi = u + (size_t)cap * WS_U;
    float* h0 = gi + (size_t)cap * WS_GI;
    float* h1 = h0 + (size_t)cap * WS_H;
    const float* pk = m->packed;

    for (int c0 = 0; c0 < n; c0 += cap) {
        const int nc = (n - c0) < cap ? (n - c0) : cap;
        const int rows = nc * COLS;
        const int front_ctas = launch_cap(m, nc, m->geo_front, m->num_sms);
        const int proj_ctas = launch_cap(m, (long long)((rows + TC_BM - 1) / TC_BM) * (GI_N / TC_BN), m->geo_proj, m->num_sms);
        const int head_ctas = launch_cap(m, rows, m->geo_head, HEAD_BLOCKS_PER_SM * m->num_sms);
        if (ev) CU(cudaEventRecord(ev[0], s));
        if (m->front_kind == 1) CU(launch_front_tc(x + (size_t)c0 * WIN_BYTES, pk, u, nc, m->status, front_ctas, s));
        else CU(launch_front(x + (size_t)c0 * WIN_BYTES, pk, u, nc, m->status, m->num_sms, s));
        if (taps && taps->front)
            CU(cudaMemcpy2DAsync(taps->front, IN0 * sizeof(float), u, IN0P * sizeof(float), IN0 * sizeof(float),
                                 rows, cudaMemcpyDeviceToDevice, s));
        const float* in = u;
        float* outs[3] = {h0, h1, h0};
        for (int l = 0; l < LAYERS; ++l) {
            if (ev) CU(cudaEventRecord(ev[1 + 2 * l], s));
            CU(proj_dispatch(m, in, l, gi, rows, proj_ctas, s));
            if (ev) CU(cudaEventRecord(ev[2 + 2 * l], s));
            CU(rec_dispatch(m, gi, l, outs[l], nc, s));
            if (taps && taps->gru[l])
                CU(cudaMemcpyAsync(taps->gru[l], outs[l], (size_t)rows * OUT_W * sizeof(float),
                                   cudaMemcpyDeviceToDevice, s));
            in = outs[l];
        }
        if (ev) CU(cudaEventRecord(ev[7], s));
        CU(launch_head(in, pk + PK_W4, pk + PK_B4, logits ? logits + (size_t)c0 * COLS * CLASSES : nullptr,
                       labels ? labels + (size_t)c0 * COLS : nullptr, rows, head_ctas, s));
        if (ev) CU(cudaEventRecord(ev[8], s));
    }
    return ROKO_B200_OK;
}

// ---- CUDA-graph replay of the 8-kernel chain ------------------------------------------------------
// A forward over a batch that fits the workspace is always the same 8 launches; only the input and
// output pointers differ from call to call.  The chain is captured once per (batch size, workspace,
// outputs wanted) and replayed with cudaGraphLaunch after patching the first kernel's `x` and the last
// kernel's `logits` / `labels` (cudaGraphExecKernelNodeSetParams): one driver call instead of eight, and
// no host-side gaps between the kernels of a batch.  A graph instance runs one launch at a time, so
// callers that keep several batches in flight use one workspace (hence one instance) per stream.
constexpr int GRAPH_UNAVAILABLE = -1;
constexpr size_t MAX_GRAPHS = 64;

void drop_graphs(roko_b200_model* m) {
    for (auto* e : m->graphs) {
        if (e->exec) cudaGraphExecDestroy(e->exec);
        if (e->graph) cudaGraphDestroy(e->graph);
        delete e;
    }
    m->graphs.clear();
}

int graph_forward(roko_b200_model* m, const uint8_t* x, int n, float* logits, uint8_t* labels, void* ws, cudaStream_t s) {
    std::lock_guard<std::mutex> lock(m->mu);
    roko_b200_model::GraphEntry* e = nullptr;
    for (auto* c : m->graphs)
        if (c->n == n && c->ws == ws && c->want_logits == (logits != nullptr) && c->want_labels == (labels != nullptr)) { e = c; break; }
    if (!e) {
        if (m->graphs.size() >= MAX_GRAPHS) {                       // evict the least recently used instance
            size_t lru = 0;
            for (size_t i = 1; i < m->graphs.size(); ++i) if (m->graphs[i]->last_use < m->graphs[lru]->last_use) lru = i;
            auto* old = m->graphs[lru];
            cudaGraphExecDestroy(old->exec); cudaGraphDestroy(old->graph); delete old;
            m->graphs.erase(m->graphs.begin() + lru);
        }
        e = new (std::nothrow) roko_b200_model::GraphEntry();
        if (!e) return GRAPH_UNAVAILABLE;
        e->n = n; e->ws = ws; e->want_logits = logits != nullptr; e->want_labels = labels != nullptr;
        bool ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (ok) {
            const int rc = run_forward(m, x, n, logits, labels, ws, (size_t)n * WS_PER_WINDOW * sizeof(float), s, nullptr,
                                       WS_PER_WINDOW * sizeof(float));
            const cudaError_t ce = cudaStreamEndCapture(s, &e->graph);
            ok = rc == ROKO_B200_OK && ce == cudaSuccess && e->graph;
        }
        if (ok) ok = cudaGraphInstantiate(&e->exec, e->graph, 0) == cudaSuccess;
        if (ok) {   // the chain is linear: its root is the front-end kernel, its leaf the head kernel
            size_t nn = 0;
            ok = cudaGraphGetNodes(e->graph, nullptr, &nn) == cudaSuccess && nn >= 2 && nn <= 16;
            cudaGraphNode_t nodes[16];
            if (ok) ok = cudaGraphGetNodes(e->graph, nodes, &nn) == cudaSuccess;
            for (size_t i = 0; ok && i < nn; ++i) {
                size_t ndep = 0, nout = 0;
                cudaGraphNodeType ty;
                ok = cudaGraphNodeGetType(nodes[i], &ty) == cudaSuccess && ty == cudaGraphNodeTypeKernel &&
                     cudaGraphNodeGetDependencies(nodes[i], nullptr, &ndep) == cudaSuccess &&
                     cudaGraphNodeGetDependentNodes(nodes[i], nullptr, &nout) == cudaSuccess;
                if (ok && ndep == 0) e->front = nodes[i];
                if (ok && nout == 0) e->head = nodes[i];
            }
            ok = ok && e->front && e->head && e->front != e->head &&
                 cudaGraphKernelNodeGetParams(e->front, &e->fp) == cudaSuccess &&
                 cudaGraphKernelNodeGetParams(e->head, &e->hp) == cudaSuccess;
            if (ok) {   // front_kernel(x, packed, u, nwin, status); head_kernel(h, w4, b4, logits, labels, rows)
                for (int i = 0; i < 5; ++i) e->fargs[i] = e->fp.kernelParams[i];
                for (int i = 0; i < 6; ++i) e->hargs[i] = e->hp.kernelParams[i];
                e->fargs[0] = &e->x; e->hargs[3] = &e->logits; e->hargs[4] = &e->labels;
                e->fp.kernelParams = e->fargs; e->hp.kernelParams = e->hargs;
            }
        }
        if (!ok) {
            cudaGetLastError();                                     // clear the sticky capture error, fall back for good
            if (e->exec) cudaGraphExecDestroy(e->exec);
            if (e->graph) cudaGraphDestroy(e->graph);
            delete e;
            m->use_graphs = 0;
            return GRAPH_UNAVAILABLE;
        }
        m->graphs.push_back(e);
    }
    e->last_use = ++m->graph_clock;
    e->x = x; e->logits = logits; e->labels = labels;
    CU(cudaGraphExecKernelNodeSetParams(e->exec, e->front, &e->fp));
    CU(cudaGraphExecKernelNodeSetParams(e->exec, e->head, &e->hp));
    CU(cudaGraphLaunch(e->exec, s));
    return ROKO_B200_OK;
}

int check_common(roko_b200_model* m, const void* x, int n, void* ws) {
    if (!m) return fail(ROKO_B200_EARG, "model is NULL%s%s");
    if (!m->loaded) return fail(ROKO_B200_ESTATE, "no weights loaded (call roko_b200_model_load)%s%s");
    if (n < 0) return fail(ROKO_B200_EARG, "n_windows < 0%s%s");
    if (n > 0 && (!x || !ws)) return fail(ROKO_B200_EARG, "x / workspace is NULL%s%s");
    if (((uintptr_t)x & 15) || ((uintptr_t)ws & 15)) return fail(ROKO_B200_EARG, "x / workspace must be 16-byte aligned%s%s");
    return ROKO_B200_OK;
}

int ensure_slots(roko_b200_model* m, int batch) {
    if (m->slot_cap >= batch) return ROKO_B200_OK;
    for (auto& sl : m->slot) {
        if (!sl.stream) CU(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        if (!sl.done) CU(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        cudaFree(sl.x); cudaFree(sl.labels); cudaFree(sl.logits); cudaFree(sl.ws);
        sl.x = nullptr; sl.labels = nullptr; sl.logits = nullptr; sl.ws = nullptr;
        CU(cudaMalloc(&sl.x, (size_t)batch * WIN_BYTES));
        CU(cudaMalloc(&sl.labels, (size_t)batch * COLS));
        CU(cudaMalloc(&sl.logits, (size_t)batch * COLS * CLASSES * sizeof(float)));
        CU(cudaMalloc(&sl.ws, (size_t)batch * WS_WIN_BYTES));
    }
    m->slot_cap = batch;
    return ROKO_B200_OK;
}

}  // namespace

char* roko_b200_errbuf() { return g_err; }

extern "C" {

int roko_b200_abi_version(void) { return ROKO_B200_ABI_VERSION; }
const char* roko_b200_last_error(void) { return g_err; }
int roko_b200_window_reads(void) { return READS; }
int roko_b200_window_cols(void) { return COLS; }
int roko_b200_num_classes(void) { return CLASSES; }
size_t roko_b200_raw_weight_count(void) { return RAW_TOTAL; }

size_t roko_b200_workspace_bytes(int max_windows) {
    return max_windows < 1 ? WS_WIN_BYTES : (size_t)max_windows * WS_WIN_BYTES;
}

int roko_b200_model_create(roko_b200_model** out, int device) {
    if (!out) return fail(ROKO_B200_EARG, "out is NULL%s%s");
    *out = nullptr;
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(ROKO_B200_EARG, "no such CUDA device%s%s");
    DeviceGuard g(device);
    if (!g.ok) return fail(ROKO_B200_ECUDA, "cudaSetDevice failed%s%s");
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(ROKO_B200_ECUDA, "libroko_b200 is built for sm_100a only; device is %s%s", prop.name);
    roko_b200_model* m = new (std::nothrow) roko_b200_model();
    if (!m) return fail(ROKO_B200_EARG, "out of host memory%s%s");
    m->device = device;
    m->num_sms = prop.multiProcessorCount;
    cudaError_t e = cudaMalloc(&m->packed, (size_t)PK_TOTAL * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&m->raw_stage, (size_t)RAW_TOTAL * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&m->raw_al, (size_t)(RAW_TOTAL + RAW_AL_PAD) * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&m->train_img, train_tc_image_floats() * sizeof(float));
    if (e == cudaSuccess) e = train_tc_setup();
    if (e == cudaSuccess) e = gemm_setup();
    if (const char* tt = getenv("ROKO_B200_TRAIN_TC")) m->train_tc = atoi(tt);
    if (e == cudaSuccess) e = cudaMalloc(&m->status, sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(m->status, 0, sizeof(int));
    if (e == cudaSuccess) e = front_setup();
    if (e == cudaSuccess) e = front_tc_setup();
    if (e == cudaSuccess) e = rec_setup();
    if (e == cudaSuccess) e = proj_tc3_setup();
    if (e == cudaSuccess) e = proj_h_setup();
    if (e == cudaSuccess) e = rec_tc_setup();
    if (e == cudaSuccess) e = rec_h_setup();
    if (const char* rt = getenv("ROKO_B200_REC_TC_MIN")) m->rec_tc_min = atoi(rt);
    if (const char* sb = getenv("ROKO_B200_SUPERBATCH")) m->superbatch = atoi(sb) > 0 ? atoi(sb) : 1;
    if (const char* pj = getenv("ROKO_B200_PROJ")) m->use_tc = strcmp(pj, "ffma") == 0 ? 0 : (strcmp(pj, "tf32") == 0 ? 3 : 4);
    if (const char* rk = getenv("ROKO_B200_REC")) m->rec_kind = strcmp(rk, "tf32") == 0 ? 1 : 2;
    if (const char* gr = getenv("ROKO_B200_GRAPHS")) m->use_graphs = atoi(gr);
    if (const char* fr = getenv("ROKO_B200_FRONT")) m->front_kind = strcmp(fr, "tc") == 0 ? 1 : 0;
    if (const char* ge = getenv("ROKO_B200_GEOMETRY")) m->geometry = atoi(ge) != 0;
    if (e != cudaSuccess) {
        roko_b200_model_destroy(m);
        return fail(ROKO_B200_ECUDA, "model_create: %s%s", cudaGetErrorString(e));
    }
    *out = m;
    return ROKO_B200_OK;
}

int roko_b200_model_load(roko_b200_model* m, const float* raw, int raw_on_device, void* stream) {
    if (!m || !raw) return fail(ROKO_B200_EARG, "model / raw is NULL%s%s");
    Range r("roko_b200_model_load");
    DeviceGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool on_device = raw_on_device & 1, no_sync = raw_on_device & 2;
    CU(cudaMemcpyAsync(m->raw_stage, raw, (size_t)RAW_TOTAL * sizeof(float),
                       on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(m->raw_al, m->raw_stage, (size_t)RAW_GRU * sizeof(float), cudaMemcpyDeviceToDevice, s));
    CU(cudaMemcpyAsync(m->raw_al + RAW_GRU + RAW_AL_PAD, m->raw_stage + RAW_GRU,
                       (size_t)(RAW_TOTAL - RAW_GRU) * sizeof(float), cudaMemcpyDeviceToDevice, s));
    CU(launch_pack(m->raw_stage, m->packed, m->status, s));
    // Every kernel reads its weights from `packed` (nothing rides in kernel parameters), so later work on
    // the SAME stream needs no host synchronisation; work on other streams does (bit 1 of raw_on_device unset).
    if (!no_sync) CU(cudaStreamSynchronize(s));
    m->loaded = true;
    return ROKO_B200_OK;
}

int roko_b200_model_destroy(roko_b200_model* m) {
    if (!m) return ROKO_B200_OK;
    DeviceGuard g(m->device);
    for (auto& sl : m->slot) {
        if (sl.stream) { cudaStreamSynchronize(sl.stream); cudaStreamDestroy(sl.stream); }
        if (sl.done) cudaEventDestroy(sl.done);
        cudaFree(sl.x); cudaFree(sl.labels); cudaFree(sl.logits); cudaFree(sl.ws);
    }
    drop_graphs(m);
    cudaFree(m->packed); cudaFree(m->raw_stage); cudaFree(m->raw_al); cudaFree(m->train_img); cudaFree(m->status);
    delete m;
    return ROKO_B200_OK;
}

int roko_b200_forward_u8(roko_b200_model* m, const uint8_t* x, int n_windows, float* logits,
                         uint8_t* labels, void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = check_common(m, x, n_windows, workspace)) return rc;
    if (n_windows == 0) return ROKO_B200_OK;
    Range r("roko_b200_forward_u8");
    DeviceGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t per = WS_PER_WINDOW * sizeof(float);
    if (m->use_graphs && s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread &&
        (size_t)n_windows * per <= workspace_bytes) {
        const int rc = graph_forward(m, x, n_windows, logits, labels, workspace, s);
        if (rc != GRAPH_UNAVAILABLE) return rc;
    }
    return run_forward(m, x, n_windows, logits, labels, workspace, workspace_bytes, s, nullptr, per);
}

int roko_b200_forward_i64(roko_b200_model* m, const int64_t* x, int n_windows, float* logits,
                          uint8_t* labels, void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = check_common(m, x, n_windows, workspace)) return rc;
    if (n_windows == 0) return ROKO_B200_OK;
    DeviceGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long cap_ll = (long long)(workspace_bytes / WS_WIN_BYTES);
    if (cap_ll < 1) return fail(ROKO_B200_EARG, "workspace smaller than one window%s%s");
    const int cap = cap_ll > n_windows ? n_windows : (int)cap_ll;
    // the narrowed copy of a chunk lives behind the fp32 scratch of that chunk
    uint8_t* x8 = static_cast<uint8_t*>(workspace) + (size_t)cap * WS_PER_WINDOW * sizeof(float);
    for (int c0 = 0; c0 < n_windows; c0 += cap) {
        const int nc = (n_windows - c0) < cap ? (n_windows - c0) : cap;
        CU(launch_narrow_i64(reinterpret_cast<const long long*>(x) + (size_t)c0 * WIN_BYTES, x8,
                             (size_t)nc * WIN_BYTES, m->status, s));
        int rc = run_forward(m, x8, nc, logits ? logits + (size_t)c0 * COLS * CLASSES : nullptr,
                             labels ? labels + (size_t)c0 * COLS : nullptr, workspace,
                             (size_t)cap * WS_PER_WINDOW * sizeof(float), s, nullptr,
                             WS_PER_WINDOW * sizeof(float));
        if (rc) return rc;
    }
    return ROKO_B200_OK;
}

int roko_b200_forward_taps(roko_b200_model* m, const uint8_t* x, int n_windows, float* front, float* gru0,
                           float* gru1, float* gru2, float* logits, uint8_t* labels, void* workspace,
                           size_t workspace_bytes, void* stream) {
    if (int rc = check_common(m, x, n_windows, workspace)) return rc;
    if (n_windows == 0) return ROKO_B200_OK;
    DeviceGuard g(m->device);
    Taps t{front, {gru0, gru1, gru2}};
    return run_forward(m, x, n_windows, logits, labels, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream), &t, WS_PER_WINDOW * sizeof(float));
}

int roko_b200_infer_host(roko_b200_model* m, const uint8_t* x_host, long long n_windows, int batch,
                         uint8_t* labels_host, float* logits_host) {
    if (!m) return fail(ROKO_B200_EARG, "model is NULL%s%s");
    if (!m->loaded) return fail(ROKO_B200_ESTATE, "no weights loaded (call roko_b200_model_load)%s%s");
    if (n_windows < 0 || batch < 1) return fail(ROKO_B200_EARG, "bad n_windows / batch%s%s");
    if (n_windows == 0) return ROKO_B200_OK;
    if (!x_host || !labels_host) return fail(ROKO_B200_EARG, "x_host / labels_host is NULL%s%s");
    DeviceGuard g(m->device);
    // Windows are independent, so the caller's batch size is only a lower bound on the granularity:
    // consecutive batches are coalesced into device passes of up to `superbatch` windows (a multiple of
    // the caller's batch), which is what lets the tensor-core recurrence fill the machine.
    long long pass = batch;
    if (m->superbatch > batch) pass = (long long)(m->superbatch / batch) * batch;
    if (pass > n_windows) pass = n_windows;
    if (int rc = ensure_slots(m, (int)pass)) return rc;
    int i = 0;
    for (long long b0 = 0; b0 < n_windows; b0 += pass, ++i) {
        const int nb = (n_windows - b0) < pass ? (int)(n_windows - b0) : (int)pass;
        auto& sl = m->slot[i % NSLOT];
        // stream order already protects the slot's device buffers against the previous use
        CU(cudaMemcpyAsync(sl.x, x_host + (size_t)b0 * WIN_BYTES, (size_t)nb * WIN_BYTES, cudaMemcpyHostToDevice, sl.stream));
        int rc = run_forward(m, sl.x, nb, logits_host ? sl.logits : nullptr, sl.labels, sl.ws,
                             (size_t)m->slot_cap * WS_WIN_BYTES, sl.stream, nullptr, WS_PER_WINDOW * sizeof(float));
        if (rc) return rc;
        CU(cudaMemcpyAsync(labels_host + (size_t)b0 * COLS, sl.labels, (size_t)nb * COLS, cudaMemcpyDeviceToHost, sl.stream));
        if (logits_host)
            CU(cudaMemcpyAsync(logits_host + (size_t)b0 * COLS * CLASSES, sl.logits,
                               (size_t)nb * COLS * CLASSES * sizeof(float), cudaMemcpyDeviceToHost, sl.stream));
    }
    for (auto& sl : m->slot) CU(cudaStreamSynchronize(sl.stream));
    return ROKO_B200_OK;
}

int roko_b200_forward_timed(roko_b200_model* m, const uint8_t* x, int n_windows, uint8_t* labels,
                            void* workspace, size_t workspace_bytes, void* stream, int iters, float* stage_ms) {
    if (int rc = check_common(m, x, n_windows, workspace)) return rc;
    if (n_windows < 1 || iters < 1 || !stage_ms) return fail(ROKO_B200_EARG, "bad n_windows / iters / stage_ms%s%s");
    if ((size_t)n_windows * WS_PER_WINDOW * sizeof(float) > workspace_bytes)
        return fail(ROKO_B200_EARG, "forward_timed needs the whole batch in the workspace%s%s");
    DeviceGuard g(m->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaEvent_t ev[9];
    for (auto& e : ev) CU(cudaEventCreate(&e));
    for (int k = 0; k < 8; ++k) stage_ms[k] = 0.f;
    int rc = ROKO_B200_OK;
    for (int it = 0; it < iters && rc == ROKO_B200_OK; ++it) {
        rc = run_forward(m, x, n_windows, nullptr, labels, workspace, workspace_bytes, s, nullptr,
                         WS_PER_WINDOW * sizeof(float), ev);
        if (rc) break;
        CU(cudaStreamSynchronize(s));
        for (int k = 0; k < 8; ++k) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
            stage_ms[k] += ms / iters;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
}

int roko_b200_measure_fp32_peak(int device, double* tflops) {
    if (!tflops) return fail(ROKO_B200_EARG, "tflops is NULL%s%s");
    DeviceGuard g(device);
    if (!g.ok) return fail(ROKO_B200_ECUDA, "cudaSetDevice failed%s%s");
    double best = 0.0;
    CU(measure_fp32_peak(&best));
    *tflops = best;
    return ROKO_B200_OK;
}

int roko_b200_model_set_option(roko_b200_model* m, const char* name, long long value) {
    if (!m || !name) return fail(ROKO_B200_EARG, "model / name is NULL%s%s");
    {   // captured graphs bake the kernel choice in: start over
        std::lock_guard<std::mutex> lock(m->mu);
        drop_graphs(m);
    }
    if (strcmp(name, "rec_tc_min") == 0) { m->rec_tc_min = (int)value; return ROKO_B200_OK; }
    if (strcmp(name, "superbatch") == 0) { if (value < 1) return fail(ROKO_B200_EARG, "superbatch < 1%s%s"); m->superbatch = (int)value; return ROKO_B200_OK; }
    if (strcmp(name, "proj") == 0) { if (value != 0 && value != 3 && value != 4) return fail(ROKO_B200_EARG, "proj must be 0 (ffma), 3 (tf32) or 4 (fp16)%s%s"); m->use_tc = (int)value; return ROKO_B200_OK; }
    if (strcmp(name, "rec") == 0) { if (value != 1 && value != 2) return fail(ROKO_B200_EARG, "rec must be 1 (tf32) or 2 (fp16)%s%s"); m->rec_kind = (int)value; return ROKO_B200_OK; }
    if (strcmp(name, "graphs") == 0) { m->use_graphs = value != 0; return ROKO_B200_OK; }
    if (strcmp(name, "front") == 0) { if (value != 0 && value != 1) return fail(ROKO_B200_EARG, "front must be 0 (mma.sync) or 1 (tcgen05)%s%s"); m->front_kind = (int)value; return ROKO_B200_OK; }
    if (strcmp(name, "geometry") == 0) { if (value != 0 && value != 1) return fail(ROKO_B200_EARG, "geometry must be 0 (full-chip grids) or 1 (work-sized grids)%s%s"); m->geometry = (int)value; return ROKO_B200_OK; }
    int* geo = strcmp(name, "geo_front") == 0 ? &m->geo_front : strcmp(name, "geo_proj") == 0 ? &m->geo_proj
             : strcmp(name, "geo_head") == 0 ? &m->geo_head : nullptr;
    if (geo) { if (value < 1 || value > (1 << 20)) return fail(ROKO_B200_EARG, "%s must be 1 .. 1048576%s", name); *geo = (int)value; return ROKO_B200_OK; }
    return fail(ROKO_B200_EARG, "unknown option '%s'%s", name);
}

int roko_b200_model_check(roko_b200_model* m) {
    if (!m) return fail(ROKO_B200_EARG, "model is NULL%s%s");
    DeviceGuard g(m->device);
    CU(cudaDeviceSynchronize());
    int st = 0;
    CU(cudaMemcpy(&st, m->status, sizeof(int), cudaMemcpyDeviceToHost));
    if (st) {
        CU(cudaMemset(m->status, 0, sizeof(int)));
        if (st & 1) return fail(ROKO_B200_ECODES, "input code outside 0..11 (index out of range in embedding)%s%s");
        if (st & 2) return fail(ROKO_B200_ERANGE, "a GRU weight is outside the fp16-split range (|w| >= 253): set option proj=3, rec=1 (tf32 kernels)%s%s");
        return fail(ROKO_B200_ERANGE, "an activation left the fp16-split range (|u| >= 4062): set option proj=3 (tf32 kernel)%s%s");
    }
    return ROKO_B200_OK;
}

}  // extern "C"
