// Private definition of the opaque roko_b200_model handle (include/roko_b200.h), shared by api.cu
// and train_api.cu.
#pragma once
#include <mutex>
#include <vector>

#include "common.cuh"
#include "tc.cuh"

constexpr int NSLOT = 3;
// launch geometry of the inference chain (launch_cap): least work per CTA of front_tc (windows), proj_h (128x256 tiles) and head (rows)
constexpr int GEO_FRONT_DEFAULT = 4, GEO_PROJ_DEFAULT = 6, GEO_HEAD_DEFAULT = 128;
constexpr int ROKO_ERRBUF = 512;
char* roko_b200_errbuf();         // the calling thread's roko_b200_last_error() buffer (api.cu)

struct roko_b200_model {
    int device = 0;
    int num_sms = 148;
    float* packed = nullptr;
    float* raw_stage = nullptr;     // device copy of the raw (state_dict order) weights; the training backward reads them
    float* raw_al = nullptr;        // the same with 2 floats of padding before the GRU section: every tensor 16-byte aligned
    float* train_img = nullptr;     // tf32 hi / lo images of fc1.weight for the tcgen05 training products (train_tc.cu)
    static constexpr int TRAIN_TC_DEFAULT = 6;
    int train_tc = TRAIN_TC_DEFAULT; // ROKO_B200_TRAIN_TC: which training products run on tcgen05 (train_tc.cu) instead of the
                                    // generic GEMM: >= 1 fc1 and d(ep), >= 2 dW1, >= 3 the GRU d(in), 4 dW_ih / dW_hh (a launch
                                    // per product), >= 5 the masked embedding is rebuilt in the consumers' producer warps, never
                                    // stored, >= 6 dW_ih / dW_hh as one tile-list launch per layer (default)
    int* status = nullptr;          // device flag word, bit 0: code outside 0..11
    bool loaded = false;
    int use_tc = 4;                 // projection: 4 = tcgen05, fp16-split operands (proj_h.cu, default); 3 = tcgen05 3xTF32
                                    // (proj_tc3.cu); 0 = FFMA SGEMM (proj.cu, the fp32-exact A/B reference).  ROKO_B200_PROJ=fp16|tf32|ffma
    int rec_kind = 2;               // tensor-core recurrence: 2 = fp16-split, W_hh resident in tensor memory (rec_h.cu, default);
                                    // 1 = 3xTF32 (rec_tc.cu).  ROKO_B200_REC=fp16|tf32
    int superbatch = 2368;          // windows per device pass of infer_host (148 SMs x 16; ROKO_B200_SUPERBATCH)
    int rec_tc_min = 64;            // chunks of at least this many windows use the tcgen05 recurrence (ROKO_B200_REC_TC_MIN; 0 = never);
                                    // smaller ones the register-resident FFMA recurrence (rec.cu), which spreads few windows over many SMs
    struct Slot {
        cudaStream_t stream = nullptr;
        cudaEvent_t done = nullptr;
        uint8_t* x = nullptr;
        uint8_t* labels = nullptr;
        float* logits = nullptr;
        void* ws = nullptr;
    } slot[NSLOT];
    int slot_cap = 0;
    // CUDA-graph instances of the forward chain (api.cu: graph_forward)
    struct GraphEntry {
        int n = 0;
        const void* ws = nullptr;
        bool want_logits = false, want_labels = false;
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        cudaGraphNode_t front = nullptr, head = nullptr;
        cudaKernelNodeParams fp{}, hp{};
        void* fargs[5] = {};
        void* hargs[6] = {};
        const uint8_t* x = nullptr;       // the per-launch values the patched parameters point at
        float* logits = nullptr;
        uint8_t* labels = nullptr;
        unsigned long long last_use = 0;
    };
    std::vector<GraphEntry*> graphs;
    std::mutex mu;
    unsigned long long graph_clock = 0;
    int use_graphs = 1;             // replay the chain as a CUDA graph when the batch fits the workspace (ROKO_B200_GRAPHS=0 disables)
    int front_kind = 1;             // front end: 1 = all three contractions on tcgen05 (front_tc.cu, default); 0 = SIMT gather + warp-level
                                    // mma.sync stages (front.cu, round 1).  ROKO_B200_FRONT=tc|mma
    int geometry = 1;               // grids of front_tc / proj_h / head in the inference chain (launch_cap): 1 = at least geo_* units of
                                    // work per CTA, 0 = one CTA per unit up to the full chip.  ROKO_B200_GEOMETRY=0|1
    int geo_front = GEO_FRONT_DEFAULT;  // windows per front_tc CTA at least
    int geo_proj = GEO_PROJ_DEFAULT;    // 128x256 tiles per proj_h CTA at least
    int geo_head = GEO_HEAD_DEFAULT;    // rows per head block at least
};

// offset of raw element `off` inside raw_al (RAW_GRU is 2 mod 4 and every later tensor size is a multiple of 4)
constexpr int RAW_AL_PAD = 2;
static_assert((roko::RAW_GRU + RAW_AL_PAD) % 4 == 0 && roko::RAW_W1 % 4 == 0 && roko::RAW_W2 % 4 == 0, "raw_al alignment");
__host__ __device__ constexpr int raw_al_off(int off) { return off >= roko::RAW_GRU ? off + RAW_AL_PAD : off; }

// Grid of a launch over `units` of work with CTA limit `full`.  Geometry 1 gives each CTA at least `min_per_cta` units: every
// CTA pays its prologue (tensor-memory images, barrier set-up, pipeline fill and drain) once per launch, so a 128-window batch
// on 148 CTAs spends a large share of its SM-time there, while with several batches in flight on other streams the SMs a smaller grid
// leaves free run their kernels.  Batches large enough for `full` CTAs at `min_per_cta` get `full` either way.  The kernels
// stride their work by gridDim.x, so the grid changes no result.
inline int launch_cap(const roko_b200_model* m, long long units, int min_per_cta, int full) {
    if (!m->geometry) return full;
    const long long ctas = (units + min_per_cta - 1) / min_per_cta;
    return ctas < 1 ? 1 : (ctas < full ? (int)ctas : full);
}

// Input projection of GRU layer `l` with the kernel the model is configured for (see use_tc); proj_ctas caps the grid of the
// fp16-split kernel (the tf32 and FFMA kernels keep their own).
inline cudaError_t proj_dispatch(const roko_b200_model* m, const float* in, int l, float* gi, int rows, int proj_ctas,
                                 cudaStream_t s) {
    using namespace roko;
    const float* pk = m->packed;
    if (m->use_tc == 4)
        return launch_proj_h(in, gru_inp(l), pk + pk_wh16(l), pk + pk_bgi(l), gi, rows, l == 0 ? tc::U_SCALE : tc::H_SCALE,
                             m->status, proj_ctas, s);
    if (m->use_tc == 3) return launch_proj_tc3(in, gru_inp(l), pk + pk_wtc(l), pk + pk_bgi(l), gi, rows, m->num_sms, s);
    return launch_proj(in, gru_inp(l), pk + pk_wih(l), pk + pk_bgi(l), gi, rows, s);
}

// Recurrence of GRU layer `l` over `nc` windows (both directions): tensor cores from rec_tc_min windows on.
inline cudaError_t rec_dispatch(const roko_b200_model* m, const float* gi, int l, float* out, int nc, cudaStream_t s) {
    using namespace roko;
    const float* pk = m->packed;
    if (m->rec_tc_min > 0 && nc >= m->rec_tc_min) {
        if (m->rec_kind == 2) return launch_rec_h(gi, pk + pk_rh16(l, 0), out, nc, m->num_sms, s);
        if (nc >= 64)       // (>= 64 windows keeps rec_tc's unguarded gi reads of a ragged last group inside the scratch)
            return launch_rec_tc(gi, pk + pk_rtc(l, 0), pk + pk_rtc(l, 0) + RTC_W, (size_t)RTC_DIR, pk + pk_rtc(l, 0) + 2 * RTC_W,
                                 out, nc, m->num_sms, s);
    }
    return launch_rec(gi, pk + pk_whh(l, 0), (size_t)(pk_whh(0, 1) - pk_whh(0, 0)), pk + pk_bhn(l, 0), out, nc, m->num_sms, s);
}
