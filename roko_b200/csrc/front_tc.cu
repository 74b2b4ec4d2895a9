// Front end of the roko network on tcgen05 (reference roko/rnn_model.py:47-56): embedding gather, read-axis
// fc1 + ReLU, fc2 + ReLU, flatten to the GRU input  u[b][p][10*e + k].  Successor of front.cu, same contract.
//
// front.cu evaluates the exact one-hot factorisation (SURVEY.md App. B.2)
//     M[p][c][j] = sum_{r : x[r][p] == c} W1[j][r]
//     a[p][e][j] = relu(b1[j] + sum_c E[c][e] M[p][c][j])
//     g[p][e][k] = relu(b2[k] + sum_j W2[k][j] a[p][e][j])
// with a SIMT gather for M (7.2 MB of shared-memory reads per window) and warp-level mma.sync for a and g;
// it is bound by shared-memory wavefronts and by the legacy MMA's issue cost, and the two do not overlap.
// Here ALL THREE contractions run on the tensor cores as fp16-split MMAs with fp32 accumulation (tc.cuh):
//   MMA1  D1[j][(p,c)]   = sum_r W1[j][r] . OneHot[(p,c)][r]         M=128 (j), N=96 (8 columns x 12 codes), K=208
//         the gather as a GEMM: the one-hot operand is exact in fp16 (so 2 terms: W1_hi, W1_lo), it is built by 4
//         warps straight from the window bytes (12 x 16-byte stores per 8 reads), W1_hi lives in tensor memory
//   MMA2  D2[(p,e)][j]   = sum_{(p',c)} Eblk[(p,e)][(p',c)] . M[j][(p',c)]      M=128 (2 columns x 64 e), N=112, K=32
//         A = block-diagonal E^T (resident in tensor memory), B = M of two columns, read back from D1 by the thread
//         that owns row j (tcgen05.ld), split to fp16 hi/lo and written as a K-major shared-memory image;
//         b1 rides along as code slot 12 (E row 12 = 1)
//   MMA3  D3[(p,e)][k]   = sum_j a[(p,e)][j] . W2[k][j]                         M=128, N=32|16, K=112
//         A = relu(D2) split to fp16 hi/lo IN PLACE in tensor memory (tcgen05.ld -> registers -> tcgen05.st: the
//         accumulator of MMA2 becomes the A operand of MMA3 without touching shared memory); b2 rides along as
//         column j = 100 (M row 100 is 1 in slot 12, so a[.][100] = 1).  An MMA this small costs ~35 cycles whatever
//         its N, so a_hi multiplies the 32-row image [W2_hi ; W2_lo] in ONE instruction (hi.hi in columns 0..15,
//         hi.lo in 16..31) and a_lo . W2_hi accumulates onto columns 0..15: 14 MMAs per column pair instead of 21
// Roles (21 warps): 0-3 M converters, 4-11 a-stage epilogue (2 warps per TMEM lane quarter), 12-15 g-stage epilogue
// (ReLU + the only global stores), 16-19 one-hot builders (+ the window's TMA bulk copy), 20 MMA issuer.  Every
// hand-over is an mbarrier; TMEM / shared buffers are double buffered so that the tensor pipe always has the next
// MMA batch queued.  The kernel is persistent: one CTA per SM walks windows.
#include "common.cuh"
#include "tc.cuh"

namespace roko {

using namespace tc;

constexpr int FT_THREADS = 21 * 32;
constexpr int FT_GROUPS = 12;                    // 8-column groups per window (the last one holds 2 columns)
constexpr int FT_GP = 4;                         // column pairs per group
constexpr int FT_PAIRS = COLS / 2;               // 45 column pairs per window
constexpr int FT_N1 = 96;                        // MMA1 N: 8 columns x 12 codes (an MMA costs ~40-55 cycles from N = 32 to 96: twice the columns per instruction)
constexpr int FT_N2 = 112;                       // MMA2 N: fc1 width 100 + bias-one row 100, padded to 16
constexpr int FT_KSTEPS1 = FT_K1 / 16;           // 13
// power-of-two operand scales (fp16 range management, undone exactly): W1 x 64, M x 4, E x 4  =>  D2 = 16 a;  W2 x 256  =>  D3 = 4 096 g.
// Headroom: |W1| < 1 000, |M| < 16 000, |E| < 16 000, a < 4 094 (beyond that roko_b200_model_check reports ROKO_B200_ERANGE
// through the NaN / range test of the projection's producers, and `front` 0 -- the fp32-operand round-1 kernel -- serves the model).
constexpr float FT_SW1 = 64.f, FT_SM = 4.f, FT_SE = 4.f;
constexpr float FT_M_RESCALE = FT_SM / FT_SW1;   // D1 = 64 M  ->  M image = 4 M
constexpr float FT_INV3 = 1.f / (FT_SE * FT_SM * 256.f);

// tensor-memory columns (every accumulator starts at a multiple of 16)
constexpr int FT_T_EHI = 0, FT_T_ELO = 16, FT_T_D3 = 32, FT_T_D1 = 64, FT_T_D2 = 160, FT_T_W1 = 384;
static_assert(FT_T_D3 + 32 == FT_T_D1 && FT_T_D1 + FT_N1 == FT_T_D2 && FT_T_D2 + 2 * FT_N2 == FT_T_W1 && FT_T_W1 + FT_K1 / 2 <= 512, "TMEM map");

// shared memory (bytes, from a 1024-aligned base)
constexpr int FT_S_W1LO = 0;                                   // 57 344  [7 atoms][128 rows][64 B]
constexpr int FT_S_OH = FT_S_W1LO + 7 * 128 * 64;              // 2 x 43 008  [7 atoms][96 rows][64 B]
constexpr int FT_OH_BYTES = 7 * FT_N1 * 64;
constexpr int FT_S_MIMG = FT_S_OH + 2 * FT_OH_BYTES;           // 2 x (hi 7 168 + lo 7 168)  [112 rows][64 B]
constexpr int FT_MIMG_BYTES = FT_N2 * 64;
constexpr int FT_S_W2 = FT_S_MIMG + 4 * FT_MIMG_BYTES;         // 8 192  [2 atoms][32 rows: W2_hi 0..15, W2_lo 16..31][128 B]
constexpr int FT_S_XS = FT_S_W2 + 8192;                        // 2 x 18 432 (window bytes, 18 000 used)
constexpr int FT_XS_BYTES = 18432;
constexpr int FT_S_BAR = FT_S_XS + 2 * FT_XS_BYTES;
constexpr int FT_SMEM = FT_S_BAR + 256 + 1024;
static_assert(FT_S_OH % 1024 == 0 && FT_S_MIMG % 512 == 0 && FT_S_W2 % 1024 == 0 && FT_S_XS % 128 == 0, "alignment");
static_assert(FT_SMEM <= 232448, "shared memory budget");

// barrier slots (8 bytes each)
enum { B_XFULL = 0, B_XEMPTY = 2, B_OHFULL = 4, B_OHEMPTY = 6, B_D1FULL = 8, B_D1EMPTY = 10, B_MFULL = 12, B_MEMPTY = 14,
       B_D2FULL = 16, B_AFULL = 18, B_D3FULL = 20, B_D3EMPTY = 22, B_CONST = 24, B_COUNT = 25 };

// K-major SWIZZLE_64B: 64-byte rows, 8-row groups of 512 B, 16-byte chunk c of row r at position c ^ ((r >> 1) & 3)
__device__ __forceinline__ uint64_t desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (32ull << 32) | (1ull << 46) | (4ull << 61);
}
__host__ __device__ constexpr uint32_t sw64_off(uint32_t row, uint32_t chunk) {
    return (row >> 3) * 512u + (row & 7u) * 64u + (((chunk ^ (row >> 1)) & 3u) << 4);
}

#define ROKO_TMEM_ST16(taddr, v)                                                                                      \
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "                                                       \
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"                            \
                 ::"r"(taddr), "r"((v)[0]), "r"((v)[1]), "r"((v)[2]), "r"((v)[3]), "r"((v)[4]), "r"((v)[5]), "r"((v)[6]), \
                   "r"((v)[7]), "r"((v)[8]), "r"((v)[9]), "r"((v)[10]), "r"((v)[11]), "r"((v)[12]), "r"((v)[13]),        \
                   "r"((v)[14]), "r"((v)[15]) : "memory")

// relu(D2) -> fp16 hi / lo words for two adjacent j (D2 is already 16 a: scales 4 x 4)
__device__ __forceinline__ void relu_split2(uint32_t d0, uint32_t d1, uint32_t& hi, uint32_t& lo) {
    relu_split_f16x2(__uint_as_float(d0), __uint_as_float(d1), hi, lo);
}

__global__ void __launch_bounds__(FT_THREADS, 1)
front_tc_kernel(const uint8_t* __restrict__ x, const float* __restrict__ packed, float* __restrict__ u, int nwin,
                int* __restrict__ status) {
    extern __shared__ unsigned char ft_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)ft_smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = smem_u32(smem);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FT_S_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + B_COUNT);
    const uint32_t bar0 = sbase + FT_S_BAR;
    auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr uint32_t WIN_BYTES = READS * COLS;

    if (tid == 0) {
        for (int b = 0; b < 2; ++b) {
            mbar_init(BAR(B_XFULL + b), 1);
            mbar_init(BAR(B_XEMPTY + b), 128);
            mbar_init(BAR(B_OHFULL + b), 128);
            mbar_init(BAR(B_OHEMPTY + b), 1);
            mbar_init(BAR(B_D1FULL + b), 1);
            mbar_init(BAR(B_D1EMPTY + b), 128);
            mbar_init(BAR(B_MFULL + b), 128);
            mbar_init(BAR(B_MEMPTY + b), 1);
            mbar_init(BAR(B_D2FULL + b), 1);
            mbar_init(BAR(B_AFULL + b), 256);
            mbar_init(BAR(B_D3FULL + b), 1);          // (slot 0 only: D3 is single buffered)
            mbar_init(BAR(B_D3EMPTY + b), 128);
        }
        mbar_init(BAR(B_CONST), 1);
        mbar_init_fence();
    }
    if (warp == 20) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // ---- one-time operand residency ---------------------------------------------------------------------------
    if (tid == 640) {                                   // W1_lo and W2 images -> shared memory (bulk copies)
        mbar_expect_tx(BAR(B_CONST), 7 * 128 * 64 + 8192);
        bulk_g2s(sbase + FT_S_W1LO, packed + PK_FT_W1LO, 7 * 128 * 64, BAR(B_CONST));
        bulk_g2s(sbase + FT_S_W2, packed + PK_FT_W2, 8192, BAR(B_CONST));
    }
    if (warp < 4) {                                     // W1_hi (lane = j) and block-diagonal E^T (lane = (pl, e)) -> tensor memory
        const int row = warp * 32 + lane;
        const uint4* src = reinterpret_cast<const uint4*>(packed + PK_FT_W1HI + (size_t)row * (FT_K1 / 2));
#pragma unroll 1
        for (int c0 = 0; c0 < FT_K1 / 2; c0 += 8) {     // 104 words = 13 x 8
            uint32_t v[8];
            const uint4 f0 = __ldg(src + c0 / 4), f1 = __ldg(src + c0 / 4 + 1);
            v[0] = f0.x; v[1] = f0.y; v[2] = f0.z; v[3] = f0.w; v[4] = f1.x; v[5] = f1.y; v[6] = f1.z; v[7] = f1.w;
            ROKO_TMEM_ST8(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(FT_T_W1 + c0), v);
        }
        const int pl = row >> 6, e = row & 63;
        uint32_t eh[16], el[16];
#pragma unroll
        for (int wd = 0; wd < 16; ++wd) {                // word wd: k = 2 wd, 2 wd + 1;  k = 16 p' + c
            float v2[2];
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int k = 2 * wd + t, pp = k >> 4, c = k & 15;
                float val = 0.f;
                if (pp == pl && e < EMB) val = c < NCODES ? FT_SE * __ldg(packed + PK_E + c * EMB + e) : (c == NCODES ? FT_SE : 0.f);
                v2[t] = val;
            }
            split_f16x2(v2[0], v2[1], eh[wd], el[wd]);
        }
        ROKO_TMEM_ST16(tmem + ((uint32_t)(warp * 32) << 16) + FT_T_EHI, eh);
        ROKO_TMEM_ST16(tmem + ((uint32_t)(warp * 32) << 16) + FT_T_ELO, el);
        tmem_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int nmine = (nwin - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;    // windows this CTA processes

    if (warp < 4) {
        // ================================ M converters: D1 -> fp16 hi/lo B operand of MMA2 =====================
        const int j = warp * 32 + lane;                                // row of M == TMEM lane of D1
        const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
        // slot 12 of every column: b1[j] x 4 (row 100: the constant one that turns column 100 of a into 1)
        const float bias = j < FC1 ? FT_SM * __ldg(packed + PK_B1 + j) : (j == FC1 ? FT_SM : 0.f);
        uint32_t bh, bl;
        split_f16x2(bias, 0.f, bh, bl);
        const uint32_t roff[4] = {sw64_off(j, 0), sw64_off(j, 1), sw64_off(j, 2), sw64_off(j, 3)};
        for (int it = 0; it < nmine; ++it) {
#pragma unroll 1
            for (int h = 0; h < FT_GROUPS; ++h) {
                const uint32_t hg = (uint32_t)it * FT_GROUPS + h;
                mbar_wait(BAR(B_D1FULL), hg & 1);                       // D1 is single buffered
                tc_fence_after();
                const int npairs = h < FT_GROUPS - 1 ? FT_GP : 1;
                for (int q = 0; q < npairs; ++q) {
                    const uint32_t gg = (uint32_t)it * FT_PAIRS + FT_GP * h + q, gb = gg & 1;
                    uint32_t v[24];
                    const uint32_t ta = lane_base + FT_T_D1 + q * 24;
                    ROKO_TMEM_LD8(v, ta);
                    ROKO_TMEM_LD8(v + 8, ta + 8);
                    ROKO_TMEM_LD8(v + 16, ta + 16);
                    tmem_wait_ld();
                    if (q == npairs - 1) {                              // the group's last columns are in registers: D1 may be overwritten
                        tc_fence_before();
                        mbar_arrive(BAR(B_D1EMPTY));
                    }
                    uint4 hi[4], lo[4];                                 // chunks: [p0 c0-7] [p0 c8-11, bias, 0] [p1 c0-7] [p1 c8-11, bias, 0]
#pragma unroll
                    for (int pl = 0; pl < 2; ++pl) {
                        const uint32_t* m = v + pl * 12;
                        uint4 &h0 = hi[2 * pl], &l0 = lo[2 * pl], &h1 = hi[2 * pl + 1], &l1 = lo[2 * pl + 1];
                        auto mv = [&](int i) { return __uint_as_float(m[i]) * FT_M_RESCALE; };
                        split_f16x2(mv(0), mv(1), h0.x, l0.x);
                        split_f16x2(mv(2), mv(3), h0.y, l0.y);
                        split_f16x2(mv(4), mv(5), h0.z, l0.z);
                        split_f16x2(mv(6), mv(7), h0.w, l0.w);
                        split_f16x2(mv(8), mv(9), h1.x, l1.x);
                        split_f16x2(mv(10), mv(11), h1.y, l1.y);
                        h1.z = bh; l1.z = bl; h1.w = 0u; l1.w = 0u;
                    }
                    mbar_wait(BAR(B_MEMPTY + gb), ((gg >> 1) & 1) ^ 1);   // MMA2 of pair gg - 2 has consumed this image
                    if (j < FT_N2) {
                        unsigned char* img = smem + FT_S_MIMG + gb * 2 * FT_MIMG_BYTES;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            *reinterpret_cast<uint4*>(img + roff[c]) = hi[c];
                            *reinterpret_cast<uint4*>(img + FT_MIMG_BYTES + roff[c]) = lo[c];
                        }
                    }
                    fence_async_smem();
                    mbar_arrive(BAR(B_MFULL + gb));
                }
            }
        }
    } else if (warp < 12) {
        // ================================ a-stage epilogue: relu(D2) -> fp16 hi/lo A operand of MMA3, in place ==
        const int q = warp & 3, hf = (warp - 4) >> 2;                   // hf 0: j blocks 0, 1;  hf 1: block 2 and the half block 3
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16) + FT_T_D2;
        for (int it = 0; it < nmine; ++it) {
#pragma unroll 1
            for (int g = 0; g < FT_PAIRS; ++g) {
                const uint32_t gg = (uint32_t)it * FT_PAIRS + g, gb = gg & 1;
                mbar_wait(BAR(B_D2FULL + gb), (gg >> 1) & 1);
                tc_fence_after();
                const uint32_t d2 = lane_base + gb * FT_N2;
                // a 32-column block of D2 (j = 32 b .. 32 b + 31) becomes 16 hi words followed by 16 lo words in the same columns
#pragma unroll 1
                for (int blk = 2 * hf; blk < 2 * hf + 1 + (hf ? 0 : 1); ++blk) {
                    uint32_t v[32], lo[16];
                    ROKO_TMEM_LD32(v, d2 + blk * 32);
                    tmem_wait_ld();
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        uint32_t hw;
                        relu_split2(v[2 * i], v[2 * i + 1], hw, lo[i]);
                        v[i] = hw;                                       // v[2i], v[2i+1] are consumed (i <= 2i)
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[16 + i] = lo[i];
                    ROKO_TMEM_ST32(d2 + blk * 32, v);
                }
                if (hf) {                                               // half block: j = 96 .. 111 -> 8 hi + 8 lo words
                    uint32_t v[16], lo[8];
                    ROKO_TMEM_LD16(v, d2 + 96);
                    tmem_wait_ld();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        uint32_t hw;
                        relu_split2(v[2 * i], v[2 * i + 1], hw, lo[i]);
                        v[i] = hw;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[8 + i] = lo[i];
                    ROKO_TMEM_ST16(d2 + 96, v);
                }
                tmem_wait_st();
                tc_fence_before();
                mbar_arrive(BAR(B_AFULL + gb));
            }
        }
    } else if (warp < 16) {
        // ================================ g-stage epilogue: relu(D3) -> u ======================================
        const int q = warp & 3;
        const int L = q * 32 + lane, pl = L >> 6, e = L & 63;
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16) + FT_T_D3;
        for (int it = 0; it < nmine; ++it) {
            const int w = blockIdx.x + it * gridDim.x;
#pragma unroll 1
            for (int g = 0; g < FT_PAIRS; ++g) {
                const uint32_t gg = (uint32_t)it * FT_PAIRS + g;
                mbar_wait(BAR(B_D3FULL), gg & 1);
                tc_fence_after();
                uint32_t v[32];
                ROKO_TMEM_LD32(v, lane_base);
                tmem_wait_ld();
                tc_fence_before();
                mbar_arrive(BAR(B_D3EMPTY));                            // D3 is in registers
#pragma unroll
                for (int i = 0; i < FC2; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(v[16 + i]));   // hi.hi + lo.hi + hi.lo
                float* urow = u + ((size_t)w * COLS + 2 * g + pl) * IN0P;
                if (e < EMB) {
                    float2* dst = reinterpret_cast<float2*>(urow + e * FC2);
#pragma unroll
                    for (int i = 0; i < FC2 / 2; ++i)
                        dst[i] = make_float2(fmaxf(__uint_as_float(v[2 * i]) * FT_INV3, 0.f), fmaxf(__uint_as_float(v[2 * i + 1]) * FT_INV3, 0.f));
                } else if (e < EMB + 3) {                               // zero the k padding of the row (500 .. 511)
                    reinterpret_cast<float4*>(urow + IN0)[e - EMB] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    } else if (warp < 20) {
        // ================================ one-hot builders (+ window TMA) ======================================
        const int t = tid - 16 * 32;                                     // 0 .. 127
        auto fetch_window = [&](int it_) {
            const int w_ = blockIdx.x + it_ * gridDim.x;
            mbar_expect_tx(BAR(B_XFULL + (it_ & 1)), WIN_BYTES);
            bulk_g2s(sbase + FT_S_XS + (it_ & 1) * FT_XS_BYTES, x + (size_t)w_ * WIN_BYTES, WIN_BYTES, BAR(B_XFULL + (it_ & 1)));
        };
        if (t == 0) {
            fetch_window(0);
            if (nmine > 1) fetch_window(1);
        }
        bool bad = false;
        // tasks of a group: (column pl of 8, read chunk rc of 26) = 208; thread t takes tasks t and t + 128
        for (int it = 0; it < nmine; ++it) {
            mbar_wait(BAR(B_XFULL + (it & 1)), (it >> 1) & 1);
            const unsigned char* xs = smem + FT_S_XS + (it & 1) * FT_XS_BYTES;
#pragma unroll 1
            for (int h = 0; h < FT_GROUPS; ++h) {
                const uint32_t hg = (uint32_t)it * FT_GROUPS + h, hb = hg & 1;
                uint32_t c03[2], c47[2];                                 // my 8 codes per task, one per byte (0xFF = no read)
                bool live[2];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int task = t + 128 * k, pl = task / 26, rc = task % 26, p = 8 * h + pl;
                    live[k] = task < 208 && p < COLS;
                    c03[k] = c47[k] = 0xFFFFFFFFu;
                    if (live[k]) {
                        uint32_t code[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int r = 8 * rc + i;
                            code[i] = r < READS ? xs[r * COLS + p] : 255u;
                            bad |= (r < READS && code[i] >= NCODES);
                        }
                        c03[k] = code[0] | (code[1] << 8) | (code[2] << 16) | (code[3] << 24);
                        c47[k] = code[4] | (code[5] << 8) | (code[6] << 16) | (code[7] << 24);
                    }
                }
                mbar_wait(BAR(B_OHEMPTY + hb), ((hg >> 1) & 1) ^ 1);     // MMA1 of group hg - 2 has consumed this buffer
                unsigned char* oh = smem + FT_S_OH + hb * FT_OH_BYTES;
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    if (!live[k]) continue;
                    const int task = t + 128 * k, pl = task / 26, rc = task % 26;
                    // my 16-byte chunk of row n = pl * 12 + c: k atom rc >> 2, chunk rc & 3
                    unsigned char* base = oh + (uint32_t)(rc >> 2) * (FT_N1 * 64);
#pragma unroll
                    for (int c = 0; c < NCODES; ++c) {
                        // byte-wise compare (0xFF where the read carries code c), bytes spread to the high byte of each half,
                        // masked to fp16 1.0 = 0x3C00
                        const uint32_t m0 = __vcmpeq4(c03[k], 0x01010101u * (uint32_t)c), m1 = __vcmpeq4(c47[k], 0x01010101u * (uint32_t)c);
                        uint4 o;
                        o.x = __byte_perm(m0, 0u, 0x1404) & 0x3C003C00u;
                        o.y = __byte_perm(m0, 0u, 0x3424) & 0x3C003C00u;
                        o.z = __byte_perm(m1, 0u, 0x1404) & 0x3C003C00u;
                        o.w = __byte_perm(m1, 0u, 0x3424) & 0x3C003C00u;
                        *reinterpret_cast<uint4*>(base + sw64_off((uint32_t)(pl * NCODES + c), (uint32_t)(rc & 3))) = o;
                    }
                }
                fence_async_smem();
                mbar_arrive(BAR(B_OHFULL + hb));
            }
            mbar_arrive(BAR(B_XEMPTY + (it & 1)));                       // this window's bytes are no longer needed
            if (t == 0 && it + 2 < nmine) {
                mbar_wait(BAR(B_XEMPTY + (it & 1)), (it >> 1) & 1);
                fetch_window(it + 2);
            }
        }
        if (bad) atomicOr(status, 1);                                    // nn.Embedding would raise IndexError (CPU) / assert (CUDA)
    } else {
        // ================================ MMA issuer (whole warp, uniform) =====================================
        if (tmem != 0) __trap();                                         // all 512 columns are ours -> base 0: literal TMEM addresses
        const uint32_t elected = elect_one();
        mbar_wait(BAR(B_CONST), 0);                                      // W1_lo and W2 images have landed
        constexpr uint32_t ID1 = idesc_f16(128, FT_N1), ID2 = idesc_f16(128, FT_N2), ID3 = idesc_f16(128, 32), ID3L = idesc_f16(128, 16);
        auto mma1 = [&](uint32_t hg) {                                   // D1 = W1 . OneHot(group hg)
            const uint32_t hb = hg & 1;
            mbar_wait(BAR(B_OHFULL + hb), (hg >> 1) & 1);
            mbar_wait(BAR(B_D1EMPTY), (hg & 1) ^ 1);                     // the M converters hold the previous group's columns in registers
            tc_fence_after();
            const uint32_t d = FT_T_D1, oh = sbase + FT_S_OH + hb * FT_OH_BYTES, wl = sbase + FT_S_W1LO;
#pragma unroll
            for (int kk = 0; kk < FT_KSTEPS1; ++kk) {
                const uint64_t db = desc_sw64(oh + (kk >> 1) * (FT_N1 * 64) + (kk & 1) * 32);
                mma_f16_ss(d, desc_sw64(wl + (kk >> 1) * (128 * 64) + (kk & 1) * 32), db, ID1, kk ? 1u : 0u, elected);   // W1_lo
                mma_f16_ts(d, FT_T_W1 + kk * 8, db, ID1, 1u, elected);                                                    // W1_hi
            }
            mma_commit(BAR(B_D1FULL), elected);
            mma_commit(BAR(B_OHEMPTY + hb), elected);
            __syncwarp();
        };
        auto mma2 = [&](uint32_t gg) {                                   // D2[gb] = Eblk . M(pair gg)
            const uint32_t gb = gg & 1;
            mbar_wait(BAR(B_MFULL + gb), (gg >> 1) & 1);
            tc_fence_after();
            const uint32_t d = FT_T_D2 + gb * FT_N2, mh = sbase + FT_S_MIMG + gb * 2 * FT_MIMG_BYTES, ml = mh + FT_MIMG_BYTES;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const uint64_t dh = desc_sw64(mh + kk * 32), dl = desc_sw64(ml + kk * 32);
                mma_f16_ts(d, FT_T_ELO + kk * 8, dh, ID2, kk ? 1u : 0u, elected);    // E_lo M_hi   (small terms first)
                mma_f16_ts(d, FT_T_EHI + kk * 8, dl, ID2, 1u, elected);              // E_hi M_lo
                mma_f16_ts(d, FT_T_EHI + kk * 8, dh, ID2, 1u, elected);              // E_hi M_hi
            }
            mma_commit(BAR(B_D2FULL + gb), elected);
            mma_commit(BAR(B_MEMPTY + gb), elected);
            __syncwarp();
        };
        auto mma3 = [&](uint32_t gg) {                                   // D3 = a(pair gg) . [W2_hi ; W2_lo]^T
            const uint32_t gb = gg & 1;
            mbar_wait(BAR(B_AFULL + gb), (gg >> 1) & 1);
            mbar_wait(BAR(B_D3EMPTY), (gg & 1) ^ 1);
            tc_fence_after();
            const uint32_t d = FT_T_D3, a0 = FT_T_D2 + gb * FT_N2, w2 = sbase + FT_S_W2;
#pragma unroll
            for (int kk = 0; kk < FT_N2 / 16; ++kk) {                    // j = 16 kk .. 16 kk + 15: block kk >> 1 of the in-place a image
                const uint32_t ahi = a0 + (kk < 6 ? 32 * (kk >> 1) + 8 * (kk & 1) : 96), alo = ahi + (kk < 6 ? 16 : 8);
                const uint64_t dw = desc_sw128(w2 + (uint32_t)(kk >> 2) * (32 * 128) + (uint32_t)(kk & 3) * 32);
                mma_f16_ts(d, ahi, dw, ID3, kk ? 1u : 0u, elected);      // a_hi . [W2_hi ; W2_lo]   (32 columns)
                mma_f16_ts(d, alo, dw, ID3L, 1u, elected);               // a_lo . W2_hi            (columns 0..15)
            }
            mma_commit(BAR(B_D3FULL), elected);
            __syncwarp();
        };
        for (int it = 0; it < nmine; ++it) {
            const uint32_t h0 = (uint32_t)it * FT_GROUPS, g0 = (uint32_t)it * FT_PAIRS;
            mma1(h0);
#pragma unroll 1
            for (int h = 0; h < FT_GROUPS; ++h) {
                const int npairs = h < FT_GROUPS - 1 ? FT_GP : 1;
                for (int q = 0; q < npairs; ++q) {
                    const uint32_t gg = g0 + FT_GP * h + q;
                    mma2(gg);
                    if (FT_GP * h + q > 0) mma3(gg - 1);                 // a of the previous pair has been split meanwhile
                    // D1 is single buffered: the next group's gather is issued once this group's second pair is under way -- by
                    // then the converters have read (or are about to read) the group's last columns out of D1
                    if (q == 1 && h + 1 < FT_GROUPS) mma1(h0 + h + 1);
                }
            }
            mma3(g0 + FT_PAIRS - 1);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 20) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

cudaError_t front_tc_setup() {
    return cudaFuncSetAttribute(front_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM);
}

cudaError_t launch_front_tc(const uint8_t* x, const float* packed, float* u, int nwin, int* status, int max_ctas,
                            cudaStream_t s) {
    if (nwin <= 0) return cudaSuccess;
    if (max_ctas < 1) return cudaErrorInvalidValue;
    const int grid = nwin < max_ctas ? nwin : max_ctas;
    front_tc_kernel<<<grid, FT_THREADS, FT_SMEM, s>>>(x, packed, u, nwin, status);
    return cudaGetLastError();
}

}  // namespace roko
