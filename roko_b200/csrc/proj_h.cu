// GRU input projection on tcgen05 with fp16-split operands (reference op: the gi half of nn.GRU,
// roko/rnn_model.py:57):  gi[M x 768] = A[M x K] . W_ih^T + b   for both directions of a layer.
// Same persistent organisation as proj_tc3.cu (its 3xTF32 predecessor, kept for A/B): one CTA per SM loops
// over 128 x 256 output tiles, the 512 TMEM columns hold two fp32 accumulators so the epilogue of tile i
// overlaps the MMAs of tile i+1, 2-stage mbarrier pipeline, warp roles 0-7 A producers / 8 TMA W loader /
// 9 MMA issuer / 10-13 epilogue, epilogue staged through shared memory for whole-row-segment stores.
// What changes with the fp16 split (tc.cuh): a 96 KB stage now covers K = 64 instead of 32 (half the operand
// bytes per product) and a k block is 12 kind::f16 MMAs of K = 16 -- half the tensor time of the tf32 form
// at the same 2^-22 accuracy.  The A producers scale by a power of two (in_scale), split fp32 -> fp16 hi/lo
// and write the K-major SWIZZLE_128B images; W_ih images (x 256) come pre-split from pack.cu by bulk copy;
// the epilogue undoes both scales exactly.
#include <stdlib.h>

#include "common.cuh"
#include "tc.cuh"

namespace roko {

using namespace tc;

constexpr int PH_THREADS = 14 * 32;                      // warps 0-7 A producers, 8 W loader, 9 MMA issuer (+TMEM alloc), 10-13 epilogue
constexpr int PH_STAGES = 2;
constexpr int PH_A_IMG = TC_BM * H16_BK * 2;            // 16 KB: 128 rows x 64 fp16
constexpr int PH_W_IMG = TC_BN * H16_BK * 2;            // 32 KB
constexpr int PH_STAGE = 2 * PH_A_IMG + 2 * PH_W_IMG;   // 96 KB
constexpr int PH_EPI_ROW = 36;                          // floats per staged row (144 B: 16-byte aligned, conflict free both ways)
constexpr int PH_EPI_BYTES = 4 * 32 * PH_EPI_ROW * 4;   // one 32 x 32 staging tile per epilogue warp
constexpr int PH_SMEM = PH_STAGES * PH_STAGE + 1024 + 256 + PH_EPI_BYTES;
constexpr int PH_TMEM_COLS = 512;
constexpr uint32_t PH_IDESC = idesc_f16(TC_BM, TC_BN);

// A producers: 256 threads turn fp32 activation rows into the fp16 hi / lo K-major swizzled
// images of one k block (128 rows x 64 k) per pipeline stage.  thread = (16-byte chunk of 8 fp16 = 8 consecutive k, rows rr + 32 i).
// TWO k blocks of loads are in flight per thread: with one, the loop was bound by the latency of its own loads (3.9 k cycles per
// k block against 1.5 k of MMA work: ncu `long_scoreboard` 7 warps per issue, L2 -> SM path at 60 %).
//   row0_of(j)   first row of the j-th tile of this CTA        arrive(s)  "images of stage s are written"
template <int K, int NSTAGE, typename RowOf, typename Arrive>
__device__ __forceinline__ void produce_a(const float* __restrict__ A, int M, int ntiles_mine, RowOf row0_of, unsigned char* stages,
                                          int stage_bytes, uint32_t empty_bar0, float in_scale, int* status, Arrive arrive, int ptid) {
    constexpr int KB = K / H16_BK;
    const int chunk = ptid & 7, rr = ptid >> 3;                            // rr 0..31
    const int nkb = ntiles_mine * KB;
    auto src_of = [&](int it, int i) -> const float4* {
        const int r = row0_of(it / KB) + rr + 32 * i;
        return r < M ? reinterpret_cast<const float4*>(A + (size_t)r * K + (it % KB) * H16_BK + chunk * 8) : nullptr;
    };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    bool overflow = false;
    float4 v[2][4][2];
#pragma unroll
    for (int d = 0; d < 2; ++d)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4* p = d < nkb ? src_of(d, i) : nullptr;
            v[d][i][0] = p ? __ldg(p) : zero4;
            v[d][i][1] = p ? __ldg(p + 1) : zero4;
        }
#pragma unroll 1
    for (int it = 0; it < nkb; it += 2) {
#pragma unroll
        for (int d = 0; d < 2; ++d) {
            const int cur = it + d;
            if (cur < nkb) {
                const int s = cur % NSTAGE;
                mbar_wait(empty_bar0 + 8u * s, ((cur / NSTAGE) & 1) ^ 1);
                unsigned char* ahi = stages + s * stage_bytes;
                unsigned char* alo = ahi + PH_A_IMG;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = rr + 32 * i;
                    const int off = (r >> 3) * 1024 + (r & 7) * 128 + ((chunk ^ (r & 7)) << 4);
                    const float4 a = v[d][i][0], b = v[d][i][1];
                    const float mx = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))),
                                           fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w))));
                    overflow |= !(mx * in_scale <= 65000.f);               // also catches NaN
                    uint4 h, l;
                    split_f16x2(a.x * in_scale, a.y * in_scale, h.x, l.x);
                    split_f16x2(a.z * in_scale, a.w * in_scale, h.y, l.y);
                    split_f16x2(b.x * in_scale, b.y * in_scale, h.z, l.z);
                    split_f16x2(b.z * in_scale, b.w * in_scale, h.w, l.w);
                    *reinterpret_cast<uint4*>(ahi + off) = h;
                    *reinterpret_cast<uint4*>(alo + off) = l;
                }
                fence_async_smem();
                arrive(s);
#pragma unroll
                for (int i = 0; i < 4; ++i) {                              // refill this slot with k block cur + 2
                    const float4* p = cur + 2 < nkb ? src_of(cur + 2, i) : nullptr;
                    v[d][i][0] = p ? __ldg(p) : zero4;
                    v[d][i][1] = p ? __ldg(p + 1) : zero4;
                }
            }
        }
    }
    if (overflow) atomicOr(status, 4);                                     // activation outside the fp16-split range (roko_b200_model_check)
}


template <int K>
__global__ void __launch_bounds__(PH_THREADS, 1)
proj_h_kernel(const float* __restrict__ A, const float* __restrict__ wimg, const float* __restrict__ bias,
              float* __restrict__ C, int M, int ntiles, float in_scale, int* __restrict__ status) {
    constexpr int KB = K / H16_BK;
    extern __shared__ unsigned char ph_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)ph_smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PH_STAGES * PH_STAGE);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
    float* epi_stage = reinterpret_cast<float*>(smem + PH_STAGES * PH_STAGE + 256);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar0 = smem_u32(bars);
    // barriers: full_a[s] = s, full_w[s] = 2+s, empty[s] = 4+s, acc_full[b] = 6+b, acc_empty[b] = 8+b
    auto BAR = [&](int i) { return bar0 + 8u * i; };

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int s = 0; s < PH_STAGES; ++s) {
            mbar_init(BAR(s), 256);
            mbar_init(BAR(2 + s), 1);
            mbar_init(BAR(4 + s), 1);
            mbar_init(BAR(6 + s), 1);
            mbar_init(BAR(8 + s), 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 9) {
        tmem_alloc<PH_TMEM_COLS>(tmem_slot);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    if (warp < 8) {
        // ------------------------------- A producers (produce_a above) -----------------------------
        const int mine = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
        produce_a<K, PH_STAGES>(A, M, mine, [&](int j) { return ((int)(blockIdx.x + j * gridDim.x) / 3) * TC_BM; }, smem, PH_STAGE,
                                BAR(4), in_scale, status, [&](int s_) { mbar_arrive(BAR(s_)); }, tid);
    } else if (warp == 8) {
        // ------------------------------- W loader (TMA bulk copies) --------------------------------
        if (lane == 0) {
            int it = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const float* src = wimg + (size_t)(tile % 3) * KB * 2 * H16_IMG;
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int s = it & 1;
                    mbar_wait(BAR(4 + s), ((it >> 1) & 1) ^ 1);
                    mbar_expect_tx(BAR(2 + s), 2 * PH_W_IMG);
                    bulk_g2s(sbase + s * PH_STAGE + 2 * PH_A_IMG, src + (size_t)kb * 2 * H16_IMG, 2 * PH_W_IMG, BAR(2 + s));
                }
            }
        }
    } else if (warp == 9) {
        // ------------------------------- MMA issuer (whole warp, uniform) ---------------------------
        if (tmem_d != 0) __trap();                                 // all 512 columns are ours -> base 0
        const uint32_t elected = elect_one();
        int it = 0, j = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++j) {
            const uint32_t buf = j & 1;
            mbar_wait(BAR(8 + buf), ((j >> 1) & 1) ^ 1);        // epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t d = buf * TC_BN;
            for (int kb = 0; kb < KB; ++kb, ++it) {
                const int s = it & 1;
                const uint32_t ph = (it >> 1) & 1;
                mbar_wait(BAR(s), ph);
                mbar_wait(BAR(2 + s), ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_hi = sbase + s * PH_STAGE, a_lo = a_hi + PH_A_IMG;
                const uint32_t w_hi = a_lo + PH_A_IMG, w_lo = w_hi + PH_W_IMG;
#pragma unroll
                for (int kk = 0; kk < H16_BK / 16; ++kk) {
                    const uint64_t dah = desc_sw128(a_hi + kk * 32), dal = desc_sw128(a_lo + kk * 32);
                    const uint64_t dwh = desc_sw128(w_hi + kk * 32), dwl = desc_sw128(w_lo + kk * 32);
                    mma_f16_ss(d, dal, dwh, PH_IDESC, (kb | kk) ? 1u : 0u, elected);   // small terms first
                    mma_f16_ss(d, dah, dwl, PH_IDESC, 1u, elected);
                    mma_f16_ss(d, dah, dwh, PH_IDESC, 1u, elected);
                }
                mma_commit(BAR(4 + s), elected);
                __syncwarp();
            }
            mma_commit(BAR(6 + buf), elected);                     // accumulator complete
            __syncwarp();
        }
    } else {
        // ------------------------------- epilogue warps (10..13; TMEM lane quarter = warp & 3) ------
        const int q = warp & 3;                                    // TMEM lane quarter this warp may read
        const float inv = 1.f / (W_SCALE * in_scale);              // exact: both scales are powers of two
        int j = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++j) {
            const uint32_t buf = j & 1;
            const int m0 = (tile / 3) * TC_BM, n_tile = tile % 3;
            mbar_wait(BAR(6 + buf), (j >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // TMEM lane == tile row: this thread owns row q*32 + lane.  Rows are staged through a 32 x 32
            // shared tile so that every global store instruction writes four whole 128-byte row segments
            // (storing straight from the TMEM layout puts the 32 lanes of an instruction on 32 different rows,
            // 16 bytes each: the epilogue then takes longer than the K=256 main loop it should hide behind).
            const uint32_t taddr = ((uint32_t)(q * 32) << 16) + buf * TC_BN;
            float* T = epi_stage + (warp - 10) * 32 * PH_EPI_ROW;
            const float* brow = bias + n_tile * TC_BN;
            const int rsub = lane >> 3, csub = (lane & 7) * 4;      // read-back role: 4 rows x 8 float4 per instruction
#pragma unroll 1
            for (int c0 = 0; c0 < TC_BN; c0 += 32) {
                uint32_t r[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                      "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr + (uint32_t)c0));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int qq = 0; qq < 8; ++qq)                       // my row, 32 columns -> staging tile (row-wise STS.128)
                    *reinterpret_cast<float4*>(T + lane * PH_EPI_ROW + qq * 4) =
                        make_float4(__uint_as_float(r[qq * 4 + 0]), __uint_as_float(r[qq * 4 + 1]),
                                    __uint_as_float(r[qq * 4 + 2]), __uint_as_float(r[qq * 4 + 3]));
                __syncwarp();
                const float4 b = __ldg(reinterpret_cast<const float4*>(brow + c0 + csub));
#pragma unroll
                for (int it = 0; it < 8; ++it) {                     // rows 4*it .. 4*it+3, all 32 columns, coalesced
                    const int rr = it * 4 + rsub;
                    const int m = m0 + q * 32 + rr;
                    float4 v = *reinterpret_cast<const float4*>(T + rr * PH_EPI_ROW + csub);
                    v.x = fmaf(v.x, inv, b.x); v.y = fmaf(v.y, inv, b.y); v.z = fmaf(v.z, inv, b.z); v.w = fmaf(v.w, inv, b.w);
                    if (m < M) *reinterpret_cast<float4*>(C + (size_t)m * GI_N + n_tile * TC_BN + c0 + csub) = v;
                }
                __syncwarp();
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(BAR(8 + buf));                          // accumulator may be overwritten
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 9) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem_dealloc<PH_TMEM_COLS>(tmem_d);
    }
}



cudaError_t proj_h_setup() {
    cudaError_t e = cudaFuncSetAttribute(proj_h_kernel<IN0P>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(proj_h_kernel<OUT_W>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM);
}

cudaError_t launch_proj_h(const float* A, int K, const float* wimg, const float* bias, float* C, int M, float in_scale,
                          int* status, int max_ctas, cudaStream_t s) {
    if (M <= 0) return cudaSuccess;
    if (max_ctas < 1) return cudaErrorInvalidValue;
    const int ntiles = ((M + TC_BM - 1) / TC_BM) * (GI_N / TC_BN);
    const int grid = ntiles < max_ctas ? ntiles : max_ctas;
    if (K == IN0P) proj_h_kernel<IN0P><<<grid, PH_THREADS, PH_SMEM, s>>>(A, wimg, bias, C, M, ntiles, in_scale, status);
    else if (K == OUT_W) proj_h_kernel<OUT_W><<<grid, PH_THREADS, PH_SMEM, s>>>(A, wimg, bias, C, M, ntiles, in_scale, status);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

}  // namespace roko
