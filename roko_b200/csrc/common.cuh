// Shared constants, packed-weight layout and small device helpers for the roko hot path.
//
// Geometry follows the reference: a window is 200 sampled reads x 90 pileup columns of uint8
// codes 0..11 (reference include/generate.h:19, generate.cpp:18-25,145); the network is
// roko/rnn_model.py:24-59 (embedding 12x50, fc1 200->100 over the READ axis, fc2 100->10,
// 3-layer bidirectional GRU hidden 128, fc4 256->5).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace roko {

constexpr int READS = 200;     // generate.h:19
constexpr int COLS = 90;       // generate.h:19  (GRU time axis, rnn_model.py:56)
constexpr int NCODES = 12;     // rnn_model.py:28
constexpr int EMB = 50;        // rnn_model.py:28
constexpr int FC1 = 100;       // rnn_model.py:31
constexpr int FC2 = 10;        // rnn_model.py:34
constexpr int IN0 = 500;       // rnn_model.py:10
constexpr int IN0P = 512;      // IN0 padded to a multiple of the GEMM k-tile (pad columns are zero)
constexpr int HID = 128;       // rnn_model.py:11
constexpr int G3 = 3 * HID;    // gate rows per direction, reference order [r; z; n]
constexpr int GI_N = 2 * G3;   // both directions
constexpr int LAYERS = 3;      // rnn_model.py:12
constexpr int OUT_W = 2 * HID; // [fwd ; bwd]
constexpr int CLASSES = 5;     // rnn_model.py:44

// ---- raw weights: the 31 state_dict tensors of the reference module, flattened in state_dict
// ---- order (SURVEY.md App. A), fp32 ----------------------------------------------------------
constexpr int RAW_E = 0;
constexpr int RAW_W1 = RAW_E + NCODES * EMB;     // (100,200)
constexpr int RAW_B1 = RAW_W1 + FC1 * READS;
constexpr int RAW_W2 = RAW_B1 + FC1;             // (10,100)
constexpr int RAW_B2 = RAW_W2 + FC2 * FC1;
constexpr int RAW_GRU = RAW_B2 + FC2;
__host__ __device__ constexpr int gru_in(int l) { return l == 0 ? IN0 : OUT_W; }
__host__ __device__ constexpr int gru_inp(int l) { return l == 0 ? IN0P : OUT_W; }
__host__ __device__ constexpr int raw_dir_size(int l) { return G3 * gru_in(l) + G3 * HID + 2 * G3; }
__host__ __device__ constexpr int raw_gru(int l, int d) {
    int off = RAW_GRU;
    for (int i = 0; i < l; ++i) off += 2 * raw_dir_size(i);
    return off + d * raw_dir_size(l);
}
__host__ __device__ constexpr int raw_wih(int l, int d) { return raw_gru(l, d); }
__host__ __device__ constexpr int raw_whh(int l, int d) { return raw_gru(l, d) + G3 * gru_in(l); }
__host__ __device__ constexpr int raw_bih(int l, int d) { return raw_whh(l, d) + G3 * HID; }
__host__ __device__ constexpr int raw_bhh(int l, int d) { return raw_bih(l, d) + G3; }
constexpr int RAW_W4 = raw_gru(LAYERS, 0);       // (5,256)
constexpr int RAW_B4 = RAW_W4 + CLASSES * OUT_W;
constexpr int RAW_TOTAL = RAW_B4 + CLASSES;
static_assert(RAW_TOTAL == 1099731, "state_dict size (SURVEY.md App. A)");

// ---- packed weights: what the kernels read (fp32, every section 128-byte aligned) ------------
__host__ __device__ constexpr int align32(int x) { return (x + 31) & ~31; }
constexpr int W1T_ROWS = READS + 1;              // row 200 is all zero: padding target of the read lists
constexpr int PK_E = 0;                                          // [c][e]           12 x 50
constexpr int PK_W1T = align32(PK_E + NCODES * EMB);             // [r][j]          201 x 100
constexpr int PK_B1 = align32(PK_W1T + W1T_ROWS * FC1);          // [j]
constexpr int PK_W2 = align32(PK_B1 + FC1);                      // [k][j]           10 x 100
constexpr int PK_B2 = align32(PK_W2 + FC2 * FC1);                // [k]
constexpr int PK_GRU = align32(PK_B2 + FC2);
// per layer:  WIH  [n][k]  n = d*384 + j*3 + g  (gate-interleaved),  k padded to gru_inp(l)
//             BGI  [n]     b_ih + (g<2 ? b_hh : 0)   (b_hn stays separate: it sits inside r*(.))
// per (l,d):  WHH  [idx][tid]  the register image of the recurrent kernel (see rec.cu)
//             BHN  [j]
constexpr int WHH_REGS = 96;
constexpr int REC_THREADS = 512;
__host__ __device__ constexpr int pk_layer_size(int l) {
    return align32(GI_N * gru_inp(l)) + align32(GI_N) + 2 * (align32(WHH_REGS * REC_THREADS) + align32(HID));
}
__host__ __device__ constexpr int pk_layer(int l) {
    int off = PK_GRU;
    for (int i = 0; i < l; ++i) off += pk_layer_size(i);
    return off;
}
__host__ __device__ constexpr int pk_wih(int l) { return pk_layer(l); }
__host__ __device__ constexpr int pk_bgi(int l) { return pk_wih(l) + align32(GI_N * gru_inp(l)); }
__host__ __device__ constexpr int pk_whh(int l, int d) {
    return pk_bgi(l) + align32(GI_N) + d * (align32(WHH_REGS * REC_THREADS) + align32(HID));
}
__host__ __device__ constexpr int pk_bhn(int l, int d) { return pk_whh(l, d) + align32(WHH_REGS * REC_THREADS); }
constexpr int PK_W4 = pk_layer(LAYERS);                          // [c][q]            5 x 256
constexpr int PK_B4 = align32(PK_W4 + CLASSES * OUT_W);
// tensor-core projection weights: W_ih split into tf32 hi/lo and stored as ready-to-copy shared-memory
// images (K-major, 128-byte swizzle) -- see proj_tc.cu.  [n_tile][k_block][hi|lo][256 rows x 32 floats]
constexpr int TC_BM = 128, TC_BN = 256, TC_BK = 32;
constexpr int TC_IMG = TC_BN * TC_BK;            // floats in one hi (or lo) image: 32 KB
__host__ __device__ constexpr int pk_wtc_size(int l) { return (GI_N / TC_BN) * (gru_inp(l) / TC_BK) * 2 * TC_IMG; }
__host__ __device__ constexpr int pk_wtc(int l) {
    int off = align32(PK_B4 + CLASSES);
    for (int i = 0; i < l; ++i) off += pk_wtc_size(i);
    return off;
}
// tensor-core recurrence operands per (layer, direction) -- see rec_tc.cu:
//   WHI  [384][128] tf32-rounded W_hh, row major (goes to tensor memory)
//   WLO  W_hh - WHI as a ready-to-copy shared-memory image [gate tile][k atom][128 rows][128 B swizzled]
//   BHN  [128]
constexpr int RTC_W = G3 * HID;                  // 49 152
constexpr int RTC_DIR = 2 * RTC_W + HID;         // floats per direction
__host__ __device__ constexpr int pk_rtc(int l, int d) { return pk_wtc(LAYERS) + (l * 2 + d) * RTC_DIR; }
// fp16-split operands (tc.cuh) -- the default kernels:
//   WH16 (proj_h.cu)  W_ih x 256 as fp16 hi / lo shared-memory images  [n_tile 3][k block of 64][hi|lo][256 rows x 128 B, SWIZZLE_128B]
//   RH16 (rec_h.cu)   W_hh x 256: hi halves as a tensor-memory image [gate tile 3][row 128][64 words: k = 2c, 2c+1], lo halves as a
//                     shared-memory image [gate tile 3][k atom 2][128 rows x 128 B, SWIZZLE_128B], then b_hn[128]
constexpr int H16_BK = 64;                       // fp16 elements per k block (one 128-byte swizzle row)
constexpr int H16_IMG = TC_BN * H16_BK / 2;      // floats in one hi (or lo) image of 256 rows: 32 KB
__host__ __device__ constexpr int pk_wh16_size(int l) { return (GI_N / TC_BN) * (gru_inp(l) / H16_BK) * 2 * H16_IMG; }
__host__ __device__ constexpr int pk_wh16(int l) {
    int off = pk_rtc(LAYERS, 0);
    for (int i = 0; i < l; ++i) off += pk_wh16_size(i);
    return off;
}
constexpr int RH16_W = 3 * 2 * HID * (HID / 2);  // 49 152 words
constexpr int RH16_DIR = RH16_W + HID;
__host__ __device__ constexpr int pk_rh16(int l, int d) { return pk_wh16(LAYERS) + (l * 2 + d) * RH16_DIR; }
// fp16-split operands of the tcgen05 front end (front_tc.cu); scales: W1 x 64, E and M x 4 (so a x 16), W2 x 256
//   FT_W1HI  [128 rows j][104 words: r = 2c, 2c+1]   W1[j][r] x 64, hi halves -- tensor-memory image (rows >= 100 zero)
//   FT_W1LO  [7 k atoms of 32 r][128 rows j][64 B]   lo halves, K-major SWIZZLE_64B shared-memory image (r < 208 used)
//   FT_W2    [2 k atoms of 64 j][32 rows: hi of k = row, lo of k = row - 16][128 B]   W2[k][j] x 256, column j = 100 holds b2[k] x 256, SWIZZLE_128B
constexpr int FT_K1 = 208;                       // read axis padded to 13 k steps of 16
constexpr int FT_W1HI_WORDS = 128 * (FT_K1 / 2);
constexpr int FT_W1LO_WORDS = 7 * 128 * 16;
constexpr int FT_W2_WORDS = 2 * 2 * 16 * 32;
constexpr int PK_FT_W1HI = pk_rh16(LAYERS, 0);
constexpr int PK_FT_W1LO = PK_FT_W1HI + FT_W1HI_WORDS;
constexpr int PK_FT_W2 = PK_FT_W1LO + FT_W1LO_WORDS;
constexpr int PK_TOTAL = PK_FT_W2 + FT_W2_WORDS;

// ---- workspace per window (floats) ------------------------------------------------------------
constexpr size_t WS_U = (size_t)COLS * IN0P;     // front-end output, k-padded
constexpr size_t WS_GI = (size_t)COLS * GI_N;    // input projection of one layer, both directions
constexpr size_t WS_H = (size_t)COLS * OUT_W;    // one layer's output; two buffers ping-pong
constexpr size_t WS_PER_WINDOW = WS_U + WS_GI + 2 * WS_H;

// ---- launchers (one per translation unit) ------------------------------------------------------
cudaError_t launch_pack(const float* raw, float* packed, int* status, cudaStream_t s);
cudaError_t launch_narrow_i64(const long long* x64, uint8_t* x8, size_t n, int* status, cudaStream_t s);
cudaError_t launch_front(const uint8_t* x, const float* packed, float* u, int nwin,
                         int* status, int num_sms, cudaStream_t s);
cudaError_t launch_proj(const float* A, int K, const float* W, const float* bias, float* C, int M,
                        cudaStream_t s);
cudaError_t launch_proj_tc3(const float* A, int K, const float* wimg, const float* bias, float* C, int M,
                            int num_sms, cudaStream_t s);
cudaError_t proj_tc3_setup();
// fp16-split projection (proj_h.cu): in_scale = power-of-two scale applied to A before the split (tc::U_SCALE / tc::H_SCALE)
// max_ctas caps the grid (at most one CTA per 128x256 tile); the CTAs stride over the tiles, so it moves no arithmetic
cudaError_t launch_proj_h(const float* A, int K, const float* wimg, const float* bias, float* C, int M, float in_scale,
                          int* status, int max_ctas, cudaStream_t s);
cudaError_t proj_h_setup();
// fp16-split recurrence (rec_h.cu): rh16_d0 = pk_rh16(l, 0), directions RH16_DIR floats apart
cudaError_t launch_rec_h(const float* gi, const float* rh16_d0, float* out, int nwin, int num_sms, cudaStream_t s);
cudaError_t rec_h_setup();
cudaError_t launch_rec_tc(const float* gi, const float* whi_d0, const float* wlo_d0, size_t dir_stride,
                          const float* bhn_d0, float* out, int nwin, int num_sms, cudaStream_t s);
cudaError_t rec_tc_setup();
cudaError_t launch_rec(const float* gi, const float* whh_d0, size_t dir_stride, const float* bhn_d0,
                       float* out, int nwin, int num_sms, cudaStream_t s);
// head (head.cu): at most max_blocks blocks of 8 warps, two rows per warp and pass; HEAD_BLOCKS_PER_SM x SMs is the full chip
constexpr int HEAD_BLOCKS_PER_SM = 8;
cudaError_t launch_head(const float* h, const float* w4, const float* b4, float* logits, uint8_t* labels,
                        int rows, int max_blocks, cudaStream_t s);
cudaError_t measure_fp32_peak(double* tflops);
cudaError_t front_setup();
// front_tc.cu: at most max_ctas persistent CTAs (one per SM), each walking windows blockIdx.x, blockIdx.x + gridDim.x, ...
cudaError_t launch_front_tc(const uint8_t* x, const float* packed, float* u, int nwin, int* status, int max_ctas,
                            cudaStream_t s);
cudaError_t front_tc_setup();
cudaError_t rec_setup();

}  // namespace roko
