/* roko_b200 -- C ABI of the B200-native replacement for roko's inference hot path.
 *
 * The reference implements this path in Python on top of PyTorch (roko/rnn_model.py `RNN`,
 * called from roko/inference.py:110-117); it has no FFI of its own for it.  The entry points
 * below are what a binding for that path needs, one per reference call site; a Python binding
 * (ctypes, roko_b200/_cabi.py) and the drop-in `RNN` class built on it (roko_b200/rnn_model.py)
 * ship in this repo, and INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * ROKO_B200_E* code, with a human-readable message available from roko_b200_last_error()
 * (thread local).  Device pointers must belong to the model's device.  Nothing here
 * synchronises the stream unless stated; work is enqueued on the `stream` argument
 * (a cudaStream_t / CUstream passed as void*, NULL = legacy default stream).
 * There is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef ROKO_B200_H
#define ROKO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ROKO_B200_ABI_VERSION 1

#define ROKO_B200_OK 0
#define ROKO_B200_EARG 1     /* bad argument (null pointer, bad size, misaligned buffer) */
#define ROKO_B200_ECUDA 2    /* a CUDA runtime call failed; message carries cudaGetErrorString */
#define ROKO_B200_ESTATE 3   /* model has no weights loaded */
#define ROKO_B200_ECODES 4   /* an input code was outside 0..11 (nn.Embedding would raise IndexError) */
#define ROKO_B200_ERANGE 5   /* a weight or activation left the range of the fp16-split tensor-core kernels */

typedef struct roko_b200_model roko_b200_model;

int roko_b200_abi_version(void);
const char* roko_b200_last_error(void);

/* Geometry of the path (reference include/generate.h:19; roko/rnn_model.py:10-12,28-44). */
int roko_b200_window_reads(void);        /* 200 */
int roko_b200_window_cols(void);         /* 90  */
int roko_b200_num_classes(void);         /* 5   */
size_t roko_b200_raw_weight_count(void); /* 1 099 731 fp32 = the 31 state_dict tensors, in order */

/* Bytes of device scratch a forward over `max_windows` windows wants.  A smaller buffer is legal:
 * forward then walks the batch in chunks that fit (at least one window must fit). */
size_t roko_b200_workspace_bytes(int max_windows);

/* RNN(IN_SIZE, HIDDEN_SIZE, NUM_LAYERS).to(device)        -- roko/inference.py:94, rnn_model.py:25-44 */
int roko_b200_model_create(roko_b200_model** out, int device);
/* model.load_state_dict(torch.load(path))                 -- roko/inference.py:95
 * `raw` holds the 31 tensors flattened in state_dict order (SURVEY.md App. A); `raw_on_device` bit 0 says
 * whether that is device (1) or host (0) memory.  Repacks them into the kernels' layouts (fp32 tables, fp16
 * hi/lo operand images for the tensor-core kernels); call again whenever the parameters change.
 * Synchronises `stream` before returning unless bit 1 of `raw_on_device` is set (2 | on_device): every kernel
 * reads its weights from the packed buffer, so later work on the SAME stream is ordered without a host
 * synchronisation (the training path reloads every step this way). */
int roko_b200_model_load(roko_b200_model* m, const float* raw, int raw_on_device, void* stream);
int roko_b200_model_destroy(roko_b200_model* m);

/* logits = model(x); Y = argmax(logits, 2)                -- roko/rnn_model.py:46-59, inference.py:115-116
 * x: device, (n_windows, 200, 90) codes 0..11, contiguous, 16-byte aligned.
 * logits (n_windows, 90, 5) fp32 and labels (n_windows, 90) uint8 are device buffers; either may
 * be NULL.  The u8 form is the native one (the .hdf5 dtype, reference roko/data.py:48); the i64
 * form accepts what the reference caller builds at inference.py:113. */
int roko_b200_forward_u8(roko_b200_model* m, const uint8_t* x, int n_windows, float* logits,
                         uint8_t* labels, void* workspace, size_t workspace_bytes, void* stream);
int roko_b200_forward_i64(roko_b200_model* m, const int64_t* x, int n_windows, float* logits,
                          uint8_t* labels, void* workspace, size_t workspace_bytes, void* stream);

/* The loop body of roko/inference.py:111-117 for HOST buffers: for each batch of `batch` windows
 * copy x to the device, run the path, copy labels (and logits if not NULL) back.  Windows are
 * independent, so consecutive batches are coalesced into device passes of up to
 * ROKO_B200_SUPERBATCH (default 2368) windows, pipelined over internal streams; returns after
 * everything has landed in the host buffers.  Pinned host memory makes the copies asynchronous. */
int roko_b200_infer_host(roko_b200_model* m, const uint8_t* x_host, long long n_windows, int batch,
                         uint8_t* labels_host, float* logits_host);

/* Scheduling and kernel-selection knobs (no effect on results beyond fp32 rounding order; every setting passes the
 * same parity tests):
 *   "rec_tc_min"    chunks of at least this many windows run the recurrence on tcgen05 (default 64; 0 = never).  Below it
 *                   the register-resident FFMA recurrence spreads few windows over many SMs for the lowest latency.
 *   "rec"           tensor-core recurrence kernel: 2 fp16-split, 48 MMAs per step (rec_h.cu, default); 1 3xTF32 (rec_tc.cu)
 *   "proj"          projection kernel: 4 tcgen05 fp16-split (proj_h.cu, default), 3 tcgen05 3xTF32, 0 FFMA SGEMM
 *   "front"         front end: 1 all contractions on tcgen05 (front_tc.cu, default), 0 SIMT gather + mma.sync (front.cu)
 *   "graphs"        replay the 8-kernel chain of roko_b200_forward_u8 as a CUDA graph (default 1; needs a non-default stream)
 *   "superbatch"    windows per device pass of roko_b200_infer_host (default 2368)
 *   "geometry"      grids of the front end, the fp16-split projection and the head: 1 work-sized (default), 0 one CTA per unit of
 *                   work up to the full chip (148 CTAs; the head 8 blocks per SM).  Geometry 1 gives each CTA at least
 *                   "geo_front" windows (default 4), "geo_proj" 128x256 projection tiles (default 6) and "geo_head" rows
 *                   (default 128), each 1 .. 1048576: a 128-window batch then runs on 32 / 45 / 90 CTAs instead of
 *                   128 / 148 / 720, so each CTA spreads its fixed prologue over more work and, with several batches in
 *                   flight on other streams, the SMs left free serve them (8.6 % more windows/s at 12 streams on a B200,
 *                   for a longer single-batch latency, 0.88 instead of 0.67 ms; DESIGN.md section 4.1).  From 2368
 *                   windows on both give the full chip.  Environment: ROKO_B200_GEOMETRY=0|1.  Training keeps full-chip grids.
 * The fp16-split kernels scale their operands by powers of two (weights x 256, activations x 16 / x 256); a GRU weight
 * with |w| >= 253 or a front-end activation >= 4062 (fc1 or fc2 output) leaves their range: roko_b200_model_check then returns
 * ROKO_B200_ERANGE and the tf32 kernels ("proj" 3, "rec" 1) serve such a model. */
int roko_b200_model_set_option(roko_b200_model* m, const char* name, long long value);

/* Synchronises the device and reports sticky errors seen by earlier calls, then clears them: ROKO_B200_ECODES for an
 * input code outside 0..11, ROKO_B200_ERANGE for a weight / activation outside the fp16-split range (see above). */
int roko_b200_model_check(roko_b200_model* m);

/* Stage taps for parity tests: run the path over n_windows (<= what fits the workspace) and copy
 * out intermediate device buffers.  Any pointer may be NULL.
 *   front (n,90,500)   gru[l] (n,90,256) for l = 0..2  */
int roko_b200_forward_taps(roko_b200_model* m, const uint8_t* x, int n_windows, float* front,
                           float* gru0, float* gru1, float* gru2, float* logits, uint8_t* labels,
                           void* workspace, size_t workspace_bytes, void* stream);

/* Measurement helpers used by bench.py (not part of the reference's interface).
 * forward_timed: `iters` forwards of one chunk with CUDA events between the 8 kernels of the chain
 *   (front, proj0, rec0, proj1, rec1, proj2, rec2, head); stage_ms[8] = mean milliseconds each.
 * measure_fp32_peak: dependent-free FFMA loop on every SM, best of 5, TFLOP/s. */
int roko_b200_forward_timed(roko_b200_model* m, const uint8_t* x, int n_windows, uint8_t* labels,
                            void* workspace, size_t workspace_bytes, void* stream, int iters,
                            float* stage_ms);
int roko_b200_measure_fp32_peak(int device, double* tflops);

/* ---- training path (reference roko/train.py:41-55 calls model(x) in train mode and backpropagates
 * F.cross_entropy through it; SURVEY.md 8 rows a11 / f1) ---------------------------------------------
 * train_forward: the train-mode forward of roko/rnn_model.py:46-59 -- the four dropout sites
 *   (rnn_model.py:29,32,35 and nn.GRU's inter-layer dropout :41) active with probability `p_drop`
 *   (0 turns them off: the eval-mode function, differentiable) and masks derived from `seed`.
 *   x (n_windows,200,90) uint8, logits (n_windows,90,5) fp32, both device.  n_windows <= 1024.
 *   `tws` (roko_b200_train_workspace_bytes(n_windows), about 4.7 MB per window, 16-byte aligned)
 *   receives the saved activations; hand the same buffer, x, p_drop and seed to train_backward.
 *   (The size follows the ROKO_B200_TRAIN_TC environment variable exactly as model creation does: the
 *   A/B chains <= 4 keep the masked embedding, 3.6 MB per window more.)
 * train_backward: given dlogits = dLoss/dlogits (n_windows,90,5), writes the gradient of every
 *   parameter into grad_raw: 1 099 731 fp32 in state_dict order, the layout roko_b200_model_load reads.
 *   Consumes `tws` (one backward per forward).  The cross-entropy itself (train.py:52) stays with the caller.
 * dropout_mask: the keep mask (1 = kept) these kernels use for `site` and element indices 0..n-1 in the
 *   reference tensor's row-major order -- sites: 0 embedding (B,200,90,50), 1 fc1 (B,90,50,100),
 *   2 fc2 (B,90,50,10), 3 / 4 output of GRU layer 0 / 1 (B,90,256).  For tests. */
size_t roko_b200_train_workspace_bytes(int n_windows);
int roko_b200_train_forward(roko_b200_model* m, const uint8_t* x, int n_windows, float p_drop,
                            unsigned long long seed, float* logits, void* tws, size_t tws_bytes, void* stream);
int roko_b200_train_backward(roko_b200_model* m, const uint8_t* x, int n_windows, float p_drop,
                             unsigned long long seed, const float* dlogits, float* grad_raw, void* tws,
                             size_t tws_bytes, void* stream);
int roko_b200_dropout_mask(float p_drop, unsigned long long seed, int site, size_t n, uint8_t* mask_out,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ROKO_B200_H */
