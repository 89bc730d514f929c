/*
 * riser_b200 -- C ABI of the B200-native RISER read-classification hot path.
 *
 * This is the drop-in boundary: a plain C interface (pointers + sizes, no torch
 * types) over hand-written sm_100a kernels.  The reference (comprna/riser) has no
 * FFI of its own -- its hot path is three Python objects -- so each entry point
 * below cites the reference function it replaces (paths relative to the reference
 * checkout).  The Python host side (riser_b200/{preprocess,model,control}.py)
 * mirrors the reference's Kit / SignalProcessor / Model / SequencerControl call
 * surface and reaches these functions through ctypes (riser_b200/_lib.py);
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - every launch function takes the cudaStream_t to run on, never synchronises
 *     and never allocates: the caller owns all buffers (capturable in CUDA graphs);
 *   - return value 0 = ok, otherwise a RISER_E* code; riser_last_error() returns a
 *     thread-local message; no C++ exception crosses the boundary;
 *   - there is NO CPU fallback: without an sm_100 device the calls return
 *     RISER_ECUDA.
 */
#ifndef RISER_B200_H
#define RISER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* riser_stream_t; /* == cudaStream_t */

enum {
  RISER_OK = 0,
  RISER_EINVAL = 1, /* bad argument (null pointer, size out of range, misalignment) */
  RISER_ECUDA = 2,  /* CUDA runtime / driver error, or no sm_100 device            */
  RISER_ENOMEM = 3, /* workspace too small                                         */
};

/* Decision codes written by riser_decide (riser/control.py:75-82; 4 = the two
 * `continue` branches at control.py:50,56). */
enum {
  RISER_TRY_AGAIN = 0,
  RISER_ACCEPT = 1,
  RISER_REJECT = 2,
  RISER_NO_DECISION = 3,
  RISER_SKIPPED = 4,
};

/* mode argument of riser_decide (riser/riser.py:91-95, control.py:76,78) */
enum { RISER_MODE_ENRICH = 0, RISER_MODE_DEPLETE = 1 };

/* Arithmetic of the convolution stack (layers 1..n-1; layer 0 and the head are
 * always fp32).  Operands are fp16 (10-bit mantissa, the same as tf32, at twice
 * the tensor rate); accumulation is fp32 in TMEM.
 *   F16    : one tcgen05 pass; weights and activations rounded to fp16.
 *   F16_W2 : two passes; weights split hi + lo fp16 (exact to ~22 bits), only the
 *            activation rounding remains.
 *   F16_X3 : three passes; weights AND activations split hi + lo
 *            (W_hi a_hi + W_lo a_hi + W_hi a_lo): fp32-class results.
 *   F16_F8 : the fp16 pass plus ONE e4m3 pass (kind::f8f6f4, twice the fp16 rate)
 *            that carries both correction terms, (W_lo 2^3)(a 2^-3) + (W 2^-9)(a_lo 2^9):
 *            the corrections are ~2^-11 of the result, so 3 mantissa bits suffice
 *            (format error ~6e-5 on the probabilities).  Two pass-equivalents of
 *            tensor work instead of three; activation rows are
 *            [hi fp16 | e4m3(a 2^-3) | e4m3(a_lo 2^9)] = the bytes of hi + lo.   */
enum { RISER_PREC_F16 = 0, RISER_PREC_F16_W2 = 1, RISER_PREC_F16_X3 = 2, RISER_PREC_F16_F8 = 3 };

int riser_version(void);
const char* riser_last_error(void);

/* Device properties the host side needs: fills sm_count, cc_major, cc_minor. */
int riser_device_info(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------ preprocessing */

/* Maximum window length riser_normalise accepts (samples staged in shared memory). */
int riser_normalise_max_len(void);

/* Replaces SignalProcessor.mad_normalise + _calculate_mad + _normalise +
 * _smooth_outliers + _clip_if_outlier (riser/preprocess.py:108-147), batched over
 * ragged windows.  Read b's window is sig[off[b] + start[b] .. + len[b]).
 * Exact integer selection of median and MAD, float64 normalise and sequential
 * outlier smoothing exactly as the reference, result rounded to fp32 (the cast
 * riser/model.py:25 applies) into out[b * ld_out + i], i < len[b].  Elements
 * i >= len[b] of the row are not written.  len[b] == 0 writes nothing.
 * mad == 0 writes zeros (preprocess.py:122-124).
 * out must be 16-byte aligned and ld_out a multiple of 4.  max_len bounds every len[b]
 * (<= riser_normalise_max_len()); a longer window is processed as its first max_len samples.
 * The window is staged by a bulk copy of whole 16-byte blocks: the sig allocation must
 * reach the end of the 16-byte block that holds a window's last sample (any cudaMalloc'd
 * buffer does).  off[b] may be a VIRTUAL start (the caller uploaded only part of read b),
 * as long as [off[b] + start[b], off[b] + start[b] + len[b]) lies inside the allocation.
 * med2_mad4 (optional, may be NULL): int32 [B,2] = {2*median, 4*MAD} (exact).  */
int riser_normalise(const int16_t* sig, const int64_t* off, const int32_t* start,
                    const int32_t* len, int B, int max_len, float* out, int64_t ld_out,
                    int32_t* med2_mad4, riser_stream_t stream);

/* float32 variant for the training-data preparation path: replaces mad_normalise /
 * smooth_outliers / calculate_mad / normalise of riser/retrain/preprocess.py:8-44, where the
 * input is the pA-scaled float32 signal and numpy keeps every step in float32 (no MAD == 0
 * guard: IEEE inf / nan as numpy gives).  Read b is sig[off[b] .. off[b] + len[b]).         */
int riser_normalise_f32_max_len(void);
int riser_normalise_f32(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                        float outlier_lim, float* out, int64_t ld_out, riser_stream_t stream);

/* The live path's SignalProcessor.mad_normalise (riser/preprocess.py:108-147) for float32 input -- the
 * secondary input mode (calibrated signal; SURVEY.md 8c): numpy keeps float32 throughout there too
 * (np.median, np.vectorize over float32 scalars), so the arithmetic is that of riser_normalise_f32 with
 * the outlier limit 3.5 and WITH the MAD == 0 guard of preprocess.py:122-124 (all-zero output).
 * med_mad (optional, may be NULL): float32 [B,2] = {median, MAD}, so the host mirror can return the
 * reference's int64 zeros when MAD == 0.                                                         */
int riser_normalise_f32_live(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                             float* out, int64_t ld_out, float* med_mad, riser_stream_t stream);

/* Windows of any length (max_len up to INT32_MAX): the three entry points above hold a whole window in one
 * CTA's shared memory and refuse longer ones; these keep it in global memory and work on it with many CTAs
 * (exact multi-pass radix select for median and MAD, then the elementwise normalise and the sequential
 * outlier smoothing).  The results are those of riser_normalise / riser_normalise_f32(_live) bit for bit, at
 * any length, short windows included.  The arguments mean what they mean there, except:
 *   - out needs no alignment and ld_out only ld_out >= max_len; elements i >= len[b] of a row are not
 *     written, len[b] == 0 writes nothing, and a window longer than max_len is processed as its first
 *     max_len samples (riser_normalise_f32_long too);
 *   - riser_normalise_f32_long: outlier_lim and zero_if_mad0 choose between riser_normalise_f32 (the
 *     caller's limit, 0 = no MAD == 0 guard: IEEE inf / nan) and riser_normalise_f32_live (3.5, 1 = zeros
 *     when MAD == 0); med_mad (optional) as riser_normalise_f32_live's;
 *   - workspace: device memory of at least riser_normalise_long_workspace_bytes(B, max_len) bytes, 16-byte
 *     aligned, any content (RISER_ENOMEM when smaller).  Its contents are scratch between calls; two calls in
 *     flight at once need two workspaces.
 * Each call launches a fixed sequence of kernels for a given (B, max_len), so it can be captured in a CUDA
 * graph.  On short windows the shared-memory entry points are faster; callers pick by length
 * (SignalProcessor.mad_normalise_batch sends only windows above riser_normalise_max_len() here).          */
size_t riser_normalise_long_workspace_bytes(int B, int max_len);
int riser_normalise_long(const int16_t* sig, const int64_t* off, const int32_t* start, const int32_t* len, int B,
                         int max_len, float* out, int64_t ld_out, int32_t* med2_mad4,
                         void* workspace, size_t workspace_bytes, riser_stream_t stream);
int riser_normalise_f32_long(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                             float outlier_lim, int zero_if_mad0, float* out, int64_t ld_out, float* med_mad,
                             void* workspace, size_t workspace_bytes, riser_stream_t stream);

/* Replaces SignalProcessor.get_polyA_end (riser/preprocess.py:42-79), batched.
 * Read b is sig[off[b] .. off[b] + n[b]).  polya_end[b] = the returned window
 * start index, or -1 for None.  Window statistics are exact integers; the
 * mean-change test is evaluated in float64 in the reference's operation order.
 * polya_start (optional, may be NULL): the poly(A) start window the scan found, -1 for
 * None (riser/test.py:80-117 get_polyA_coords returns both, at resolution 500 / MAD 20).
 * stats (optional, may be NULL): int32 [B, max_windows, 3] = {sum, 2*median,
 * 4*MAD} per 500-sample window.  At most the first 512 windows (256,000 samples) of a
 * prefix are scanned; the live loop never holds more than ~18,500 (control.py:42-46).    */
int riser_polya_end(const int16_t* sig, const int64_t* off, const int32_t* n, int B,
                    int32_t* polya_end, int32_t* polya_start, int32_t* stats, int max_windows,
                    riser_stream_t stream);

/* riser_polya_end for float32 (calibrated, pA) signal -- the secondary input mode: the same windows, scan,
 * 512-window cap and -1 conventions, with every window statistic computed as numpy computes it for float32
 * input (float32 median / MAD of the two middle values, np.mean's pairwise float32 sum, the rolling mean of
 * the previous 1,000 samples as its own pairwise sum, the mean-change test in float32).  Read b is
 * sig[off[b] .. off[b] + n[b]); 16-byte aligned reads take vector loads.
 * stats (optional, may be NULL): float32 [B, max_windows, 4] = {median, MAD, mean, rolling mean}.          */
int riser_polya_end_f32(const float* sig, const int64_t* off, const int32_t* n, int B,
                        int32_t* polya_end, int32_t* polya_start, float* stats, int max_windows,
                        riser_stream_t stream);

/* Replaces the length gating of riser/control.py:36-60 (with preprocess.py:84-85,
 * 100, 104-106), batched: for read b of n[b] samples and poly(A) end `end` =
 * cached_end[b] if >= 0 else detected_end[b] (-1 = none found):
 *   found    : start = end + 1; skip if n - start < min_len; len = min(n - start, max_len)
 *   not found: if n > fixed_trim + max_len  -> start = fixed_trim, len = max_len; else skip
 * Skipped reads get len 0 (and start 0).                                          */
int riser_select_window(const int32_t* n, const int32_t* cached_end, const int32_t* detected_end,
                        int B, int min_len, int max_len, int fixed_trim, int32_t* start,
                        int32_t* len, riser_stream_t stream);

/* ------------------------------------------------------------------ network */

typedef struct riser_model riser_model; /* packed weights of one ConvNet on one device */
typedef struct riser_plan riser_plan;   /* launch plan for one (batch, max length) shape */

/* Replaces Model.__init__'s ConvNet(config.cnn) + load_state_dict
 * (riser/model.py:18-20, riser/nets/cnn.py:8-41,52-65; depth 1, 'gap_fc' head,
 * 2 classes, kernel 3 -- the only shape the shipped configs use,
 * riser/model/\*.yaml:6-12).  conv_w_host[i] is the fp32 [channels[i], cin_i, 3]
 * weight of layers.{i}.0 (cin_0 = 1, cin_i = channels[i-1]); conv_b_host[i] its
 * bias; fc_w_host [2, channels[n-1]], fc_b_host [2] the classifier.2 tensors.
 * Packs them on the host into the tap-major, channel-padded fp16 layout the
 * tcgen05 kernel reads and uploads them to `device`.                           */
int riser_model_create(riser_model** out, int n_layers, const int* channels,
                       const float* const* conv_w_host, const float* const* conv_b_host,
                       const float* fc_w_host, const float* fc_b_host, int precision,
                       int device);
int riser_model_destroy(riser_model* m);

/* Bytes of activation workspace a plan for (B reads, longest window max_len) needs. */
size_t riser_workspace_bytes(const riser_model* m, int B, int max_len);

/* Builds the TMA tensor maps and per-layer launch geometry for (B, max_len) over
 * the caller's workspace (256-byte aligned, >= riser_workspace_bytes; it is
 * zeroed once here, asynchronously on `stream`).                               */
int riser_plan_create(riser_plan** out, const riser_model* m, int B, int max_len,
                      void* workspace, size_t workspace_bytes, riser_stream_t stream);
int riser_plan_destroy(riser_plan* p);

/* Replaces Model.classify (riser/model.py:22-28) and ConvNet.forward
 * (riser/nets/cnn.py:43-50), batched over ragged reads: x is the normalised
 * signal, fp32 [B, ld_x], read b valid for len[b] samples (4096 <= len[b] <=
 * max_len).  Per-layer length masks (L_{i+1} = floor(L_i / 2)) make every read's
 * result equal to classifying it alone.  probs [B, 2] = softmax(logits) =
 * (p_off_target, p_on_target).  A read with len[b] < 4096 gets NaN (the
 * reference raises in max_pool1d for such input).
 * x must be 16-byte aligned with ld_x a multiple of 4 (>= max_len): the fused layers
 * 0 + 1 stage the signal with bulk copies (RISER_EINVAL otherwise).  Values beyond
 * len[b] in a row are never read as signal.
 * feat (optional, may be NULL): fp32 [B, channels[n-1]] pooled features.       */
int riser_forward(const riser_plan* p, const float* x, int64_t ld_x, const int32_t* len,
                  float* probs, float* feat, riser_stream_t stream);

/* The stages of riser_forward, callable separately so that a caller can put CUDA
 * events between them (bench.py times the conv stack):
 *   0 = tile activity flags (+ layer 0 when it is not fused into layer 1's launch);
 *   1 = the conv layers (tcgen05; layers 0 + 1 are one launch by default);  2 = head;
 *   3 = the layer-0 launches of stage 0 alone (timing aid, not part of riser_forward);
 *   16 + i = conv layer i (>= 1) alone, so that a tool can bracket every layer of a forward with
 *   CUDA events (stage 0, then 16 + 1 .. 16 + n_layers - 1, then 2 == riser_forward).          */
int riser_forward_stage(const riser_plan* p, int stage, const float* x, int64_t ld_x,
                        const int32_t* len, float* probs, float* feat, riser_stream_t stream);

/* Number of kernels one riser_forward launches (for gpu_launches accounting). */
int riser_forward_launches(const riser_plan* p);

/* 1 when the plan computes layer 0 inside layer 1's kernel (its activation buffer is then
 * never written and stage 3 launches nothing). */
int riser_plan_fused_layer0(const riser_plan* p);

/* Introspection for tests / profiling: layer i (1..n_layers) reads (i < n) or, for
 * i == n_layers, the head reads, an activation buffer at workspace + *offset laid out
 * [B * *rows_per_read][*channels_padded], fp16 for i < n_layers, fp32 for i == n_layers.
 * *channels = unpadded channel count, *n_tile = the tcgen05 N tile of the layer that
 * WROTE it.                                                                      */
int riser_plan_layer_info(const riser_plan* p, int i, int64_t* offset, int* rows_per_read,
                          int* channels_padded, int* channels, int* n_tile);

/* 1 when layer i's input buffer uses the even / odd plane layout: all even rows of every
 * read (row = b * rows_per_read / 2 + t / 2) followed by all odd rows, instead of the flat
 * [B * rows_per_read] order.  Same size, same row format.                            */
int riser_plan_layer_eo(const riser_plan* p, int i);

/* Row format of layer i's input buffer (i = 1..n_layers-1), decided per layer by the precision
 * mode (DESIGN.md section 2):
 *   1 = one fp16 plane [channels_padded];
 *   2 = fp16 hi | fp16 lo planes (a = hi + lo; the F16_X3 terms W_hi*a_hi + W_lo*a_hi + W_hi*a_lo);
 *   3 = fp16 hi | e4m3(a * 2^-3) | e4m3((a - hi) * 2^9): the operands of the fp16 pass and of the single
 *       e4m3 correction pass of RISER_PREC_F16_F8 (same bytes per row as format 2).
 * 0 for i outside that range, -1 when the buffer is never materialised (layer i is computed inside layer
 * i - 1's launch: conv_eo2_kernel).  Tests decode activations with it; bench.py derives the tensor passes
 * executed per algorithmic FLOP from it (riser/nets/cnn.py:55-64 is one fp32 pass).            */
int riser_plan_layer_format(const riser_plan* p, int i);

/* Which kernel runs conv layer i (1..n_layers-1) in this plan: 0 = conv_tc_kernel (one CTA per SM),
 * 1 = conv_eo_kernel (even / odd planes, resident weights), 2 = conv_pair_kernel (cta_group::2 CTA
 * pairs), 3 = fused01_kernel (layers 0 + 1 in one launch), 5 = conv_eo2_kernel (this layer and its
 * neighbour in one launch, the activation between them kept in shared memory).  -1 outside the range.  For bench.py's launch description. */
int riser_plan_layer_kernel(const riser_plan* p, int i);

/* Replaces the decision rule of riser/control.py:75-82 for M models:
 * probs [M, B, 2]; len [B] = post-trim window length, 0 = read was skipped
 * (control.py:50,56) -> RISER_SKIPPED.  Strict '>' against thr in fp32.        */
int riser_decide(const float* probs, const int32_t* len, int B, int M, float thr, int mode,
                 int max_len, uint8_t* decision, riser_stream_t stream);

/* ------------------------------------------------------------------ ResNet variant
 * riser/nets/resnet.py (selectable only in train.py:177-178; no shipped config or weights).
 * Generic fp32 building blocks on CUDA cores, channel-last activations [B][L_pad][C], per-read
 * valid lengths; BatchNorm is folded into w / bias by the host (riser_b200/resnet.py).      */

/* The stem in one launch: Conv1d(1 -> C, K, stride, padding) + folded BatchNorm + ReLU + MaxPool1d(2, 2, padding 1)
 * (resnet.py:79-84).  x: fp32 [B][ld_x] normalised signal; w [K][Cp], bias [Cp] (Cp = channels padded to 4, zeros in
 * the padding); len_conv / len_out: valid lengths after the convolution / after the pool; out [B][Lout_pad][Cp].   */
int riser_stem_pool_cl(const float* x, int64_t ld_x, const int32_t* len_in, const float* w, const float* bias,
                       float* out, const int32_t* len_conv, const int32_t* len_out, int B, int Lout_pad, int Cp, int K,
                       int stride, int pad, riser_stream_t stream);

/* The ResNet blocks on the tensor pipe (tcgen05, fp16 hi + lo operand planes = three passes, fp32 accumulation
 * in TMEM).  One entry point, two modes:
 *   w2 == NULL  one conv_block of resnet.py:26-37: Conv1d(k = taps in {1, 3}, stride in {1, 2}, padding (k-1)/2)
 *               with the BatchNorm folded in, + residual (optional, the output's layout) + ReLU (`relu`);
 *   w2 != NULL  a whole BasicBlock (resnet.py:50-57 + ResidualBlock.forward, resnet.py:39-47):
 *               out = ReLU(conv2(ReLU(conv1_stride(x))) + shortcut(x)); the shortcut is the 1x1 stride-s conv
 *               `wsc` (accumulated into conv2's accumulator; bias2 = conv2 bias + shortcut bias), else
 *               `residual` (= x for the identity shortcut), else nothing.  The intermediate stays on the SM.
 * Activations: fp32 channel-last [B][L_pad][C_p], channels padded to a multiple of 8 (padding channels zero),
 * 32-byte aligned; rows outside [0, len_in[b]) read as zero, rows >= len_out[b] are not written.
 * Weights: host-packed operand images (riser_b200/resnet.py pack_tc_weights): fp16 [tap][K block of 32 channels]
 * [plane hi, lo][N rows][32] in the K-major SWIZZLE_64B layout, multiplied by a power of two whose inverse is
 * inv_scale*.  n1 / n2: output channels padded to 16 (<= 256).  cmid_p: conv1's output channels (fused mode).
 * riser_res_tc_smem: shared memory a shape needs, 0 if unsupported (the caller falls back to riser_conv1d_cl). */
size_t riser_res_tc_smem(int cin_p, int cmid_p, int n1, int n2, int taps, int stride, int fused, int shortcut_conv);
int riser_res_tc(const float* in, const int32_t* len_in, const int32_t* len_out, float* out, const float* residual,
                 const void* w1, const void* w2, const void* wsc, const float* bias1, const float* bias2,
                 float inv_scale1, float inv_scale2, int B, int Lin_pad, int Lout_pad, int cin_p, int cmid_p,
                 int cout_p, int n1, int n2, int taps, int stride, int relu, riser_stream_t stream);

/* The same launches in a chosen arithmetic (RISER_PREC_*; with RISER_PREC_F16_X3 these ARE riser_res_tc_smem /
 * riser_res_tc, bit for bit).  Per mode, the MMAs of a tap and 16-channel K step and the weight image (per tap and
 * 32-channel K block, planes of N rows x 64 bytes, each SWIZZLE_64B, weights w = W * 2^e):
 *   F16     a_hi W_hi                                    image [hi]: fp16(w)
 *   F16_W2  a_hi [W_hi; W_lo] (one MMA when 2N <= 256)    image [hi, lo]: fp16(w), fp16(w - hi)
 *   F16_X3  + a_lo W_hi                                  image [hi, lo] (as riser_res_tc)
 *   F16_F8  a_hi W_hi, plus per K block two kind::f8f6f4 MMAs (K = 32) of the activation row
 *           [e4m3(a 2^-3) x32 | e4m3((a - a_hi) 2^9) x32] against the weight row [e4m3((w - hi) 2^3) x32 |
 *           e4m3(w 2^-9) x32]: image [hi, e4m3 row] (64 bytes per row, the size of an fp16 plane row).
 * Activations stay fp32 in memory whatever the mode; the kernel converts them to the mode's operand tiles (the fused
 * BasicBlock's intermediate too).  e4m3(a 2^-3) saturates at |a| = 3584.  riser_res_tc_smem_ex returns 0 for an
 * unknown mode; F16 and F16_W2 need less shared memory than F16_X3 (no lo / e4m3 activation tiles; F16 no weight lo
 * plane), so a block may fit in those modes and not in F16_X3.                                                  */
size_t riser_res_tc_smem_ex(int cin_p, int cmid_p, int n1, int n2, int taps, int stride, int fused, int shortcut_conv,
                            int precision);
int riser_res_tc_ex(const float* in, const int32_t* len_in, const int32_t* len_out, float* out, const float* residual,
                    const void* w1, const void* w2, const void* wsc, const float* bias1, const float* bias2,
                    float inv_scale1, float inv_scale2, int B, int Lin_pad, int Lout_pad, int cin_p, int cmid_p,
                    int cout_p, int n1, int n2, int taps, int stride, int relu, riser_stream_t stream, int precision);

/* Conv1d(Cin->Cout, K, stride, padding) [+ residual] [+ ReLU] -- resnet.py:26-43,79-81.
 * w is packed [K][Cin][Cout]; rows outside [0, len_in[b]) are zero padding; rows
 * t >= len_out[b] are not written.  residual (optional) has the output's layout.          */
int riser_conv1d_cl(const float* in, const int32_t* len_in, const float* w, const float* bias,
                    const float* residual, float* out, const int32_t* len_out, int B, int Lin_pad,
                    int Lout_pad, int Cin, int Cout, int K, int stride, int pad, int relu,
                    riser_stream_t stream);

/* Valid lengths after every op of the main chain (stem conv, stem max-pool, the convolutions of every block),
 * from the input lengths, in one launch: ksp int32 [n_ops][3] = (kernel, stride, padding) per op, kernel < 0 for
 * MaxPool1d(2, 2, padding p); out int32 [n_ops][B].  torch's own formulas: Conv1d floor((n + 2p - k) / s) + 1
 * (0 when the window does not fit), pool (n + 2p) / 2 (resnet.py:79-83: p = 1; nets/cnn.py:64: p = 0).  */
int riser_len_chain(const int32_t* len0, int B, const int32_t* ksp, int n_ops, int32_t* out,
                    riser_stream_t stream);

/* MaxPool1d(kernel 2, stride 2, padding 1) -- resnet.py:83.                                 */
int riser_maxpool1d_cl(const float* in, const int32_t* len_in, float* out, const int32_t* len_out,
                       int B, int Lin_pad, int Lout_pad, int C, riser_stream_t stream);

/* MaxPool1d(kernel 2, stride 2, padding `pad` in {0, 1}) on the same layout: pad 0 is the pool that ends every
 * ConvNet layer (nets/cnn.py:64; the generic, non-shipped ConvNet shapes run through these fp32 channel-last ops,
 * riser_b200/convnet_generic.py), pad 1 the ResNet stem's (resnet.py:83).                     */
int riser_maxpool1d_pad_cl(const float* in, const int32_t* len_in, float* out, const int32_t* len_out,
                           int B, int Lin_pad, int Lout_pad, int C, int pad, riser_stream_t stream);

/* AdaptiveAvgPool1d(1) + Flatten + Linear(C, n_classes) + softmax -- resnet.py:94-98,
 * model.py:27.  probs [B][n_classes]; NaN for len 0.                                        */
int riser_gap_linear_softmax(const float* in, const int32_t* len, const float* fc_w, const float* fc_b,
                             float* probs, int B, int L_pad, int C, int n_classes,
                             riser_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RISER_B200_H */
