/*
 * timbre_trap_b200 - C ABI of the B200 (sm_100a) hot path of sony/timbre-trap.
 *
 * The reference has no FFI: its boundary for this path is the Python class API of
 * timbre_trap.framework (reference: timbre_trap/framework/__init__.py:1-4).  The Python host
 * side of this repo (timbre_trap_b200/framework) mirrors those classes and binds the entry
 * points below with ctypes; each entry point cites the reference method it replaces.
 *
 * Conventions
 *   - plain C: raw DEVICE pointers, sizes, a cudaStream_t passed as void*; no torch types.
 *   - every function returns 0 (TT_OK) on success, non-zero otherwise; tt_last_error() gives
 *     the message of the last failure on the calling thread.  Nothing throws.
 *   - no ownership transfer: callers own every buffer except the plan's private scratch.
 *   - calls are asynchronous on `stream`; a plan (it owns scratch) must be used from one
 *     stream at a time.
 *
 * Layouts
 *   audio         (B, n_blocks * L)            fp32, L = block_length
 *   coefficients  (B, F, n_blocks * M, 2)      fp32 interleaved (re, im) - i.e. exactly the memory
 *                                              behind the reference's (B, 2, F, T) `to_real` view
 *                                              (cqtwrapper.py:91-95): channels-last
 */
#ifndef TIMBRE_TRAP_B200_H
#define TIMBRE_TRAP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tt_cqt_plan tt_cqt_plan;

/* library / error plumbing */
const char* tt_last_error(void);
int tt_version(void);
/* number of kernels this library has launched since load (or since the last call with reset != 0) */
long long tt_launch_count(int reset);

/*
 * Replaces cqt_pytorch.CQT.__init__ as called from cqtwrapper.py:31-35 (the window / index /
 * dual tables).  All table pointers are HOST arrays in the packed form documented in
 * oracle/nsgt_ref.py::NSGTTables: per bin k, `length[k]` non-zero taps that start at crop
 * index `first[k]` and at spectrum index `start[k]`; `offset[k]` is the prefix sum.
 * `max_blocks_per_launch` bounds the plan's scratch (blocks are processed in groups).
 */
int tt_cqt_plan_create(tt_cqt_plan** plan, int block_length, int n_bins, int max_window_length,
                       const int32_t* start, const int32_t* length, const int32_t* first, const int32_t* offset,
                       const float* win_packed, const float* dual_packed, int n_taps,
                       int max_blocks_per_launch);
int tt_cqt_plan_destroy(tt_cqt_plan* plan);
/* Number of internal streams ("lanes", 1..4, default 2) consecutive groups of `max_blocks_per_launch` blocks rotate over: the FFT
 * front end of one group overlaps the HBM-bound per-bin kernel of another.  Results do not depend on it. */
int tt_cqt_plan_set_lanes(tt_cqt_plan* plan, int n_lanes);
/* bytes of device scratch held by the plan */
int64_t tt_cqt_plan_scratch_bytes(const tt_cqt_plan* plan);

/*
 * CQT.forward / encode + to_real  (cqtwrapper.py:50-97).
 *   audio   (batch, n_blocks * L) fp32
 *   coeffs  (batch, F, n_blocks * M, 2) fp32
 */
int tt_cqt_forward(tt_cqt_plan* plan, const float* audio, int batch, int n_blocks, float* coeffs, void* stream);

/*
 * CQT.decode  (cqtwrapper.py:184-213): to_complex + synthesis + global infinity-norm normalise.
 *   coeffs     (batch, F, n_blocks * M, 2) fp32
 *   audio      (batch, n_blocks * L) fp32
 *   peak       device scalar (fp32, >= 0): receives max|audio| BEFORE normalisation; must be
 *              zero-initialised by the caller OR pass accumulate_peak = 0 to have it reset here.
 *   normalise  0: leave audio un-normalised (peak still written) - the sharded path all-reduces
 *              `peak` across ranks and then calls tt_scale_by_peak;
 *              1: divide by the peak when it is non-zero (reference semantics).
 */
int tt_cqt_inverse(tt_cqt_plan* plan, const float* coeffs, int batch, int n_blocks, float* audio,
                   float* peak, int normalise, void* stream);

/* audio[i] /= *peak when *peak != 0  (cqtwrapper.py:209-211) */
int tt_scale_by_peak(float* audio, int64_t n, const float* peak, void* stream);

/*
 * ---- many clips of different lengths in one call (TimbreTrap.transcribe_many / reconstruct_many) ---------------------------------
 * A clip table is a device int32 prefix array of n_clips + 1 entries: clip c owns entries [t[c], t[c+1]) (at least one), counted
 * from t[0], so a slice of a longer table describes the clips it covers.  clip_block0 counts blocks (n_c = ceil(samples / L)),
 * clip_chunk0 chunks (2 n_c + 1 per clip).  Per-clip tensors follow one another, each in the layout a one-clip call produces.
 */
/* tt_cqt_inverse over clips: coeffs = the clips' (F, n_c * M, 2) tensors, audio = their (n_c * L) samples, n_blocks = t[n] - t[0];
 * peaks (n_clips) fp32 device: max|audio| of each clip before normalisation (reset here); normalise as tt_cqt_inverse, per clip */
int tt_cqt_inverse_clips(tt_cqt_plan* plan, const float* coeffs, const int* clip_block0, int n_clips, int n_blocks, float* audio,
                         float* peaks, int normalise, void* stream);

/* audio of the clips of clip_block0 (n_blocks blocks of block_length samples): each divided by its own peak when non-zero */
int tt_scale_by_clip_peak(float* audio, const int* clip_block0, int n_clips, int n_blocks, int block_length, const float* peaks,
                          void* stream);

/* the chunk matrix: out row r = chunk chunk_lo + r of the clips (TimbreTrap._chunks, modules.py:226-234, for each clip: padded with
 * zeros to whole blocks, then by half a block on either side), r < n_rows.
 *   clips  (n_clips, 2) int64 device: (address of the clip's fp32 samples, number of samples)
 *   out    (n_rows, block_length) fp32 */
int tt_gather_chunks(const int64_t* clips, const int* clip_chunk0, int n_clips, int chunk_lo, int n_rows, int block_length,
                     float* out, void* stream);

/*
 * TimbreTrap.to_activations (modules.py:271-289) = tanh(CQT.to_magnitude) (cqtwrapper.py:122-141)
 *   coeffs (rows, 2) interleaved -> out (rows);  apply_tanh = 0 gives the plain magnitude
 */
int tt_magnitude(const float* coeffs, int64_t n, int apply_tanh, float* out, void* stream);

/*
 * CQT.to_decibels (cqtwrapper.py:143-182): per batch item 20*log10(max(x,1e-10)), floored at the
 * item's max - 80 dB; if rescale: shifted to a 0 dB ceiling and mapped to [0,1].
 *   magnitude, out  (batch, per_item)
 *   item_max        device scratch of `batch` floats
 */
int tt_to_decibels(const float* magnitude, int batch, int64_t per_item, int rescale, float* out,
                   float* item_max, void* stream);

/*
 * Hann cross-fade of 50 %-overlapped chunk outputs + trim (TimbreTrap.chunked_inference, modules.py:237-267).
 *   chunks      (batch * n_chunks, F, M, 2) fp32 - chunk i of item b at index b * n_chunks + i
 *   window      (M) fp32 device (torch.signal.windows.hann, modules.py:239)
 *   coeffs_out  (batch, F, (n_chunks-1) * M/2, 2) or NULL
 *   act_out     (batch, F, (n_chunks-1) * M/2)    or NULL: tanh(|.|) of the cross-faded coefficients
 *               (TimbreTrap.to_activations, modules.py:271-289, fused for transcribe())
 */
int tt_chunk_crossfade(const float* chunks, const float* window, int batch, int n_chunks, int n_bins, int frames_per_chunk,
                       float* coeffs_out, float* act_out, void* stream);

/* tt_chunk_crossfade over the clips of clip_chunk0: chunks (t[n] - t[0], F, M, 2); clip c's outputs (F, (n_c - 1) * M/2 [, 2]) follow
 * those of the clips before it; max_chunks = the most chunks of any clip */
int tt_chunk_crossfade_clips(const float* chunks, const float* window, const int* clip_chunk0, int n_clips, int max_chunks, int n_bins,
                             int frames_per_chunk, float* coeffs_out, float* act_out, void* stream);

/*
 * ---- evaluation post-processing, the step after `transcribe` (SURVEY.md section 8f-1) --------------------------------
 * activations (B, F, T) fp32 row-major.  Bit-exact against oracle/postproc_ref.py.
 */
/* filter_non_peaks (timbre_trap/utils/processing.py:66-98): out = activations where strictly greater than both frequency
 * neighbours (zeros beyond the edges), else 0 */
int tt_filter_non_peaks(const float* activations, float* out, int B, int F, int T, void* stream);
/* PitchDataset.activations_to_multi_pitch's binary map (datasets/PitchDataset.py:309-349): optional filter_non_peaks, then
 * threshold (processing.py:101-124, `>= threshold`), restricted to bins [bin_lo, bin_hi) (the mask of experiments/evaluate.py:48);
 * out (B, F, T) uint8 in {0, 1} */
int tt_peak_threshold(const float* activations, unsigned char* out, int B, int F, int T, float threshold, int peaks_only,
                      int bin_lo, int bin_hi, void* stream);
/* Frame-wise multi-pitch matching in the manner of mir_eval.multipitch (utils/experiments.py:354-396): per frame the maximum
 * matching between estimated and reference bins whose distance is <= tolerance_bins; counts (B, 3) int64 = true positives,
 * estimated, reference (precision = tp / est, recall = tp / ref).  counts is zeroed by the call. */
int tt_multipitch_counts(const unsigned char* est, const unsigned char* ref, int B, int F, int T, int tolerance_bins,
                         int64_t* counts, void* stream);

/*
 * ---- conv autoencoder (modules.py:396-777), bf16 tensor-core implicit GEMMs --------------------------------
 * Activations: "C8 planar" bf16  [B][ceil(C/8)][H][T][8]  (channel counts below are the PADDED counts, multiples of 8).
 * Weights: pre-packed bf16 in the tcgen05 B-operand layout [K/8][N][8]; K order and zero padding are documented at
 * timbre_trap_b200/framework/packing.py (one function per entry point).  Biases: fp32, padded to N.
 */

/* ResidualConv2dBlock.forward (modules.py:743-777), fused: y = x + ELU(W2 * ELU(W1 (*)_dilation x + b1) + b2),
 * as a warp-specialised, row-pipelined kernel (TMA row ring -> tcgen05 -> TMEM -> epilogue warps), in
 * row-stationary form: every input row meets the weights of all three vertical taps in one N = 3C MMA per horizontal tap (a third
 * of the shared-memory operand reads of one-MMA-per-tap); accumulators of the output rows are TMEM rings that start out holding
 * the fp32 bias.  c_real = un-padded channel count.  layout selects how memory maps to GEMM rows:
 *   0  C8 planar (B, C/8, H, T, 8), one frame per row                         weights packing.pack_res_rs
 *   1  packed (B, H, T, 4), a row = 2 frames x 4 channels (pass C = 8)        weights packing.pack_res_rs_pairs
 *   2  C8 planar with C = 8, folded: a row = 2 frames x 8 channels            weights packing.pack_res_rs_fold(..., fold=2)
 *   4  packed (B, H, T, 4), folded: a row = 4 frames x 4 channels (C = 8)     weights packing.pack_res_rs_fold(..., fold=4)
 * (folding makes every row 16 values wide, so the per-row hand-offs cover 2-4x more frames: the fast path for C <= 8).
 * w1 (KG1, 3 NC, 8), w2 (KG2, NC, 8) bf16 and bias (2, NC) fp32 with NC = accumulator columns per row (16, or 32 for C = 32). */
int tt_res_block_rs(const void* x, void* y, const void* w1, const void* w2, const float* bias, int B, int C, int c_real,
                    int H, int T, int dilation, int layout, void* stream);
/* The same launch, additionally writing the block's inner activation ELU(W1 * x + b1) to `mid` (layout and size of y; NULL = none):
   the loss step keeps it for the backward pass (the 3x3 data / weight gradients need ELU'(z1)) instead of recomputing the conv. */
int tt_res_block_rs_mid(const void* x, void* y, void* mid, const void* w1, const void* w2, const float* bias, int B, int C, int c_real,
                        int H, int T, int dilation, int layout, void* stream);
/* One 3x3 dilated 'same' conv (k = 3, weights packing.pack_res3x3) or 1x1 conv (k = 1, packing.pack_res1x1), optional ELU, on C8
 * planar tensors: building block of the backward pass (recompute + data gradients as convs with transformed weights) */
int tt_conv_same(const void* x, void* y, const void* w, const float* bias, int B, int C, int H, int T, int k, int dilation,
                 int act_elu, void* stream);
/* The same conv with one of the element-wise passes of the residual blocks' backward fused into its epilogue, on a tensor `e` of the
   output's shape and layout: post = 1: y = conv(x) * ELU'(e), e the ACTIVATED value (e > 0 ? 1 : e + 1); post = 2: y = conv(x) + e. */
int tt_conv_same_post(const void* x, void* y, const void* w, const float* bias, int B, int C, int H, int T, int k, int dilation,
                      int act_elu, int post, const void* e, void* stream);
/* EncoderBlock.sconv + ELU (modules.py:626-629): Conv2d(Cin, Cout, (4,1), stride (2,1)); Hout = (Hin-4)/2 + 1, and
 * DecoderBlock.tconv + ELU (modules.py:685-688): ConvTranspose2d(Cin, Cout, (4,1), stride (2,1), output_padding);
 * Hout = 2 Hin + 2 + out_pad - row-pipelined kernels (csrc/updown_strip.cu); weights from packing.pack_down_strip / pack_up_strip
 * (bias folded in).  Supported padded channel pairs: down 8->8, 8->16, 16->32, 32->64; up 64->32, 32->16, 16->8, 8->8. */
/* packed4_in / packed4_out = 1: the input (down, 4 -> 8 channels, weights from packing.pack_down_pairs) / the output (up, 8 -> 4
 * channels) is the packed 4-channel layout (B, H, T, 4) bf16; pass the padded channel counts 8 -> 8. */
/* Testing / tuning knob of the row-pipelined kernels (residual blocks, strided and transposed convs): force the number of image
 * rows (row groups) one CTA walks; 0 restores the automatic split.  Results do not depend on it (tests/test_conv_ops_gpu.py). */
int tt_set_strip_rows(int rows);
/* act_elu = 1: the model's layers (+ ELU); 0: linear - the same kernels as the data-gradient convolutions of the loss step (the data
 * gradient of a strided conv is a transposed conv and vice versa) */
int tt_conv_down_strip(const void* x, void* y, const void* w, int B, int Cin, int Cout, int Hin, int T, int packed4_in, int act_elu,
                       void* stream);
int tt_conv_up_strip(const void* x, void* y, const void* w, int B, int Cin, int Cout, int Hin, int out_pad, int T, int packed4_out,
                     int act_elu, void* stream);
/* Encoder.convlat (modules.py:446,478): Conv2d(C4, latent, (H4,1)), no activation; lat is C8 planar with H = 1 */
int tt_conv_lat(const void* x, void* lat, const void* w, const float* bias, int B, int C4, int H4, int NL, int T, void* stream);
/* Decoder.convin + ELU (modules.py:533-536) with TimbreTrap.decode's indicator channel (modules.py:139-142) folded into
 * the per-row bias table bias[H0][C0] (one table per switch setting); act_elu = 0: linear (the data gradient of Encoder.convlat) */
int tt_deconv_in(const void* lat, void* y, const void* w, const float* bias, int B, int Clat, int C0, int H0, int T, int act_elu,
                 void* stream);
/* Encoder.convin + ELU (modules.py:430-433): fp32 interleaved coefficients (B,F,T,2) -> C8 planar (packed4 = 0) or the packed
 * 4-channel layout (B,F,T,4) (packed4 = 1, C0 <= 4); w fp32 [C0][2][3][3].  packed4 = 2: packed output WITHOUT the ELU (the loss
 * step's data gradient of Decoder.convout) */
int tt_conv_in(const float* coeffs, void* y, const float* w, const float* bias, int B, int C0, int H, int T, int packed4, void* stream);
/* Decoder.convout (modules.py:543): C8 planar or packed 4-channel input -> fp32 interleaved coefficients (B,F,T,2); w fp32 [2][C][3][3] */
int tt_conv_out(const void* x, float* coeffs, const float* w, const float* bias, int B, int C, int H, int T, int packed4, void* stream);

/* Decoder.convout FUSED with the Hann cross-fade + trim of TimbreTrap.chunked_inference (modules.py:237-267) and, for act_out,
 * with TimbreTrap.to_activations (modules.py:271-289): the last decoder stage of ALL chunks in, cross-faded results out - the
 * per-chunk coefficients never exist in memory.
 *   x           (batch * n_chunks, H, M, 4) bf16 packed 4-channel layout - chunk i of item b at index b * n_chunks + i
 *   window      (M) fp32 device (torch.signal.windows.hann, modules.py:239);  w fp32 [2][C][3][3], bias fp32 [2]
 *   coeffs_out  (batch, H, (n_chunks-1) * M/2, 2) fp32 or NULL;  act_out (batch, H, (n_chunks-1) * M/2) fp32 or NULL */
int tt_conv_out_crossfade(const void* x, const float* window, const float* w, const float* bias, int batch, int n_chunks, int C,
                          int H, int M, float* coeffs_out, float* act_out, void* stream);

/* tt_conv_out_crossfade over the clips of clip_chunk0 (see tt_cqt_inverse_clips): x (total_chunks, H, M, 4) with total_chunks =
 * t[n] - t[0]; clip c's outputs (H, (n_c - 1) * M/2 [, 2]) follow those of the clips before it; max_chunks = the most of any clip */
int tt_conv_out_crossfade_clips(const void* x, const float* window, const float* w, const float* bias, const int* clip_chunk0,
                                int n_clips, int total_chunks, int max_chunks, int C, int H, int M, float* coeffs_out, float* act_out,
                                void* stream);

/*
 * ---- model variants and skip connections (modules.py:95-117, 568-589, 780-1075): single-pass element-wise kernels ----------
 */
/* out = x + (*scale) * e on bf16 tensors of one layout, n elements (multiple of 8): the decoder's skip connection with the learnable
 * weight of TimbreTrap.apply_skip_connections read from device memory; out may alias x */
int tt_add_scaled_bf16(const void* x, const void* e, const float* scale, void* out, int64_t n, void* stream);
/* *out = sum of a[i] * b[i] over two bf16 tensors of one layout (gradient of a skip connection's scalar weight in the loss step);
 * deterministic two-stage reduction through `scratch` (tt_dot_scratch_floats() floats) */
int tt_dot_scratch_floats(void);
int tt_dot_bf16(const void* a, const void* b, int64_t n, float* out, float* scratch, void* stream);
/* (x) -> interleaved (x, 0): a one-channel feature map (TimbreTrapMag / MagDB encoder input, modules.py:927-950, 1019-1031) in the
 * two-channel layout tt_conv_in reads */
int tt_widen_pairs(const float* x, int64_t n, float* out, void* stream);
/* n fp32 interleaved pairs (B, F, T, 2) -> C8 planar bf16 (B, 1, F, T, 8), channels 2..7 zero (operand of the weight-gradient GEMM) */
int tt_pairs_to_c8(const float* pairs, int64_t n, void* c8, void* stream);
/* channel 0 of n interleaved pairs through an output non-linearity: 0 identity, 1 relu (TimbreTrapMag.decode, modules.py:976),
 * 2 sigmoid (TimbreTrapMagDB.decode :1052), 3 tanh(relu(.)) (Mag decode + to_activations :996) */
int tt_channel0_activation(const float* pairs, int64_t n, int mode, float* out, void* stream);
/* its backward, for the loss step's one-channel tensors kept as pairs (x, 0): pairs_in = the n pre-activation pairs, gpairs_out = the
 * gradient of the output pairs (f(v0), 0) (channel 0 is read); gpairs_in = (g * f'(v0), 0), relu'(0) = 0.  Same modes; mode 0 is the
 * backward of taking channel 0 and of widening x -> (x, 0) */
int tt_channel0_activation_bwd(const float* pairs_in, const float* gpairs_out, int64_t n, int mode, float* gpairs_in, void* stream);

/*
 * ---- audio front-end and evaluation metric on the device (SURVEY.md section 8f-3 / 8f-4) -----------------------------------
 */
/* AudioDataset.get_audio after the file read (datasets/AudioDataset.py:69-77): mono mix (mean over channels) + band-limited
 * polyphase resampling (torchaudio.functional.resample) in one pass; *peak receives max|out| (zeroed by the call) for the
 * infinity-norm normalise, which is tt_scale_by_peak(out, n_out, peak).
 *   audio   (channels, n_in) fp32 device, channel-major as torchaudio.load returns it
 *   kernel  (new_f, 2*width + orig) fp32 device: the windowed-sinc filter of every output phase (orig, new_f already divided by
 *           their gcd; table from timbre_trap_b200/framework/frontend.py::sinc_resample_kernel); orig == new_f == 1 with the
 *           one-tap kernel {1} is the plain mono mix
 *   out     (n_out) fp32, n_out = ceil(new_f * n_in / orig) */
int tt_resample_mono(const float* audio, int channels, int64_t n_in, const float* kernel, int orig, int new_f, int width,
                     float* out, int64_t n_out, float* peak, void* stream);
/* PitchDataset.multi_pitch_to_activations (datasets/PitchDataset.py:233-307): pitches_hz (T, P) fp64 device, 0 = no pitch;
 * midi_freqs (F) fp64 device (ascending); blur (2R+1) fp32 device = the normalised Gaussian taps (R = 0, {1}: no blur);
 * activations (F, T) fp32 out; min_scratch one device float */
int tt_rasterise_pitches(const double* pitches_hz, int T, int P, const double* midi_freqs, int F, const float* blur, int R,
                         float* activations, float* min_scratch, void* stream);
/* The O(N) part of the signal-to-distortion ratio the reference's evaluation reports (experiments/evaluate.py:51,122-127,
 * torchmetrics SignalDistortionRatio, filter_length 512): per item the first `lags` auto-correlation values of target,
 * r0[l] = sum_n t[n] t[n+l], the cross-correlation b[l] = sum_n t[n] p[n+l], and the two squared norms (|t|^2, |p|^2), all
 * accumulated in fp64.  target, preds (batch, n) fp32; r0, b (batch, lags) fp64; norms (batch, 2) fp64 (all zeroed by the call). */
int tt_sdr_correlations(const float* target, const float* preds, int batch, int64_t n, int lags, double* r0, double* b,
                        double* norms, void* stream);

/*
 * ---- objectives (timbre_trap/framework/objectives.py), deterministic two-stage reductions ------------------------
 * scratch: tt_loss_scratch_floats() floats of device memory.
 */
int tt_loss_scratch_floats(void);
/* compute_reconstruction_loss / compute_consistency_loss (objectives.py:11-33, 77-104): *out = scale * sum((a-b)^2);
 * the caller passes scale = 1 / (B*T) (sum over C and F, mean over B and T).  a, b: same memory order, n floats. */
int tt_sum_sq_diff(const float* a, const float* b, int64_t n, double scale, float* out, float* scratch, void* stream);
/* compute_transcription_loss (objectives.py:36-74): estimate, target (B, F, T) contiguous fp32 */
int tt_transcription_loss(const float* estimate, const float* target, int B, int F, int T, int weight_positive_class,
                          float* out, float* scratch, void* stream);

/*
 * ---- backward half of the loss step (experiments/train.py:470-496) ---------------------------------------------------
 * Tensor-core weight gradients of the residual blocks' 'same' convolutions, straight from the inference layouts: x, dz C8 planar bf16
 * (B, C/8, H, T, 8) with the PADDED channel counts Cin / Cout (8, 16 or 32); dw (cout_real, cin_real, k, k) fp32 and db (cout_real)
 * fp32 (db may be NULL) are ACCUMULATED into.  k = 3 (dilation 1..3, zero padding = dilation) or k = 1.  The GEMM's K axis is the
 * pixel axis: both operands are MN-major tcgen05 operands read from the rows the TMA brings in; per-CTA partial sums go through
 * `scratch` (tt_wgrad_scratch_floats(B, H, T) floats) and are reduced in a fixed order (bit-reproducible).
 */
int64_t tt_wgrad_scratch_floats(int B, int H, int T);
int tt_conv_wgrad_same(const void* x, const void* dz, float* dw, float* db, int B, int Cin, int Cout, int cin_real, int cout_real,
                       int H, int T, int k, int dilation, float* scratch, void* stream);
/* The same GEMM for the (4,1) / stride (2,1) layers: `coarse` (B, Ccoarse/8, Hcoarse, T, 8) row q meets `fine` (B, Cfine/8, Hfine, T, 8)
 * rows 2q .. 2q+3.  EncoderBlock.sconv (modules.py:626-629): fine = layer input, coarse = output gradient, dw (ccoarse_real, cfine_real, 4, 1),
 * db (ccoarse_real), transposed = 0.  DecoderBlock.tconv (modules.py:685-688): coarse = layer input, fine = output gradient, dw in the
 * ConvTranspose2d layout (ccoarse_real, cfine_real, 4, 1), db (cfine_real) = pixel sums of `fine`, transposed = 1.  Accumulating. */
int tt_conv_wgrad_updown(const void* fine, const void* coarse, float* dw, float* db, int B, int Cfine, int Ccoarse, int cfine_real,
                         int ccoarse_real, int Hfine, int Hcoarse, int T, int transposed, float* scratch, void* stream);
/* ... and for the two (H, 1)-kernel layers between the 31-row embedding and the latents: `tall` (B, Ctall/8, H, T, 8), `flat`
 * (B, Cflat/8, 1, T, 8); dw (cflat_real, ctall_real, H, 1) += sum over (b, t) of flat[m] * tall[n, h]; db (cflat_real) += pixel sums
 * of `flat` (may be NULL); tall_row_sums (ctall_real, H) += sums over (b, t) of `tall` (may be NULL).  Encoder.convlat
 * (modules.py:446): tall = layer input, flat = output gradient, dw is the Conv2d weight gradient.  Decoder.convin (:533-536):
 * flat = latents, tall = output gradient (after the ELU derivative): dw = rows 0 .. D-1 of the ConvTranspose2d weight gradient,
 * tall_row_sums = its indicator row (times the indicator) and, summed over H, the bias gradient.  scratch:
 * tt_wgrad_lat_scratch_floats(B, H, T) floats. */
int64_t tt_wgrad_lat_scratch_floats(int B, int H, int T);
int tt_conv_wgrad_lat(const void* tall, const void* flat, float* dw, float* db, float* tall_row_sums, int B, int Ctall, int Cflat,
                      int ctall_real, int cflat_real, int H, int T, float* scratch, void* stream);
/* element-wise pieces of the backward pass on bf16 tensors of any common layout (n elements, multiple of 8):
 * dz = gy * ELU'(z) through the activated output a;  residual block: dz = gy * ELU'(z2) with the activated 1x1 output = y - x */
int tt_elu_bwd_bf16(const void* gy, const void* a, void* dz, int64_t n, void* stream);
int tt_res_out_bwd_bf16(const void* gy, const void* y, const void* x, void* dz, int64_t n, void* stream);
/* packed 4-channel (B, H, T, 4) <-> C8 planar with one channel group (B, 1, H, T, 8), n_pixels = B * H * T */
int tt_p4_to_c8(const void* p4, void* c8, int64_t n_pixels, void* stream);
int tt_c8_to_p4(const void* c8, void* p4, int64_t n_pixels, void* stream);
/* gradients of tt_sum_sq_diff and tt_transcription_loss (both arguments; either output may be NULL), tanh|c| */
int tt_sum_sq_diff_bwd(const float* a, const float* b, const float* gout, double scale, float* ga, float* gb, int64_t n, void* stream);
int tt_transcription_loss_bwd(const float* estimate, const float* target, const float* gout, int B, int F, int T,
                              int weight_positive_class, float* gest, float* gtarget, void* stream);
int tt_activations_bwd(const float* coeffs, const float* dact, float* dcoeffs, int64_t n, void* stream);
/* TimbreTrapFiLM's Decoder.convin (modules.py:801-809, 838-840): ConvTranspose2d(D, C0, (H0, 1)) on gamma * z + beta, with
 * gamma / beta = film_layer.gamma / .beta of the one-hot condition whose 1 is in column `hot` (0 transcribe, 1 reconstruct).
 * G (D, C0, H0) and rows (C0, H0) are tt_conv_wgrad_lat's dw and tall_row_sums for flat = latents z, tall = output gradient dz;
 * w (D, C0, H0) the weight, gamma_w / beta_w (D, 2), gamma_b / beta_b (D) the Linear parameters.  WRITES dw = gamma G + beta rows,
 * db (C0) = sum_h rows, and the Linear gradients dgamma_w / dbeta_w (D, 2) (column hot = <W[d], G[d]> / <W[d], rows>, the other 0),
 * dgamma_b / dbeta_b (D).  One CTA per latent channel, fixed-order reductions (bit-reproducible). */
int tt_film_convin_grad(const float* G, const float* rows, const float* w, const float* gamma_w, const float* gamma_b,
                        const float* beta_w, const float* beta_b, int D, int C0, int H0, int hot, float* dw, float* db,
                        float* dgamma_w, float* dgamma_b, float* dbeta_w, float* dbeta_b, void* stream);
/* clip_grad_norm_ + AdamW (train.py:493-496): accumulate sum g^2 of every gradient tensor into *acc (double, zeroed by the
 * caller), then one tt_adamw_step per tensor applies the common clip factor min(1, max_norm / (norm + 1e-6)) and the update */
int tt_grad_sumsq(const float* g, int64_t n, double* acc, void* stream);
int tt_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, const double* sumsq, float max_norm, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif
