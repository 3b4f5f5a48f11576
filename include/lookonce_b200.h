/* lookonce_b200.h -- C ABI of the B200-native LookOnceToHear inference engine.
 *
 * Drop-in boundary for ONE path of vb000/LookOnceToHear: the inference forward of its two
 * networks.  The reference is pure Python; the interface each entry point stands in for is the
 * Python method the reference's evaluation path calls (all paths relative to /root/reference):
 *
 *   l2h_sep_create / l2h_sep_load_weight / l2h_sep_commit_weights
 *        <- Net.__init__ + load_state_dict      src/models/tfgridnet_realtime/net.py:20-49,
 *                                               src/ts_hear_test.py:18-34 (load_model)
 *   l2h_sep_state_bytes / l2h_sep_state_init
 *        <- Net.init_buffers                    net.py:51-52, tfgridnet_causal.py:173-186,408-427
 *   l2h_sep_forward
 *        <- Net.predict / Net.forward           net.py:54-76  -> TFGridNet.forward
 *                                               tfgridnet_causal.py:188-283
 *   l2h_sep_stream_host
 *        <- the chunk loop around Net.predict(chunk, embed, state, pad=False)  (SURVEY.md 3.3)
 *           with host buffers: H2D of each chunk and D2H of each result inside the call
 *   l2h_embed_create / l2h_embed_load_weight / l2h_embed_commit_weights / l2h_embed_forward
 *        <- EmbedTFGridNet.__init__/forward     src/models/tfgridnet_orig/tfgridnet.py:88-127
 *
 * Conventions follow the reference's only FFI (src/datasets/motion_simulator.py:30-95): every
 * function returns int (0 = OK, non-zero = error, text via l2h_last_error()), handles are opaque
 * void*, buffers are plain float pointers + sizes, explicit *_destroy.  No torch types.  Device
 * pointers are CUDA device memory of the current device; `stream` is a cudaStream_t passed as
 * void* (NULL = default stream).  Nothing synchronises the stream except where stated.
 * One handle per device; a handle is not thread-safe.
 */
#ifndef LOOKONCE_B200_H
#define LOOKONCE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define L2H_ABI_VERSION 1

/* configs/tsh.json:5-19 -> Net(**model_params) */
typedef struct l2h_sep_config {
    int32_t stft_chunk_size; /* 128 */
    int32_t stft_pad_size;   /* 64  */
    int32_t embed_dim;       /* 256 */
    int32_t num_ch;          /* 2   */
    int32_t D;               /* 64  */
    int32_t L;               /* 4 heads */
    int32_t I;               /* 1   */
    int32_t J;               /* 1   */
    int32_t B;               /* number of GridNet blocks (3) */
    int32_t H;               /* 64  */
    int32_t local_atten_len; /* 50  */
    int32_t use_attn;        /* 1   */
    int32_t lookahead;       /* 1   */
    int32_t chunk_causal;    /* 1   */
    int32_t num_src;         /* 2   */
} l2h_sep_config;

/* flags for l2h_sep_forward */
#define L2H_FLAG_TAPS 1u  /* also copy the activations after every stage into the tap area */
#define L2H_FLAG_GRAPH 2u /* replay the kernel chain from a CUDA graph cached on the exact argument set
                             (pointers, strides, sizes): for callers that reuse fixed staging buffers */

int l2h_abi_version(void);
const char* l2h_last_error(void);

/* ---- separation network -------------------------------------------------------------------- */
int l2h_sep_create(const l2h_sep_config* cfg, void** handle);
int l2h_sep_destroy(void* handle);

/* name = a key of the reference state_dict without the Lightning "model." prefix, e.g.
 * "tfgridnet.blocks.0.intra_rnn.weight_ih_l0"; data = HOST fp32, contiguous, numel elements.
 * Repacks into the engine's layouts in a host staging buffer.  Unknown names -> error 2. */
int l2h_sep_load_weight(void* handle, const char* name, const float* host_data, int64_t numel);
/* number of reference tensors the engine expects / has received so far */
int l2h_sep_weights_expected(void* handle, int32_t* n_expected, int32_t* n_loaded);
/* the index-th expected tensor (0 <= index < n_expected, alphabetical): its reference name (owned by the handle) and
 * element count -- what a host that converts a checkpoint iterates over (examples/stream_clip.cpp) */
int l2h_sep_weight_info(void* handle, int32_t index, const char** name, int64_t* numel);
/* upload the staged weights (one H2D of ~8 MB on `stream`, then synchronises it) */
int l2h_sep_commit_weights(void* handle, void* stream);

int l2h_sep_state_bytes(void* handle, int32_t batch, size_t* bytes);
int l2h_sep_state_init(void* handle, void* state_dev, int32_t batch, void* stream);
/* floats per stream record and header bytes, for host code that builds views of the state */
int l2h_sep_state_layout(void* handle, int64_t* header_bytes, int64_t* stream_stride_floats);
/* The offsets (in floats) inside one stream record, for host code that converts to / from the reference's nested
 * state dict (tfgridnet_causal.py:173-186, :408-427) -- SepState.to_reference() / load_reference().  out[i]:
 * 0 ring slots per head, 1 K row stride, 2 K row length (582), 3 V row length (1552), 4 attention window (50),
 * 5 embedding copy, 6 cached speaker gate, 7 conv tail, 8 deconv tail, 9 iSTFT tail, 10 first block, then inside a
 * block: 11 K ring, 12 V ring, 13 h, 14 c, 15 block stride. */
#define L2H_STATE_OFFSETS 16
int l2h_sep_state_offsets(void* handle, int64_t* out, int32_t n);

int l2h_sep_workspace_bytes(void* handle, int32_t batch, int32_t frames, uint32_t flags, size_t* bytes);

/* One call = `frames` hops of 128 samples for `batch` independent streams.
 *   x_dev   [batch][num_ch][*]  fp32, strides in floats; samples at index >= x_len read as zero
 *           (this is where net.py's mod-pad and look-ahead zero padding happen)
 *   emb_dev [batch][256]
 *   y_dev   [batch][num_src][*] fp32; samples 0 .. min(y_len, 128*frames)-1 are written
 * The state is advanced in place.  Asynchronous on `stream`. */
int l2h_sep_forward(void* handle, const float* x_dev, int64_t x_batch_stride, int64_t x_ch_stride,
                    int32_t x_len, const float* emb_dev, void* state_dev, float* y_dev,
                    int64_t y_batch_stride, int64_t y_ch_stride, int32_t y_len, int32_t batch,
                    int32_t frames, void* workspace_dev, size_t workspace_bytes, uint32_t flags,
                    void* stream);

/* Streaming with HOST buffers (the end-to-end path).  Per round: H2D of the round's samples (+64
 * look-ahead) from pinned memory, the kernel chains, D2H of the new samples; one stream synchronise at
 * the end.  A round is one call of chunks_per_call hops -- or, for chunks_per_call == 1 with pipelining
 * enabled, a group of up to l2h_sep_pipeline_frames() one-hop calls that run as one wavefront-pipelined
 * graph (every hop is still its own T=1 chain with the state carried hop to hop).
 * x_host [batch][num_ch][x_len], y_host [batch][num_src][y_len]; x_stage_dev / y_stage_dev must hold
 * [batch][ch][128*G + 64] / [batch][src][128*G] floats with G = max(chunks_per_call, pipeline frames);
 * workspace from l2h_sep_stream_workspace_bytes(). */
int l2h_sep_stream_host(void* handle, const float* x_host, int32_t x_len, const float* emb_dev,
                        void* state_dev, float* y_host, int32_t y_len, int32_t batch,
                        int32_t n_calls, int32_t chunks_per_call, float* x_stage_dev,
                        float* y_stage_dev, void* workspace_dev, size_t workspace_bytes,
                        void* stream);

/* Streaming with DEVICE buffers: x_dev [batch][num_ch][x_len] holds whole clips, y_dev
 * [batch][num_src][y_len]; n_calls chained calls of chunks_per_call frames each, starting at the
 * beginning of x_dev and continuing the state.  Calls are CUDA-graph replays; the chunk a replay
 * works on is derived on the device from the state's frame counter.  With chunks_per_call == 1 the
 * one-hop chains of up to l2h_sep_pipeline_frames() consecutive hops are captured as ONE graph on 8
 * streams with (block, frame) wavefront dependencies, so different blocks work on different hops
 * concurrently (set L2H_PIPE=0 to run the hops strictly one after the other).  Asynchronous. */
int l2h_sep_stream_dev(void* handle, const float* x_dev, int32_t x_len, const float* emb_dev,
                       void* state_dev, float* y_dev, int32_t y_len, int32_t batch, int32_t n_calls,
                       int32_t chunks_per_call, void* workspace_dev, size_t workspace_bytes, void* stream);

/* workspace for the two streaming entry points (one slot per in-flight hop when pipelining) and the
 * number of one-hop calls a pipelined graph holds (1 = pipelining off) */
int l2h_sep_stream_workspace_bytes(void* handle, int32_t batch, int32_t chunks_per_call, size_t* bytes);
int l2h_sep_pipeline_frames(void* handle, int32_t* frames);
/* runtime switches (the only way to change them: there are no environment variables).  0 | 1: "pipeline" (wavefront graph for
 * streams of one-hop calls), "pdl", "fused_mid", "fused_tail" (one-hop calls of a few streams as 8 launches: front1_kernel, per block
 * the BiLSTM and the 16-CTA tail_kernel; default 1), "back_many" (calls of several frames / many streams through the persistent
 * front_many / back_many kernels; default 1), "pipeline_split_mid" (mid section as mid_a | mid_b | mid_c in the graph),
 * "mid_split_large" (the same three kernels for many streams), "fold_mid_c" (default 0: no mid_c -- the inter Linear moves into
 * the serial kernel, the Q/K/V projection into qkv_kernel; changes rounding, not the maths; measured slower, tested),
 * "tensor_cores" (default 1), "fuse_ih" (default 0), "graph_stats".  Values: "bf16" (0 = bf16x3 split products, 1 = bf16 weights x
 * split activations, 2 = plain bf16), "tc_lstm_min" (sequence-directions from which the recurrence runs on the tensor cores,
 * default 4096), "tc_pdl" (bit mask, default 7: programmatic launches around the tensor-core GEMMs of many-row chains),
 * "pipeline_gemm_shape" (0 | 1 | 2).  Counts: "pipeline_frames" (hops per graph, <= 500; 0 = as many as the workspace budget
 * holds), "pipeline_midb_hops" (hops per launch of the serial stage, <= 8) and the hops in flight per stage: "pipeline_lanes"
 * (BiLSTM, <= 16), "pipeline_midc_lanes" (<= 3), "pipeline_qkv_lanes" (<= 4), "pipeline_attn_lanes" (<= 4),
 * "pipeline_out_lanes" (<= 4), "pipeline_front_lanes" (<= 8), "pipeline_back_lanes" (<= 6).  Bit masks over the stages
 * front=1, W_ih gemm=2, bilstm=4, mid_a=8, mid_b=16, mid_c=32, qkv=64, attention=128, attn_out=256, back=512:
 * "pipeline_pdl" (stages launched with programmatic dependent launch; default 16) and "pipeline_debug_skip" (stages NOT
 * launched -- timing experiments only, the output is garbage).  "defaults" restores all pipeline settings.  The pipeline
 * settings never change results (bit-identical, tests/test_sep_gpu.py); "fused_tail", "fold_mid_c", "bf16", "fuse_ih" and the
 * tensor-core switches change rounding only (gates in tests/). */
int l2h_sep_set_option(void* handle, const char* name, int32_t value);

/* where the tap area starts inside the workspace (floats) and its stage count; stage s holds
 * [batch*frames*97*64] floats: 0 = encoder out, then per block: after intra, after inter, block out */
int l2h_sep_tap_info(void* handle, int32_t batch, int32_t frames, int64_t* offset_floats,
                     int32_t* n_stages);

/* Measurement aid: run the chain `iters` times (after 2 warm-ups) with a CUDA event between every
 * launch on `stream`; returns, per kernel name (<= 64), the summed device time in ms and the launch
 * count.  Advances the state by (iters+2)*frames.  Synchronises. */
int l2h_sep_profile(void* handle, const float* x_dev, int32_t x_len, const float* emb_dev, void* state_dev,
                    float* y_dev, int32_t batch, int32_t frames, void* workspace_dev, size_t workspace_bytes,
                    int32_t iters, const char** names, float* ms_total, int32_t* counts, int32_t* n_names,
                    void* stream);

/* number of kernels one l2h_sep_forward of `frames` hops launches at a few streams (see l2h_sep_launch_count for the
   exact count of everything a handle launched, pipelined streams included) */
int l2h_sep_launches_per_forward(void* handle, int32_t frames, int32_t* n);

/* kernels this handle has launched so far (a CUDA-graph replay counts its kernel nodes); reset != 0 zeroes the
   counter after reading.  bench.py's gpu_launches is read from here around the timed region. */
int l2h_sep_launch_count(void* handle, int64_t* kernels, int32_t reset);

/* diagnostics: device-side timeline of the separator's kernels.  l2h_sep_trace_start(handle, capacity) allocates a buffer
   of `capacity` records and switches tracing on (capacity 0: off); from then on thread 0 of the first CTA of every
   instrumented kernel stores one 32-byte record {u64 t0_ns, u64 t1_ns (globaltimer at entry / exit), u64 activation
   pointer, u32 kernel id (0 front, 1 W_ih gemm, 2 bilstm, 3 mid_a, 4 mid_b, 5 mid_c, 6 qkv, 7 attention, 8 attn_out,
   9 back, 10 fused mid), u32 SM}.  l2h_sep_trace_read synchronises, copies up to max_records of them to the host and
   restarts the trace.  Used by tools/pipe_trace.py; costs one atomic per kernel while on, one load while off. */
int l2h_sep_trace_start(void* handle, int32_t capacity);
int l2h_sep_trace_read(void* handle, void* records_host, int32_t max_records, int32_t* n_records);

/* ---- enrollment network (EmbedTFGridNet, configs/embed.json:5-10) ---------------------------- */
typedef struct l2h_embed_config {
    int32_t embed_dim;  /* 256 */
    int32_t num_ch;     /* 2   */
    int32_t n_fft;      /* 128 */
    int32_t stride;     /* 64  */
    int32_t num_blocks; /* 3   */
} l2h_embed_config;

int l2h_embed_create(const l2h_embed_config* cfg, void** handle);
int l2h_embed_destroy(void* handle);
/* name = a key of the reference EmbedTFGridNet state_dict (espnet2 naming: "blocks.0.intra_norm.gamma",
 * "blocks.0.attn_conv_Q_0.0.weight", "embed_proj.0.weight", ...); HOST fp32.  The unused deconv.* tensors
 * are accepted and ignored. */
int l2h_embed_load_weight(void* handle, const char* name, const float* host_data, int64_t numel);
int l2h_embed_weights_expected(void* handle, int32_t* n_expected, int32_t* n_loaded);
int l2h_embed_commit_weights(void* handle, void* stream);
int l2h_embed_workspace_bytes(void* handle, int32_t batch, int32_t n_samples, size_t* bytes);
/* "bf16" = 1: the tensor-core GEMMs take plain bf16 operands (one MMA pass); 0 (default): every product is formed from
 * bf16 hi/lo splits of both fp32 operands in three MMA passes (fp32-grade, relative error ~2^-16 per product). */
int l2h_embed_set_option(void* handle, const char* name, int32_t value);
/* largest batch one l2h_embed_forward call should be given for utterances of n_samples (workspace bound) */
int l2h_embed_max_batch(void* handle, int32_t n_samples, int32_t* max_batch);
/* x_dev [batch][2][n_samples] fp32 contiguous -> emb_dev [batch][256].  Asynchronous on `stream`. */
int l2h_embed_forward(void* handle, const float* x_dev, float* emb_dev, int32_t batch, int32_t n_samples,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation epilogue on the device (replaces the CPU metric code after `outputs.cpu()` in
 * src/ts_hear_test.py:139-146): per mixture b, out_dev[b] = { output_sisnr, si_snr_i, embedding_sim }
 *   output_sisnr  = mean over channels of SI-SNR(est, target)                 (torchmetrics definition, zero-mean)
 *   si_snr_i      = mean over channels of SI-SNR(est, target) - SI-SNR(mixture, target)   (0 if mixture_dev is NULL)
 *   embedding_sim = cosine similarity of emb and emb_gt                        (0 if either is NULL)
 * est / target / mixture: [batch][channels][n_samples] fp32 contiguous on the device (est = the separator's output
 * buffer); emb / emb_gt: [batch][emb_dim].  Asynchronous on `stream`; the caller copies 3 floats per mixture back. */
int l2h_eval_metrics(const float* est_dev, const float* target_dev, const float* mixture_dev, int32_t batch, int32_t channels,
                     int32_t n_samples, const float* emb_dev, const float* emb_gt_dev, int32_t emb_dim, float* out_dev,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * Binaural rendering of mono events on the device (the data-side arithmetic of the reference's simulators):
 *   events[b][s][ear] = convolve(src[b][s], rir[b][s][ear])[:n_samples]      src/datasets/multi_ch_simulator.py:56-58
 *   noise scaled by noise_scale[b]; norm = max|sum(events) + noise|; if norm > 1 events and noise are divided by it;
 *   mixture = sum(events) + noise                                   src/datasets/MixLibriSpeechNoisyEnrollNorm.py:179-202
 * src_dev [batch][n_src][n_samples] mono; rir_dev [batch][n_src][2][rir_len] (already at the sampling rate of src);
 * noise_dev [batch][2][n_samples] or NULL; noise_scale_dev [batch] or NULL (= 1); events_dev [batch][n_src][2][n_samples];
 * mixture_dev [batch][2][n_samples]; norm_dev [batch] or NULL; scratch_dev: batch * 4 bytes.  Asynchronous on `stream`. */
int l2h_render_binaural(const float* src_dev, const float* rir_dev, const float* noise_dev, const float* noise_scale_dev,
                        int32_t batch, int32_t n_src, int32_t n_samples, int32_t rir_len, float* events_dev,
                        float* mixture_dev, float* norm_dev, void* scratch_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Binaural cue errors on the device (src/eval/binaural.py:6-149): per mixture b,
 * out_dev[b] = { ild_diff (dB), itd_diff (microseconds) } of est against gt, both [batch][2][n_samples] fp32 contiguous,
 * ear 0 = left.  Windows of `frame` samples, the last zero-padded past n_samples (chunk_and_mask :6-42); frame = 0 is one
 * window of the whole signal (the static form).  Per window:
 *   ILD = 10 log10(sum left^2 / sum right^2)                                                    compute_ild :44-47
 *   ITD = tau / sr * 1e6, tau = first argmax over k in [-t, t] of |sum_n left[(n+k) mod L] right[n]|,
 *         t = min(t_max, L/2), L = the window length                          axiswise_xcorr :83-92, compute_itd :94-117
 *   valid = max over ears of sqrt(mean(gt^2)) >= rms_threshold (frame > 0 only; every static window is valid)
 * Per mixture: ild_diff = |mean_valid ild_est - mean_valid ild_gt|, itd_diff = mean_valid |itd_est - itd_gt|
 * (ild_diff :62-81, itd_diff :134-147; with one window these are the static |differences|).  Non-finite results are
 * the reference's: a silent ear gives +-inf or NaN ILD, a mixture without a valid window NaN.
 * The caller passes the reference's integers: frame = round(0.25 sr), t_max = round(1e-3 sr) (Python rounding).
 * t_max = 0 computes ILD only (itd entries are NaN).  Refused: t_max > 256, and t_max > 0 with an odd window length
 * (the reference's irfft drops a sample there, its "correlation" is not one).
 * windows_dev [batch][n_windows][5] = { ild_est, ild_gt, itd_est, itd_gt, valid (0/1) } or NULL,
 * n_windows = frame ? 1 + (n_samples - 1) / frame : 1.  workspace_dev: l2h_eval_binaural_workspace_bytes() bytes on the
 * device.  Asynchronous on `stream`, no allocation, no host synchronisation; fixed-order sums (bit-reproducible). */
int l2h_eval_binaural_workspace_bytes(int32_t batch, int32_t n_samples, int32_t frame, int32_t t_max, size_t* bytes);
int l2h_eval_binaural(const float* est_dev, const float* gt_dev, int32_t batch, int32_t n_samples, int32_t frame,
                      int32_t t_max, double rms_threshold, int32_t sr, float* out_dev, float* windows_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LOOKONCE_B200_H */
