/*
 * fq3.h — C ABI of the B200-native Qwen3-TTS decode engine (libfq3.so).
 *
 * This is the drop-in boundary for the hot path of andimarafioti/qwen3-tts-cuda-graphs
 * (reference = /root/reference, Python, no native code).  Every entry point replaces one seam of the
 * reference's L2/L3 operators (SURVEY.md §8b); the reference file:line each one stands in for is cited.
 * Plain pointers and sizes only — no torch types.  All device pointers are CUDA device addresses on the
 * current device; `stream` is a cudaStream_t passed as void*.  Every call returns 0 on success or a
 * negative fq3 error code; fq3_last_error() returns the message of the last failure on this thread.
 *
 * The library fails loudly: there is no CPU path behind any of these symbols.
 */
#ifndef FQ3_H_
#define FQ3_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FQ3_ABI_VERSION 2
#define FQ3_MAX_CODE_GROUPS 32

typedef struct fq3_engine fq3_engine; /* opaque */

/* One dense Qwen3 decoder stack laid out in the weight arena (bf16, byte offsets, 16-byte aligned).
 * layer_offs holds n_layers * 8 offsets in this order:
 *   0 input_layernorm [H]      1 wqkv [(nq+2nkv)*d, H]  (q rows, then k rows, then v rows)
 *   2 q_norm [d]               3 k_norm [d]              4 wo [H, nq*d]
 *   5 post_attention_layernorm [H]
 *   6 wgu [2*I, H]  (row 2j = gate_j, row 2j+1 = up_j)   7 wdown [H, I]                          */
typedef struct fq3_stack_desc {
  int32_t hidden, inter, n_layers, n_q_heads, n_kv_heads, head_dim, vocab;
  float rms_eps;
  const uint64_t* layer_offs;
  uint64_t final_norm_off;
  uint64_t rope_cos_off, rope_sin_off; /* bf16 [rope_len, head_dim] tables (HF rotary, all mrope axes equal) */
  int32_t rope_len;
  int32_t max_pos; /* KV capacity per stream: talker max_seq_len (talker_graph.py:43), predictor 17 (predictor_graph.py:46) */
} fq3_stack_desc;

typedef struct fq3_model_desc {
  int32_t abi_version;
  const void* arena; /* device pointer, all weights the kernels touch */
  uint64_t arena_bytes;
  fq3_stack_desc talker, predictor;
  uint64_t codec_head_off;  /* [V_t, H_t]   generate.py:182 */
  uint64_t codec_embed_off; /* [V_t, H_t]   generate.py:154 */
  int32_t n_code_groups;    /* 16 */
  const uint64_t* lm_head_offs;    /* n_code_groups-1 x [V_p, H_p]  predictor_graph.py:131,157 */
  const uint64_t* pred_embed_offs; /* n_code_groups-1 x [V_p, H_t]  predictor_graph.py:144, generate.py:163-166 */
  int32_t has_s2m;                 /* small_to_mtp_projection present (predictor_graph.py:118,145) */
  uint64_t s2m_w_off, s2m_b_off;   /* [H_p, H_t], [H_p] */
  int32_t eos_id;                  /* config.codec_eos_token_id (generate.py:41) */
  int32_t max_streams;             /* independent utterances decoded in lock-step (1 = the reference's bs=1) */
  int32_t max_frames;              /* capacity of the per-stream codes buffer */
} fq3_model_desc;

/* Sampling policy of the first-codebook sampler (generate.py:184-197, sampling.py:32-66). */
typedef struct fq3_policy {
  int32_t do_sample;
  int32_t top_k;
  float top_p;
  float temperature;
  float repetition_penalty;
  int32_t min_new_tokens;
  int32_t suppress_tail; /* ids in [V-suppress_tail, V) except eos are -inf (generate.py:46-50); 1024 */
  uint64_t seed;
} fq3_policy;

/* Sampling policy of codebooks 1..15, frozen at capture time in the reference (predictor_graph.py:34-50). */
typedef struct fq3_subpolicy {
  int32_t do_sample;
  int32_t top_k;
  float top_p;
  float temperature;
} fq3_subpolicy;

/* Host-visible per-stream status after fq3_decode_frames (streaming.py:157-188 needs steps + is_final). */
typedef struct fq3_status {
  int32_t n_frames;  /* frames appended so far for this utterance */
  int32_t done;      /* 0 running, 1 EOS sampled (generate.py:150), 2 static cache full (generate.py:175-177), 3 retired by the host,
                        4 waiting for text (fq3_open_text): not finished, resumes after fq3_append_text */
  int32_t position;  /* next KV position */
  int32_t gen_step;  /* generate.py:199 */
  int32_t token;     /* first-codebook id that will open the next frame */
  int32_t error;     /* device-side watchdog / protocol error code, 0 = none */
} fq3_status;

/* ---- lifetime ------------------------------------------------------------------------------ */
int fq3_abi_version(void);
const char* fq3_last_error(void);
/* Replaces TalkerGraph.__init__/capture + PredictorGraph.__init__/capture (talker_graph.py:27-147,
 * predictor_graph.py:34-202): allocates static KV caches and activation buffers, builds the phase
 * programs.  Nothing is captured lazily; the first call after create is already the steady state. */
int fq3_create(const fq3_model_desc* desc, fq3_engine** out);
int fq3_destroy(fq3_engine* e);
/* CTAs of the engine's persistent grid (one per SM; 128 by default, env FQ3_GRID overrides at create time) */
int fq3_num_sms(const fq3_engine* e);
/* number of kernel launches issued by this engine since creation (bench.py "gpu_launches") */
int64_t fq3_launch_count(const fq3_engine* e);

/* ---- per-utterance set-up ------------------------------------------------------------------ */
/* TalkerGraph.reset (talker_graph.py:149-151): forget KV, history, frame count of one stream.  Also clears the stream's
 * sampling policy record (fq3_set_stream_policy). */
int fq3_reset_stream(fq3_engine* e, int stream_idx, void* stream);
/* Serving (no counterpart in the reference): a stream's own sampling policy, so that requests with different sampling
 * arguments share one lock-step launch.  While a stream has a record, fq3_prefill / fq3_prefill_tail / fq3_prefill_head
 * (first-token sample) and fq3_decode_frames (any n_streams, both frame programs, every lock-step group) sample that stream
 * with the record instead of the `policy` argument: do_sample, top_k, top_p, temperature, repetition_penalty, min_new_tokens
 * (both EOS-suppression rules), suppress_tail and seed for the first codebook; for codebooks 1..15 the seed only (their
 * arguments stay the launch's fq3_subpolicy, frozen at capture time in the reference, predictor_graph.py:34-50).  The Philox
 * key of such a stream is seed ^ K * 1 whatever its slot — the key slot 0 gets under a launch-wide policy with the same seed —
 * so its draws depend only on its own seed and draw counter, and it draws exactly what a single-stream run in slot 0 with a
 * launch-wide policy of the same values draws.  Streams without a record sample exactly as before.  fq3_talker_step,
 * fq3_predictor_run and fq3_sample take their arguments explicitly and ignore the record.
 * Stream-ordered (the record is written by a kernel on `stream`; `policy` may be freed when the call returns).
 * policy == NULL clears the record.  The record survives the reset a prefill runs internally; fq3_reset_stream clears it.
 * -FQ3_E_INVALID for an index out of range, top_k < 0, top_p outside (0, 1], temperature <= 0 with do_sample,
 * repetition_penalty <= 0, suppress_tail outside [0, V_t]. */
int fq3_set_stream_policy(fq3_engine* e, int stream_idx, const fq3_policy* policy, void* stream);
/* Serving (no counterpart in the reference, whose servers hold one lock around a bs = 1 model: examples/openai_server.py:71,181):
 * take one stream out of the lock-step frame loop — it idles (status.done = 3) in every later fq3_decode_frames until it is
 * reset and prefilled again.  A scheduler retires the slot of a finished / cancelled / length-capped request so that the
 * other streams of the group keep decoding, and parks never-used slots the same way. */
int fq3_retire_stream(fq3_engine* e, int stream_idx, void* stream);
/* TalkerGraph.set_generation_state (talker_graph.py:172-196): left pads and rope delta of one stream. */
int fq3_set_generation_state(fq3_engine* e, int stream_idx, int n_left_pad, int rope_delta, void* stream);
/* trailing_text_hiddens / tts_pad_embed of generate.py:168-171; copied into engine-owned buffers.
 * trailing: bf16 [n_trailing, H_t]; pad_embed: bf16 [H_t].  The text is closed: it ends after these rows, also on a slot
 * whose text was open (fq3_open_text). */
int fq3_set_text_conditioning(fq3_engine* e, int stream_idx, const void* trailing, int n_trailing,
                              const void* pad_embed, void* stream);
/* Incremental text input (no counterpart in the reference): the trailing text rows of a stream arrive while it decodes.
 * fq3_open_text empties the stream's trailing text and leaves it open; fq3_append_text copies rows bf16 [n, H_t] after the
 * rows given so far and, with close != 0, ends the text (later frames add pad_embed, as after the last row of a closed text).
 * A frame of an open stream that needs text row gen_step before it has arrived is not run: the stream's sampler sets
 * status.done = 4 ("waiting for text") and the stream idles, its state unchanged, through the rest of the launch and every
 * later launch until an fq3_append_text delivers that row or closes the text, which sets done back to 0.  A wait changes no
 * arithmetic and no draw: whatever the arrival schedule, the stream's codes are the codes of the same stream with the whole
 * text given up front by fq3_set_text_conditioning.  A prefill of an open stream whose text has no row yet ends waiting.
 * A launch whose streams all wait runs one idle frame: the caller skips it.  Both calls are stream-ordered (a kernel on
 * `stream` updates the state; the rows may be freed once `stream` has passed the call) and must not overlap a launch on the
 * stream.  The open state survives fq3_reset_stream and the reset inside a prefill, as the text rows do;
 * fq3_set_text_conditioning closes it.  fq3_append_text returns -FQ3_E_INVALID when the stream's text is not open and
 * -FQ3_E_TOO_LONG when the rows would exceed max_seq_len. */
int fq3_open_text(fq3_engine* e, int stream_idx, const void* pad_embed, void* stream);
int fq3_append_text(fq3_engine* e, int stream_idx, const void* rows, int n, int close, void* stream);
/* TalkerGraph.prefill_kv (talker_graph.py:153-170): import an externally computed prefix KV.
 * k, v: bf16 [n_kv_heads, T, head_dim] of one layer.  Returns -FQ3_E_TOO_LONG if T > max_seq_len
 * (the reference raises RuntimeError, talker_graph.py:163-167). */
int fq3_import_kv(fq3_engine* e, int stream_idx, int layer, const void* k, const void* v, int T, void* stream);
/* Seed the loop state the reference carries in Python locals (generate.py:120-134): first token,
 * past_hidden bf16 [H_t], prefill_len, generation step. */
int fq3_set_loop_state(fq3_engine* e, int stream_idx, int token, const void* past_hidden, int position,
                       int gen_step, void* stream);

/* ---- the hot path -------------------------------------------------------------------------- */
/* Prefill (generate.py:107-134): full-sequence talker pass over embeds bf16 [T, H_t] (n_left_pad leading
 * rows are padding), K/V written straight into the static cache, then codec_head on the last row and
 * the first-token sample (EOS suppressed iff min_new_tokens > 0).  Leaves the stream ready for
 * fq3_decode_frames.  out_logits (optional) receives the last-row logits as fp32 [V_t]. */
int fq3_prefill(fq3_engine* e, int stream_idx, const void* embeds, int T, int n_left_pad,
                const fq3_policy* policy, void* out_logits, void* stream);
/* Prefill whose first T - n_tail rows were computed elsewhere (the dense tensor-core prefill writes their K/V straight
 * into the static cache, fq3_kv_cache_ptr): only rows [T - n_tail, T) go through the decode kernel, then head + first-token
 * sample exactly as fq3_prefill.  embeds_tail: bf16 [n_tail, H_t].  No left padding on this path. */
int fq3_prefill_tail(fq3_engine* e, int stream_idx, const void* embeds_tail, int T, int n_tail, const fq3_policy* policy,
                     void* out_logits, void* stream);
/* Prefill whose T rows were ALL computed elsewhere (dense tensor-core prefill: K/V of every layer already in the static cache):
 * last_hidden = the last row's residual stream after the last layer (bf16 [H_t], before the final norm).  Runs the final
 * RMSNorm + codec_head and the first-token sample (generate.py:119-134) and leaves the stream ready for fq3_decode_frames,
 * exactly as fq3_prefill does. */
int fq3_prefill_head(fq3_engine* e, int stream_idx, const void* last_hidden, int T, const fq3_policy* policy, void* out_logits,
                     void* stream);
/* Device address of one layer's static talker cache of one stream: bf16 [n_kv_heads][max_seq_len][head_dim];
 * which = 0 keys, 1 values (the StaticCache of talker_graph.py:43). */
void* fq3_kv_cache_ptr(fq3_engine* e, int stream_idx, int layer, int which);
/* TalkerGraph.run (talker_graph.py:198-214): one decode step of the 28-layer backbone.
 * embeds bf16 [H_t]; out_hidden bf16 [H_t] (post final norm); out_logits optional fp32 [V_t]
 * (= codec_head(out_hidden), generate.py:182). */
int fq3_talker_step(fq3_engine* e, int stream_idx, const void* embeds, int position, void* out_hidden,
                    void* out_logits, void* stream);
/* PredictorGraph.run (predictor_graph.py:204-214): pred_input bf16 [2, H_t] -> int64[15] device.
 * out_logits optional fp32 [15, V_p] (per-step logits, teacher-forced only by the sampled codes). */
int fq3_predictor_run(fq3_engine* e, int stream_idx, const void* pred_input, const fq3_subpolicy* sub,
                      uint64_t seed, void* out_codes_i64, void* out_logits, void* stream);
/* sample_logits + apply_repetition_penalty (sampling.py:10-66) on one row of fp32 logits [V].
 * history: int64 [n_history] device (may be NULL); suppress_eos mirrors suppress_tokens=[eos].
 * flags bit0: the logits came from a bf16 tensor — round penalty/temperature results to bf16 exactly
 * where the reference's bf16 tensor ops would.  out_token: int64 [1] device. */
int fq3_sample(fq3_engine* e, const void* logits_f32, int V, const void* history_i64, int n_history,
               const fq3_policy* policy, int eos_id, int suppress_eos, int flags, uint64_t draw_index,
               void* out_token_i64, void* stream);
/* apply_repetition_penalty (sampling.py:10-29) alone, in place on fp32 logits [V]; same flags. */
int fq3_apply_repetition_penalty(fq3_engine* e, void* logits_f32, int V, const void* history_i64, int n_history,
                                 float penalty, int flags, void* stream);
/* The frame loop of generate.py:149-199 / streaming.py:106-154 run on the device for up to n_frames
 * frames on streams [0, n_streams): predictor -> 16-row embedding sum (+ trailing text / pad) ->
 * talker step -> codec_head -> repetition penalty -> sample -> EOS test.  Appends int32[16] rows to the
 * stream's codes buffer.  One launch, zero host synchronisations inside. */
int fq3_decode_frames(fq3_engine* e, int n_streams, int n_frames, const fq3_policy* policy,
                      const fq3_subpolicy* sub, void* stream);
/* Prompt assembly on the device (replaces the ~60 eager tensor ops of `_build_talker_inputs_local`, model.py:331-553, behind
 * the same Python method).  Every prompt row is text part + codec part, described by one int32[4] record:
 *   [0] index into tp_rows (bf16 [n, H_t] = text_projection(text_embedding(ids)) of every text token the prompt needs), -1 = none
 *   [1] codec part: 0 none | 1 talker codec embedding row [2] | 2 row [2] of spk_rows (bf16 [n_spk, H_t]) | 3 the 16-codebook
 *       embedding sum of reference frame [2] of ref_codes_i32 (int32 [n_ref, 16]; generate_icl_prompt's running bf16 sum)
 * Rows with neither part are zeros (left padding).  out: bf16 [n_rows, H_t].  All pointers are device addresses. */
int fq3_assemble_prompt(fq3_engine* e, const void* tp_rows, const void* desc_i32x4, int n_rows, const void* spk_rows,
                        const void* ref_codes_i32, void* out_bf16, void* stream);
/* Batched multi-request decode (no counterpart in the reference, which is hard-wired to bs = 1: talker_graph.py:46-47,
 * predictor_graph.py:70-71).  fq3_decode_frames with one or two streams runs the reference-shaped frame program (two predictor
 * rows per stream in pass 0; it can take four).  From three streams on it runs the "wide" frame program in lock-step groups of up to
 * fq3_lockstep_group(e) streams (16 where the model's rows fit the staging buffer), one launch per group and chunk: every
 * stream of a group rides the same weight sweep, a stream's tokens are the ones its single-stream run produces.
 * fq3_lockstep_group returns 4 when the wide program is not available for the model (1.7B dims: a row of the 6144-wide
 * down-projection input is 12 KB, three fit next to the weight ring); fq3_decode_frames then refuses more than four streams
 * with -FQ3_E_UNSUPPORTED and the host decodes in groups of four. */
int fq3_lockstep_group(const fq3_engine* e);

/* The engine's grid may be smaller than the device (128 of 148 SMs by default: every model shape partitions evenly over
 * 128 CTAs) so that other work — the codec decode of the previous streaming chunk — runs beside the frame loop on the
 * free SMs.  fq3_reduced_grid: that grid when SMs are left free, else 0.  fq3_set_decode_grid is kept for callers of ABI 1:
 * it accepts 0, the engine's grid or the device's SM count and changes nothing (the grid is fixed at fq3_create because
 * the weight images are tiled for it). */
int fq3_reduced_grid(const fq3_engine* e);
int fq3_set_decode_grid(fq3_engine* e, int n_ctas);
/* The device watchdog turns a protocol fault into FQ3_E_DEVICE_FAULT on every later call.  fq3_clear_fault drains the
 * stream, clears the flag and forgets all exchange epochs; streams must be prefilled again afterwards. */
int fq3_clear_fault(fq3_engine* e, void* stream);
/* Test hook: set the 32-bit exchange-epoch counter (the wrap-around path is otherwise hours of serving away). */
int fq3_debug_set_epoch(fq3_engine* e, uint32_t epoch);
/* Test hook: the first-codebook logits (fp32 [V_t] device, before penalty, suppression and temperature) that stream
 * `stream_idx`'s last talker sampling phase consumed.  Valid right after an fq3_decode_frames launch of the
 * reference-shaped program (not the wide one) that ran the stream; -FQ3_E_INVALID otherwise. */
int fq3_debug_read_talker_logits(fq3_engine* e, int stream_idx, void* out_f32, void* stream);
/* Copy status / codes back (synchronises `stream`). codes_out: host int32 [n, 16]. */
int fq3_get_status(fq3_engine* e, int stream_idx, fq3_status* out, void* stream);
int fq3_read_codes(fq3_engine* e, int stream_idx, int first_frame, int n, int32_t* codes_out, void* stream);
/* Post-final-norm hidden of the last talker pass (`past_hidden`, generate.py:121,198): bf16 [H_t] device.
 * row = 0 after fq3_prefill / fq3_talker_step, = stream index inside the frame loop. */
int fq3_last_hidden(fq3_engine* e, int row, void* out_bf16, void* stream);
/* Device address of the codes buffer int32 [max_frames, 16] of one stream (zero-copy consumers). */
void* fq3_codes_device_ptr(fq3_engine* e, int stream_idx);

/* Debug aid: per-phase clock64 marks of one CTA (enable with env FQ3_PROF=<cta index> at create time). */
int fq3_debug_read_prof(fq3_engine* e, long long* out, int n_words);

/* ---- building block exposed for parity tests ------------------------------------------------ */
/* y[M,N] = epilogue(W[N,K] · prologue(x[M,K])) through the same persistent streaming kernel (W row-major, any device
 * address: its tiled image is built on the fly).
 * flags: bit0 pre-RMSNorm with gamma, bit1 bias, bit2 residual add, bit3 SwiGLU pairing (N = 2*I
 * interleaved rows, output width N/2), bit4 fp32 output, bit5 SiLU after bias.  All pointers device; W inside or outside
 * the arena. */
int fq3_linear(fq3_engine* e, const void* W, const void* x, void* y, int M, int N, int K, int flags,
               const void* gamma, float eps, const void* bias, const void* residual, void* stream);

enum {
  FQ3_OK = 0,
  FQ3_E_INVALID = 1,
  FQ3_E_CUDA = 2,
  FQ3_E_TOO_LONG = 3,
  FQ3_E_DEVICE_FAULT = 4, /* device watchdog fired: see fq3_last_error() */
  FQ3_E_UNSUPPORTED = 5
};

#ifdef __cplusplus
}
#endif
#endif /* FQ3_H_ */
