/* libwisb200 -- C ABI of the B200-native Whisper hot path that replaces, inside toverainc/willow-inference-server,
 *   (1) wis.audio.log_mel_spectrogram / pad_or_trim        (/root/reference/wis/audio.py:28-51, :72-103)
 *   (2) ctranslate2.models.Whisper(...)                     (/root/reference/main.py:341-355 and the four copies :363-443)
 *   (3) ctranslate2.StorageView.from_array(features)        (/root/reference/main.py:638, :685)
 *   (4) Whisper.generate(features, prompts, beam_size=...)  (/root/reference/main.py:687-692, positional form :535-537)
 *   (5) Whisper.detect_language(features)                   (/root/reference/main.py:638-640)
 *
 * Plain C: pointers and sizes only, no C++/torch types.  Every host buffer is owned by the caller and only borrowed for
 * the duration of the call; the handle owns device weights, workspaces, KV caches, streams and CUDA graphs.
 * All functions return 0 on success, 1 for invalid arguments (-> ValueError in the Python shim), 2 for CUDA/runtime
 * failures (-> RuntimeError); wisb_last_error() returns a thread-local message.  There is NO CPU fallback: without a
 * CUDA device every entry point except wisb_last_error / wisb_abi_version fails with code 2.
 * Calls on one handle are serialised internally; different handles may be used from different threads.
 */
#ifndef WISB200_H_
#define WISB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wisb_handle wisb_handle;

#define WISB_ABI_VERSION 1
#define WISB_PCM_F32 0 /* float32 in [-1, 1]  (what librosa.load hands do_whisper, main.py:579) */
#define WISB_PCM_S16 1 /* int16 little endian (what /api/willow receives, main.py:1277-1299); scaled by 1/32768 on device */
#define WISB_N_DIMS 20

int wisb_abi_version(void);
const char* wisb_last_error(void);

/* (2) model construction.  `weights_path` is a WISB200 blob (willow_inference_server_b200/weights.py).  The *_host and
 * *_device forms take an in-memory blob; the device form borrows an already-populated device buffer (e.g. the target of
 * the load-time NCCL broadcast) which must outlive the handle. */
int wisb_create(const char* weights_path, int device, wisb_handle** out);
int wisb_create_from_host(const void* blob, size_t nbytes, int device, wisb_handle** out);
int wisb_create_from_device(const void* device_blob, size_t nbytes, int device, wisb_handle** out);
/* a handle without a model: only wisb_logmel works on it (wis.audio.log_mel_spectrogram is a free function) */
int wisb_create_frontend(int device, wisb_handle** out);
int wisb_destroy(wisb_handle* h);
/* d_model, n_heads, n_enc_layers, n_dec_layers, n_vocab, n_vocab_pad, n_text_ctx, n_mels, n_audio_ctx, sot, eot,
 * transcribe, translate, no_timestamps, sot_prev, sot_lm, no_speech, blank, lang_first, n_langs */
int wisb_get_dims(wisb_handle* h, int32_t* dims /* [WISB_N_DIMS] */);

/* (1) batched log-mel.  Utterance b is n_samples[b] samples starting at pcm + offsets[b] (in samples); padding with
 * zeros / trimming to 480000 samples is fused.  pcm_on_device != 0: `pcm` is a device pointer.
 * mel_out (host, float32 [B,80,3000]) may be NULL; keep_on_device != 0 keeps the features in HBM for the next
 * wisb_generate / wisb_detect_language call that passes mel == NULL. */
int wisb_logmel(wisb_handle* h, const void* pcm, int pcm_dtype, int pcm_on_device, const int64_t* offsets,
                const int32_t* n_samples, int B, float* mel_out, int keep_on_device);

/* (3)+(4) features [B,80,3000] float32 host (or NULL: use the features kept by wisb_logmel) -> token ids.
 * prompts: int32 [B, prompt_len] (WIS passes the same 4-token prompt for every window, main.py:689).
 * beam_size 1 = greedy.  patience / length_penalty / max_length: CTranslate2 defaults 1, 1, 448.
 * extra_suppress: ids suppressed in addition to the model's suppress_ids (CT2 `suppress_tokens=[-1, ...]`), may be NULL.
 * out_ids: int32 [B, out_stride] (out_stride >= min(max_length/2, max_length-prompt_len)); out_len: int32 [B];
 * out_score (may be NULL): float32 [B] length-normalised log-probability of the returned hypothesis. */
int wisb_generate(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                  float patience, float length_penalty, int max_length, const int32_t* extra_suppress, int n_extra,
                  int32_t* out_ids, int out_stride, int32_t* out_len, float* out_score);

/* Same call with a per-utterance `max_length` (int32 [B], may be NULL = `max_length` for all): lets a cross-request
 * batcher put requests with different length limits into ONE shared decoder pass (CTranslate2's generate takes a single
 * max_length per call, /root/reference/main.py:687-692; the per-utterance form is what its semantics become when
 * several such calls are coalesced).  out_stride >= the largest per-utterance limit of new tokens. */
int wisb_generate_ex(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                     float patience, float length_penalty, int max_length, const int32_t* max_length_per_utt,
                     const int32_t* extra_suppress, int n_extra, int32_t* out_ids, int out_stride, int32_t* out_len,
                     float* out_score);

/* Same call with Whisper's timestamp rules, what CTranslate2 applies when the prompt lacks <|notimestamps|>
 * (the reference's prompts keep that token, main.py:529, :661; removing it asks for timestamps).  Timestamp tokens are
 * [no_timestamps + 1, n_vocab); the rules are those of openai-whisper's ApplyTimestampRules: <|notimestamps|> is never
 * generated, timestamps come in pairs (except right before <|endoftext|>) and never decrease, the first generated token
 * is a timestamp no later than no_timestamps + 1 + max_initial_timestamp_index, and when the timestamps' total
 * probability beats every text token a timestamp is generated.  out_ids keep the timestamp tokens (<|endoftext|> is
 * still left out).  Returns 1 when a prompt contains <|notimestamps|> or max_initial_timestamp_index is outside
 * [0, n_vocab - no_timestamps - 2]. */
int wisb_generate_ts(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                     float patience, float length_penalty, int max_length, const int32_t* max_length_per_utt,
                     const int32_t* extra_suppress, int n_extra, int max_initial_timestamp_index, int32_t* out_ids,
                     int out_stride, int32_t* out_len, float* out_score);

/* (5) per utterance: language token ids sorted by probability (descending) and the probabilities.
 * lang_ids_out int32 [B, n_langs], probs_out float32 [B, n_langs]. */
int wisb_detect_language(wisb_handle* h, const float* mel, int B, int32_t* lang_ids_out, float* probs_out);

/* stage timings (ms, CUDA events on the launching stream) of the last wisb_logmel / wisb_generate:
 * [0 logmel, 1 h2d, 2 encoder, 3 cross_kv, 4 decode, 5 total_generate, 6 decode_steps, 7 kernel_launches,
 *  8 sum of GEMM kernels, 9 attention kernels, 10 LayerNorm kernels, 11 conv1, 12 number of GEMM launches, 13-15 0]
 * entries 8-12 are filled only with option "profile" = 1 (per-kernel event pairs; leave it off for timed runs). */
int wisb_get_timing(wisb_handle* h, float* out16);
/* options: "use_graphs" (default 1), "attn_v_mn_major" (default 1), "attn_ref" (0), "decode_poll" (1), "profile" (0),
 * "decoder_mega" (1: persistent decoder-pass kernel; 0: the per-op kernel chain kept as a cross-check),
 * "encoder_cache" (default 0; 1: consecutive wisb_detect_language / wisb_generate calls on byte-identical host features
 * of <= 2 windows reuse the encoder output and cross K/V already in HBM -- the detect -> transcribe -> translate sequence
 * of main.py:633-644, 514-547 then encodes once instead of three times) */
int wisb_set_option(wisb_handle* h, const char* key, int value);

/* ---- diagnostics used by tests/ (run the product kernels on caller data) ---- */
/* C[M,N] (float32) = A[M,K] . W[N,K]^T with fp16 inputs given as raw uint16; impl 0 = tcgen05 kernel, 1 = SIMT check */
int wisb_debug_gemm(wisb_handle* h, const uint16_t* a, const uint16_t* w, float* c, int M, int N, int K, int impl, int bn);
/* the tcgen05 skinny-GEMV building block of the decoder pass on caller data: out[R,N] (float32) = x[R,K] (float32, rounded
 * to fp16 inside) . W[N,K]^T (fp16 as raw uint16) + bias (may be NULL); R <= 8, K % 64 == 0, K <= 5120.  avg_us (may be
 * NULL) receives the average kernel time over `iters` back-to-back launches. */
int wisb_debug_gemv_tc(wisb_handle* h, const float* x, const uint16_t* w, const float* bias, float* out, int R, int N, int K,
                       int iters, float* avg_us);
/* per-phase %globaltimer stamps of the last persistent decoder pass (option "mega_trace" = 1): n <= 2048 values */
int wisb_debug_read_trace(wisb_handle* h, unsigned long long* out, int n);
/* encoder output after the final LayerNorm, float32 [B,1500,d_model]; n_layers < 0 = all */
int wisb_debug_encode(wisb_handle* h, const float* mel, int B, float* enc_out, int n_layers);
/* teacher-forced raw decoder logits (no processors) for utterance 0: float32 [n_tokens, n_vocab] */
int wisb_debug_forced_logits(wisb_handle* h, const float* mel, const int32_t* tokens, int n_tokens, float* logits_out);

/* ---- (6) FLAC ingest (host code, no handle, no GPU): replaces the decode half of `librosa.load(audio_file, sr=16000)`
 * (/root/reference/main.py:579) for the FLAC files WIS is tested with (client/{3sec,10sec,30sec}.flac).
 * wisb_flac_info: stream parameters, number of inter-channel frames and the PCM MD5 from STREAMINFO (any pointer may be NULL).
 * wisb_flac_decode: interleaved int32 samples [n_frames, channels]; every frame's CRC-8 / CRC-16 is checked.
 * Both return 0 or a non-zero code with the reason in wisb_flac_last_error() (thread-local). */
const char* wisb_flac_last_error(void);
int wisb_flac_info(const void* data, size_t nbytes, int32_t* sample_rate, int32_t* channels, int32_t* bits_per_sample,
                   int64_t* n_frames, uint8_t* md5_16);
int wisb_flac_decode(const void* data, size_t nbytes, int32_t* out_interleaved, int64_t capacity_frames, int64_t* n_frames);

#ifdef __cplusplus
}
#endif
#endif /* WISB200_H_ */
