/* etude_b200.h -- C ABI of libetude_b200.so: the B200-native Extract-stage hot path of Etude.
 *
 * The reference (Xiugapurin/Etude) is pure Python and has no FFI; the boundary it offers for this path is the
 * Python class API of etude/data/extractor.py and etude/models/amt_apc.py.  Each entry point below names the
 * reference interface it replaces; etude_b200/extractor.py and etude_b200/model.py are the host-side mirror of
 * those classes and call only these functions (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions
 *  - plain C types; every `*_dev` pointer is a device pointer owned by the caller and kept alive across the
 *    call; `*_host` pointers are host memory read before the call returns;
 *  - `stream` is a cudaStream_t passed as void* (e.g. torch.cuda.current_stream().cuda_stream); all launches
 *    are asynchronous on it unless stated otherwise;
 *  - return value 0 = ok, negative = error; etude_last_error() gives the message (thread-local);
 *  - shapes are specialised to the default ExtractorConfig (reference etude/config/schema.py:68-121: sr 16000,
 *    hop 256, n_fft 2048, 256 mel bins, 512-frame windows with 32-frame margins, 88 notes, 128 velocities,
 *    hid 256, pf 512, 4 heads, 3+3 layers).  Anything else is rejected with an error, never emulated;
 *  - one handle per device, one stream at a time per handle (not re-entrant);
 *  - there is no CPU fallback: on a machine without an sm_100 GPU etude_create fails.
 */
#ifndef ETUDE_B200_H
#define ETUDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct etude_handle etude_handle_t;

#define ETUDE_N_WEIGHT_FLOATS 5614878 /* parameters of the hFT-Transformer extractor, 512-frame windows (SURVEY.md A14) */
#define ETUDE_N_WEIGHT_FLOATS_HFT 5516574 /* the same architecture with HFTConfig's 128-frame windows: pos_embedding_time is [128, 256] */
#define ETUDE_N_BINS 256
#define ETUDE_N_FRAME 512
#define ETUDE_MARGIN 32
#define ETUDE_N_NOTE 88
#define ETUDE_N_VELOCITY 128
#define ETUDE_MAX_WINDOWS 64 /* 512-frame windows per etude_forward_windows call (256 with 128-frame windows: etude_max_windows) */

/* One decoded note; mirrors the dict {"pitch","onset","offset","velocity"} of _mpe2note (extractor.py:406). */
typedef struct {
    int32_t pitch;
    int32_t velocity;
    double onset;
    double offset;
} etude_note_t;

const char* etude_last_error(void);
const char* etude_version(void);

/* Replaces _load_model (etude/data/extractor.py:78-113): builds the device-resident, pre-packed model.
 * `weights_host`: the fp32 state_dict flattened in the order listed in etude_b200/weights.py::STATE_DICT_LAYOUT
 * (= the reference module's state_dict() order), exactly ETUDE_N_WEIGHT_FLOATS values.  Folds conv+embedding,
 * concatenates Q|K|V and the three cross-attention K|V projections, converts GEMM operands to bf16. */
int etude_create(int device, const float* weights_host, size_t n_floats, etude_handle_t** out);
void etude_destroy(etude_handle_t* h);

/* Frames per window of the loaded model (512 or 128, decided by the weight count given to etude_create) and the largest
 * n_windows one forward call accepts (64 x 512 frames or 256 x 128 frames: the same token budget). */
int etude_n_frame(const etude_handle_t* h);
int etude_max_windows(const etude_handle_t* h);

/* Bytes of device scratch etude_forward_windows needs for up to `max_windows` windows per call. */
size_t etude_workspace_bytes(const etude_handle_t* h, int max_windows);

/* Replaces the audio ingest of _wav2feature (extractor.py:181-184): wave_mono = torch.mean(wave, dim=0) followed by
 * torchaudio.transforms.Resample(sr_in, sr_out) with torchaudio's defaults (sinc_interp_hann, lowpass_filter_width 6,
 * rolloff 0.99).  pcm_dev is planar fp32 [channels][n_in] on the device; wave_out_dev receives
 * etude_resampled_length(n_in, sr_in, sr_out) = ceil(sr_out * n_in / sr_in) samples.  sr_in == sr_out: channel mean only. */
int64_t etude_resampled_length(int64_t n_in, int sr_in, int sr_out);
int etude_ingest(etude_handle_t* h, const float* pcm_dev, int channels, int64_t n_in, int sr_in, int sr_out, float* wave_out_dev,
                 void* stream);

/* Raw PCM sample formats of etude_ingest_pcm, converted to float32 as FFmpeg does: u8 (x - 128) / 2^7, s16 x / 2^15,
 * s24 (3 bytes, little-endian) x / 2^23, s32 (float)x / 2^31, f32 as is, f64 rounded to f32. */
#define ETUDE_PCM_U8 1
#define ETUDE_PCM_S16 2
#define ETUDE_PCM_S24 3
#define ETUDE_PCM_S32 4
#define ETUDE_PCM_F32 5
#define ETUDE_PCM_F64 6

/* One song of etude_ingest_pcm.  Sample (frame f, channel c) is at pcm_dev + byte_offset + f * frame_stride +
 * c * channel_stride: interleaved frames (a WAV data chunk) have frame_stride = channels * bytes and channel_stride = bytes,
 * planar audio has frame_stride = bytes and channel_stride = n_frames * bytes.  Offsets and strides of 2/4/8-byte samples
 * are multiples of the sample size. */
typedef struct {
    int64_t byte_offset;
    int64_t n_frames;
    int64_t frame_stride;
    int64_t channel_stride;
    int64_t dst_offset;     /* first output sample in wave_out_dev */
    int32_t channels;       /* 1..64 */
    int32_t sample_rate;
    int32_t format;         /* ETUDE_PCM_* */
    int32_t reserved;
} etude_pcm_song_t;

/* Builds the resampling tables for these input rates (a synchronous upload per new rate), so that later
 * etude_ingest_pcm / etude_ingest calls at those rates enqueue kernels only. */
int etude_ingest_reserve(etude_handle_t* h, const int* sample_rates, int n, int sr_out);

/* etude_ingest for n_songs songs of raw PCM in one device buffer, each with its own format, channel count, rate and
 * layout (songs_host is read on the host).  Song s writes etude_resampled_length(n_frames, sample_rate, sr_out) samples at
 * wave_out_dev + dst_offset, bit-identical to etude_ingest on the same samples converted to planar fp32.  Uses no device
 * buffer of the handle, so it may run on another stream beside the log-mel, model and note calls.  Every song is checked
 * before anything is launched. */
int etude_ingest_pcm(etude_handle_t* h, const void* pcm_dev, const etude_pcm_song_t* songs_host, int n_songs, int sr_out,
                     float* wave_out_dev, void* stream);

/* Rows of the padded feature block of a song with n_samples samples: 32 + T_pad + 32 where
 * T = 1 + n_samples/256 and T_pad = ceil(T/512)*512 (extractor.py:210-213). */
int64_t etude_feature_rows(int64_t n_samples);

/* Replaces _wav2feature's MelSpectrogram -> log -> .T (extractor.py:186-197) and the -18 padding of
 * _transcript (extractor.py:210-213) for n_songs mono 16 kHz waves that are already on the device.
 * Song s reads wave_dev[wave_off_host[s] .. + n_samples_host[s]) and writes rows
 * [feat_row_off_host[s], + etude_feature_rows(n_samples_host[s])) of feat_dev ([rows, 256] fp32): 32 rows of
 * -18, T log-mel rows, -18 up to T_pad, 32 rows of -18.  n_samples must exceed 1024 (reflect padding). */
int etude_logmel(etude_handle_t* h, const float* wave_dev, const int64_t* wave_off_host, const int64_t* n_samples_host,
                 int n_songs, float* feat_dev, const int64_t* feat_row_off_host, void* stream);

/* The same front-end with the block layout spelled out, for the other padding schemes on the path: song s writes
 * feat_rows_host[s] rows = front_rows rows of pad_value, its T = 1 + n_samples/256 log-mel rows, pad_value to the end.
 * pad_reflect != 0: torchaudio's default pad_mode="reflect" (the AMT-APC extractor); 0: pad_mode="constant", zeros
 * outside the wave (HFT_Transformer._wav2feature, etude/models/hft_transformer.py:121-137).
 * HFT_Transformer._transcript_stride (hft_transformer.py:288-318): front_rows = margin_b + n_offset = 64, pad_value = -80,
 * rows = 64 k with k = ceil((T + 128) / 64); ._transcript (140-168): front_rows = 32, rows = 32 + ceil(T/128)*128 + 32. */
int etude_logmel_layout(etude_handle_t* h, const float* wave_dev, const int64_t* wave_off_host, const int64_t* n_samples_host,
                        int n_songs, float* feat_dev, const int64_t* feat_row_off_host, const int64_t* feat_rows_host,
                        int front_rows, float pad_value, int pad_reflect, void* stream);

/* Replaces the body of _transcript's window loop (extractor.py:227-248) = Model_SPEC2MIDI.forward
 * (etude/models/amt_apc.py:29-49) + sigmoid heads + velocity argmax, for n_windows windows at once.
 * Window w reads padded feature rows [win_row_host[w], +576) of feat_dev (i.e. input_spec[w] = those rows
 * transposed) and writes 512 rows starting at roll row out_row_host[w] of every non-null roll
 * ([rows, 88]; fp32 onset/offset/mpe, int8 velocity = argmax over the 128 logits).
 *   rolls_B_dev[4] : onset_B, offset_B, mpe_B, velocity_B  (time-axis heads; NULL = the time-axis layers are skipped:
 *                    _transcript(mode != "combination"), extractor.py:236,250-253)
 *   rolls_A_dev[4] : onset_A, offset_A, mpe_A, velocity_A  (frequency-axis heads; may be NULL = skipped; not both)
 * Optional model-level outputs for Model_SPEC2MIDI.forward's 9-tuple (each may be NULL):
 *   vel_logits_A_dev / vel_logits_B_dev : fp32 [n_windows, 512, 88, 128]
 *   attention_dev : fp32 [n_windows*512, 4, 88, 256], last cross-attention probabilities (amt_apc.py:178-179) */
int etude_forward_windows(etude_handle_t* h, const float* feat_dev, const int64_t* win_row_host,
                          const int64_t* out_row_host, int n_windows, void* const rolls_A_dev[4],
                          void* const rolls_B_dev[4], float* vel_logits_A_dev, float* vel_logits_B_dev,
                          float* attention_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* Replaces the loop body of HFT_Transformer._transcript_stride (etude/models/hft_transformer.py:282-460): like
 * etude_forward_windows, but only window frames [keep_first, keep_first + keep_count) reach the rolls, written at rows
 * out_row_host[w] .. + keep_count (hft_transformer.py:352-441: n_offset = 32, half_frame = 64 -> the centre half of every
 * 128-frame window, windows advancing by 64 frames).  The overlapped-window stitching therefore happens in the heads
 * epilogue on the device.  rolls_A_dev or rolls_B_dev may be NULL (B NULL also skips the time-axis layers). */
int etude_forward_windows_stride(etude_handle_t* h, const float* feat_dev, const int64_t* win_row_host, const int64_t* out_row_host,
                                 int n_windows, void* const rolls_A_dev[4], void* const rolls_B_dev[4], int keep_first, int keep_count,
                                 void* workspace_dev, size_t workspace_bytes, void* stream);

/* Replace _Spec2MIDI.encode / .decode (etude/data/extractor.py:58-75; sv_dim = 0): the encoder half
 * (Encoder_SPEC2MIDI.forward, amt_apc.py:74-120) writes its output as fp32 [n_windows * n_frame * 256, 256] =
 * [B, n_frame, n_bin, hid]; the decoder half (Decoder_SPEC2MIDI.forward, amt_apc.py:159-230) reads such a tensor.
 * Activations are bf16 inside, so decode(encode(x)) is bit-identical to etude_forward_windows. */
int etude_encode_windows(etude_handle_t* h, const float* feat_dev, const int64_t* win_row_host, int n_windows, float* enc_out_dev,
                         void* workspace_dev, size_t workspace_bytes, void* stream);
int etude_decode_windows(etude_handle_t* h, const float* enc_in_dev, const int64_t* out_row_host, int n_windows,
                         void* const rolls_A_dev[4], void* const rolls_B_dev[4], float* vel_logits_A_dev, float* vel_logits_B_dev,
                         float* attention_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* Replaces _mpe2note (extractor.py:256-418) for n_songs songs whose rolls live on the device.
 * Song s owns roll rows [song_row_off_host[s], + song_rows_host[s]).  mode_velocity: 0 'ignore_zero', 1 'org';
 * mode_offset: 0 'shorter', 1 'longer', 2 'offset'.  All kernels are enqueued before the call's single host round trip
 * (the per-song counts, then exactly that many records); the call returns after the records have reached the host.
 * On return *notes_out points to LIBRARY-OWNED pinned host memory holding the songs' notes back to back, each song sorted
 * like extractor.py:416, and n_notes_host[s] their counts; the memory stays valid until the next etude_notes call on this
 * handle (copy what you keep).  Bit-exact with the reference on identical rolls.
 * etude_notes_reserve sizes the stage's device scratch once for calls of up to max_rows roll rows in max_songs songs (e.g.
 * the largest notes batch); without it the first call that needs more grows the scratch itself (a device synchronisation). */
int etude_notes_reserve(etude_handle_t* h, int64_t max_rows, int max_songs);
int etude_notes(etude_handle_t* h, const float* onset_dev, const float* offset_dev, const float* mpe_dev,
                const int8_t* velocity_dev, const int64_t* song_row_off_host, const int64_t* song_rows_host, int n_songs,
                int note_min, double hop_sec, double thred_onset, double thred_offset, double thred_mpe, int mode_velocity,
                int mode_offset, const etude_note_t** notes_out, int64_t* n_notes_host, void* stream);
/* The same call in two halves for callers that own the destination (the Python mirror does: the records land straight in
 * the pinned array it returns, no staging copy): etude_notes_begin runs every kernel and returns the per-song counts
 * (the first half of the round trip; the sorted records stay on the device), etude_notes_fetch copies exactly the first
 * n_records (<= the sum of those counts) into dst_host and returns when they are there. */
int etude_notes_begin(etude_handle_t* h, const float* onset_dev, const float* offset_dev, const float* mpe_dev,
                      const int8_t* velocity_dev, const int64_t* song_row_off_host, const int64_t* song_rows_host, int n_songs,
                      int note_min, double hop_sec, double thred_onset, double thred_offset, double thred_mpe, int mode_velocity,
                      int mode_offset, int64_t* n_notes_host, void* stream);
int etude_notes_fetch(etude_handle_t* h, etude_note_t* dst_host, int64_t n_records, void* stream);

/* Launch accounting and optional per-launch CUDA-event timing, per kernel class (logmel, embed, gemm_bias, gemm_ln,
 * gemm_heads, attention, notes): what bench.py's roofline and gpu_launches are computed from.  No reference
 * counterpart.  etude_profile_reset zeroes the counters and switches event timing on/off; etude_profile_read
 * synchronises the device and fills arrays of etude_profile_classes() entries: summed event time (ms), launch
 * count, algorithmic FLOPs and algorithmic HBM bytes of the launches since the reset. */
int etude_profile_classes(void);
const char* etude_profile_class_name(int cls);
int etude_profile_reset(etude_handle_t* h, int enable_timing);
int etude_profile_read(etude_handle_t* h, double* ms, int64_t* launches, double* flops, double* bytes);
/* Per-launch timeline of the last timed pass: start (ms after the first timed launch) and duration of launch i in
 * recording order, its class; returns the number written (<= cap) or -1. */
int etude_profile_timeline(etude_handle_t* h, double* start_ms, double* dur_ms, int32_t* cls, int cap);

#ifdef __cplusplus
}
#endif
#endif /* ETUDE_B200_H */
