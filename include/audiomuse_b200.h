/*
 * audiomuse_b200.h -- C ABI of libaudiomuse_b200.so (sm_100a).
 *
 * The reference (NeptuneHub/AudioMuse-AI) has no FFI of its own: the hot path is Python
 * calling third-party wheels (librosa, onnxruntime, voyager, cuML).  Each entry point below
 * replaces one of those call sites; the Python-side binding a maintainer adds (ctypes) is
 * shown in INTEGRATION.md and lives in audiomuse-ai_b200/_lib.py.
 *
 * Conventions
 *   - every function returns 0 on success or a negative am_status; am_last_error() gives a
 *     thread-local message.  "out of memory" appears in the message for allocation failures
 *     so the reference's OOM-retry wrapper (tasks/memory_utils.py:327-426) keeps working.
 *   - `*_dev` variants take DEVICE pointers and a cudaStream_t (as void*), do not synchronise
 *     and never touch host memory; the plain variants take HOST pointers, stage through
 *     pinned buffers and return after the result is in the caller's buffer.
 *   - caller owns all buffers; opaque handles are freed by the matching *_free.
 *   - no CUDA work happens at library load: the context is created lazily by am_init or the
 *     first call (RQ workers fork per job, rq_worker.py:48-55).
 */
#ifndef AUDIOMUSE_B200_H
#define AUDIOMUSE_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define AM_API __attribute__((visibility("default")))
#else
#define AM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum am_status {
  AM_OK = 0,
  AM_ERR_INVALID = -1,     /* bad argument / unsupported configuration */
  AM_ERR_CUDA = -2,        /* CUDA runtime error (message has the cudaError string) */
  AM_ERR_OOM = -3,         /* allocation failed: message contains "out of memory" */
  AM_ERR_NO_DEVICE = -4,   /* no sm_100 device visible */
  AM_ERR_IO = -5,          /* weight file unreadable / malformed */
  AM_ERR_RECALL = -6       /* fewer than k neighbours exist (voyager.RecallError) */
} am_status;

/* ------------------------------------------------------------------ lifecycle */
AM_API int am_init(int device_ordinal /* -1 = current device */);
AM_API void am_shutdown(void);
AM_API const char* am_last_error(void);
AM_API int am_version(void);
/* kernels launched by this library in the calling process since load (bench.py gpu_launches) */
AM_API uint64_t am_launch_count(void);

/* Per-launch CUDA-event timing of this library's kernels (off by default).  am_profile_report
 * writes {"kernel": {"ms": device_ms, "count": n}, ...} for the launches recorded since the last
 * report and clears them; it returns the byte length needed (call with cap = 0 to size). */
AM_API void am_profile_enable(int on);
AM_API int am_profile_report(char* buf, int cap);
/* ------------------------------------------------------------------ K1: log-mel
 * Replaces librosa.feature.melspectrogram + power_to_db as called by
 * tasks/clap_analyzer.py:438-454 (compute_mel_spectrogram).  Parameters mirror
 * config.CLAP_AUDIO_* (config.py:386-392). */
typedef struct am_mel_cfg {
  int sr;         /* 48000 */
  int n_fft;      /* 2048 (student), 1024 (teacher, config.py:384) or 512; win_length == n_fft, periodic Hann,
                   * center=True, reflect pad */
  int hop;        /* 480 */
  int n_mels;     /* 128 */
  float fmin;     /* 0 */
  float fmax;     /* 14000 */
  int transpose;  /* 0: [B, n_mels, T] (student)   1: [B, T, n_mels] (teacher layout) */
} am_mel_cfg;

typedef struct am_mel_plan am_mel_plan;
AM_API int am_mel_plan_create(const am_mel_cfg* cfg, am_mel_plan** out);
AM_API void am_mel_plan_free(am_mel_plan* plan);
/* host-only (no GPU): the dense filterbank f32[n_mels, n_fft/2+1] the plan uploads
 * (librosa.filters.mel(htk=False, norm='slaney') semantics) */
AM_API int am_mel_filterbank(const am_mel_cfg* cfg, float* out);
/* frames for a segment of n_samples: 1 + n_samples / hop */
AM_API int am_mel_num_frames(const am_mel_cfg* cfg, int n_samples);

/* host: pcm f32[B, n_samples] -> out f32[B, n_mels, T] (or [B, T, n_mels]) */
AM_API int am_mel_batch(const float* pcm, int B, int n_samples, const am_mel_cfg* cfg, float* out);
/* host: PCM16 windows as produced by am_pcm_to_segments (value q means q / 32767.0f) */
AM_API int am_mel_batch_i16(const int16_t* pcm, int B, int n_samples, const am_mel_cfg* cfg, float* out);
/* device: pcm_is_i16 selects int16 (q/32767) or float32 samples */
AM_API int am_mel_batch_dev(const am_mel_plan* plan, const void* pcm_dev, int pcm_is_i16, int B,
                     int n_samples, float* out_dev, void* stream);

/* Sibling front end on the same kernel (SURVEY 8(f) row 4): tasks/analysis.py:371-375 feeds MusiCNN with
 * librosa.feature.melspectrogram(sr=16000, n_fft=512, hop_length=256, n_mels=96, center=False, norm='slaney') and
 * log10(1 + 10000 x).  center: 1 = reflect pad n_fft/2 (T = 1 + n/hop), 0 = frame t starts at t*hop
 * (T = 1 + (n - n_fft)/hop); log_mode: 0 = 10 log10(max(1e-10, x)), 1 = log10(1 + 10000 x). */
AM_API int am_mel_plan_create_ex(const am_mel_cfg* cfg, int center, int log_mode, am_mel_plan** out);
AM_API int am_mel_num_frames_ex(const am_mel_cfg* cfg, int center, int n_samples);
AM_API int am_mel_batch_ex(const float* pcm, int B, int n_samples, const am_mel_cfg* cfg, int center, int log_mode,
                           float* out);

/* tasks/clap_analyzer.py:502-523: clip to [-1,1], *32767 -> int16 (truncation), then the
 * 10 s / 5 s-hop windowing incl. the right-aligned tail window.  Host-side.
 * audio f32[L] -> seg i16[S, 480000]; returns S through *n_seg.  seg may be NULL to query S. */
AM_API int am_pcm_to_segments(const float* audio, int64_t L, int16_t* seg, int max_seg, int* n_seg);

/* ------------------------------------------------------------------ front end: decode + resample (SURVEY 8(f) row 1)
 * What tasks/analysis.py:170-250 (robust_load_audio_with_fallback -> librosa.load(path, sr=48000, mono=True,
 * duration=AUDIO_LOAD_TIMEOUT)) does before tasks/clap_analyzer.py:495 sees a waveform, for RIFF/WAVE files: PCM 8 /
 * 16 / 24 / 32 bit and IEEE float 32 / 64 (also WAVE_FORMAT_EXTENSIBLE), any channel count, any sample rate.  Other
 * containers stay with the reference's own pydub / ffmpeg loader.  Host-only (no GPU) unless noted. */
/* bits < 0: IEEE float of -bits bits */
AM_API int am_wav_info(const char* path, int* sample_rate, int* channels, int64_t* frames, int* bits);
/* mono float32 by the channel mean (librosa.to_mono), integers scaled by 1 / 2^(bits-1) (libsndfile's float read);
 * at most max_frames frames (< 0: all; librosa's `duration`).  out == NULL: only *n_frames / *sample_rate are set. */
AM_API int am_wav_decode_mono(const char* path, int64_t max_frames, float* out, int64_t cap, int64_t* n_frames,
                              int* sample_rate);
/* 48 kHz WAV file -> the reference's int16 windows in one call (decode + am_pcm_to_segments; no GPU).  seg == NULL: only
 * *n_seg / *duration_sec.  AM_ERR_INVALID ("needs resampling") for any other rate. */
AM_API int am_wav_to_segments(const char* path, double max_seconds, int16_t* seg, int max_seg, int* n_seg,
                              double* duration_sec);
/* Device polyphase resampler: the algorithm of scipy.signal.resample_poly(x, up, down) with up / down = sr_out / sr_in
 * reduced (44.1 kHz -> 48 kHz: 160 / 147), Kaiser(5.0)-windowed sinc of half length 10 max(up, down), float64
 * accumulation.  librosa resamples with soxr_hq, which cannot be installed here: parity is pinned against scipy, NOT
 * against librosa, for files that are not already at 48 kHz. */
typedef struct am_resample_plan am_resample_plan;
AM_API int am_resample_plan_create(int sr_in, int sr_out, am_resample_plan** out);
AM_API void am_resample_plan_free(am_resample_plan* plan);
AM_API int64_t am_resample_out_len(const am_resample_plan* plan, int64_t n_in); /* ceil(n_in * up / down) */
/* host-only: the plan's polyphase table poly f32[up, taps] (poly == NULL: sizes only) and its output offset; output
 * sample k is sum_i poly[t % up, i] * x[t / up - i] with t = (k + pre_remove) * down */
AM_API int am_resample_filter(int sr_in, int sr_out, float* poly, int cap, int* up, int* down, int* taps,
                              int64_t* pre_remove);
AM_API int am_resample_dev(const am_resample_plan* plan, const float* x_dev, int64_t n_in, float* y_dev, void* stream);
AM_API int am_resample(const float* x, int64_t n_in, int sr_in, int sr_out, float* y, int64_t cap, int64_t* n_out);
/* windows a waveform of L samples at 48 kHz produces (tasks/clap_analyzer.py:510-521) */
AM_API int am_num_segments(int64_t L);
/* device form of am_pcm_to_segments: audio f32[L] in HBM -> seg i16[S, 480000] in HBM (clip, * 32767, truncation,
 * 10 s windows every 5 s + the right-aligned tail window); seg_dev == NULL only reports S */
AM_API int am_audio_to_segments_dev(const float* audio_dev, int64_t L, int16_t* seg_dev, int max_seg, int* n_seg,
                                    void* stream);

/* ------------------------------------------------------------------ K2+K3: audio encoder
 * Replaces onnxruntime.InferenceSession(CLAP_AUDIO_MODEL_PATH).run(None, {'mel_spectrogram': mel})
 * (tasks/clap_analyzer.py:109-116,534) plus the numpy pooling at :552-562.
 *
 * am_clap_load takes the file the reference deploys: an ONNX ModelProto as written by
 * torch.onnx.export(opset 17, constant folding, input 'mel_spectrogram' f32[1,1,n_mels,T];
 * student_clap/models/student_onnx_model.py:611-626), with tensor data inline or in an external-data file next
 * to it (the `model.onnx.data` case of clap_analyzer.py:132-147).  The graph is read by hand (no onnx / protobuf
 * dependency) and LOWERED, node by node, to the engine's layer program (csrc/onnx_model.cu lists the supported
 * operators and patterns); a node outside that set fails the load with its name and operator in am_last_error().
 * A private "AMW1" blob (audiomuse-ai_b200/weights.py, from a StudentCLAPAudio state_dict) is accepted too. */
typedef struct am_model am_model;
AM_API int am_clap_load(const char* model_path, am_model** out);
/* same from memory (ONNX bytes without external data, or an AMW1 blob) */
AM_API int am_clap_load_mem(const void* blob, size_t nbytes, am_model** out);
/* host-only, needs no GPU: parses + lowers `model_path` and writes one text line per layer / head operation of the
 * resulting program into buf (NUL terminated, truncated to cap); returns the size needed, or a negative am_status */
AM_API int am_clap_describe_file(const char* model_path, char* buf, int cap);
/* frees the model's workspace (activations, staging buffers); weights stay.  The cleanup step of the reference's
 * OOM retry (tasks/clap_analyzer.py:536-549, memory_utils.py:327-426): clean up, then run the same call once more */
AM_API int am_clap_release_workspace(am_model* m);
AM_API void am_clap_free(am_model* m);
AM_API int am_clap_embedding_dim(const am_model* m);
AM_API int am_clap_n_mels(const am_model* m);
/* 2 * multiply-accumulates of one segment of T frames (for tensor-roofline accounting) */
AM_API double am_clap_flops_per_segment(const am_model* m, int T);

/* flops of one window executed by the standalone GEMM kernel vs inside the fused block kernel, and the
 * algorithmic HBM bytes (block input + output) of the fused blocks */
AM_API int am_clap_flops_split(const am_model* m, int T, double* gemm_flops, double* fused_flops,
                               double* fused_bytes);

/* host: mel f32[B,1,n_mels,T] -> out f32[B, dim], each row L2-normalised (student_onnx_model.py:285) */
AM_API int am_clap_embed(am_model* m, const float* mel, int B, int T, float* out);
AM_API int am_clap_embed_dev(am_model* m, const float* mel_dev, int B, int T, float* out_dev, void* stream);

/* Fused path: PCM16 windows -> mel -> encoder -> per-track mean + L2.
 * pcm i16[S_total, n_samples]; seg_offsets i32[n_tracks+1] (prefix sums of windows per track);
 * out f32[n_tracks, dim].  A track with zero windows yields a zero row (clap_analyzer.py:561-562). */
AM_API int am_clap_embed_tracks(am_model* m, const am_mel_cfg* cfg, const int16_t* pcm, int n_samples,
                         const int32_t* seg_offsets, int n_tracks, float* out);
/* Pipelined form of am_clap_embed_tracks for bulk analysis: _submit enqueues one batch (H2D, kernels, D2H into
 * pinned staging) and returns; _collect blocks until the OLDEST submitted batch is done and fills its `out`.
 * At most two batches in flight: the next batch's copies and early blocks overlap the previous one's tail.
 * `pcm` must stay valid until the batch is collected (pin it for a truly asynchronous H2D). */
AM_API int am_clap_embed_tracks_submit(am_model* m, const am_mel_cfg* cfg, const int16_t* pcm, int n_samples,
                                       const int32_t* seg_offsets, int n_tracks, float* out);
AM_API int am_clap_embed_tracks_collect(am_model* m);
AM_API int am_clap_embed_tracks_dev(am_model* m, const am_mel_plan* plan, const int16_t* pcm_dev,
                             int n_samples, const int32_t* seg_offsets_dev, int n_tracks,
                             int n_segments, float* out_dev, void* stream);

/* ------------------------------------------------------------------ MusiCNN tower
 * Replaces the two onnxruntime sessions of tasks/analysis.py:405-509 (analyze_track):
 *   EMBEDDING_MODEL_PATH  musicnn_embedding.onnx   'model/Placeholder:0' f32[n, 187, 96] -> 'model/dense/BiasAdd:0' f32[n, 200]
 *   PREDICTION_MODEL_PATH musicnn_prediction.onnx  'serving_default_model_Placeholder:0' f32[n, 200]
 *                                                  -> 'PartitionedCall:0' f32[n, 50] (raw logits)
 * am_musicnn_load reads either file and lowers it (csrc/musicnn.cu: front-end branches conv -> ReLU -> BatchNorm ->
 * frequency max, 7-tap mid-end with residuals, time max + mean pooling, BatchNorm / dense head; the prediction graph is
 * a row program).  Any other node fails the load with its name and operator in am_last_error(). */
typedef struct am_musicnn am_musicnn;
AM_API int am_musicnn_load(const char* model_path, am_musicnn** out);
AM_API int am_musicnn_load_mem(const void* blob, size_t nbytes, am_musicnn** out);
/* host-only, needs no GPU: the lowered program as text (one line per branch / layer / head op); returns the size
 * needed (NUL included) or a negative am_status */
AM_API int am_musicnn_describe_file(const char* model_path, char* buf, int cap);
AM_API void am_musicnn_free(am_musicnn* m);
/* frees activations and staging buffers (weights stay): the cleanup step before the reference retries after an OOM
 * (tasks/analysis.py:465-486) */
AM_API int am_musicnn_release_workspace(am_musicnn* m);
/* is_embedding: 1 for a patch graph, 0 for a row graph; in_dim: row width of a row graph (0 for patches) */
AM_API int am_musicnn_dims(const am_musicnn* m, int* is_embedding, int* in_dim, int* out_dim);
/* the graph's input and output tensor names (what onnxruntime's get_inputs() / get_outputs() report), NUL
 * terminated, each buffer `cap` bytes; returns the capacity needed (nothing is written when cap is smaller) */
AM_API int am_musicnn_io_names(const am_musicnn* m, char* in_name, char* out_name, int cap);
/* 2 * multiply-accumulates of one [T, F] patch (embedding) or one row (prediction); *front_flops (optional) gets the
 * front-end branches' share, counted from the graph's kernel shapes (no padding) */
AM_API double am_musicnn_flops_per_patch(const am_musicnn* m, int T, int F, double* front_flops);
/* run_inference (tasks/analysis.py:129-170) for either graph: embedding in f32[n, T, F] (T = 187, F = 96 in the
 * reference), prediction in f32[n, in_dim] (pass T = in_dim, F = 1); out f32[n, out_dim] */
AM_API int am_musicnn_run(am_musicnn* m, const float* in, int n, int T, int F, float* out);
AM_API int am_musicnn_run_dev(am_musicnn* m, const float* in_dev, int n, int T, int F, float* out_dev, void* stream);
/* Bulk analyze_track (tasks/analysis.py:368-544) for the MusiCNN outputs: 16 kHz mono PCM of n_tracks tracks,
 * track t = pcm[offsets[t], offsets[t+1]) -> mel (n_fft 512, hop 256, 96 mels, center=False, log10(1 + 10000 x)) ->
 * 187-frame patches -> embedding -> prediction; emb_out f32[n_tracks, 200] = mean of the patch embeddings (:544),
 * moods_out f32[n_tracks, 50] = sigmoid(mean(sigmoid(logits))) (:521-522), n_patches i32[n_tracks].  A track too
 * short for one patch gets n_patches 0 and zero rows (the reference returns no result for it, :378-381).
 * pred / moods_out may be NULL.  Device memory: the PCM and the patches of ALL n_tracks are staged at once (4 bytes
 * per sample + 72 KB per patch) on top of the model workspace (about 1.3 GB for the published widths: sub-batches of
 * 512 patches, the first mid-end layer's 7 x 576-channel im2col is the largest part); callers bound n_tracks
 * (musicnn.analyze_tracks sends at most 2^26 samples, about 70 minutes of audio, per call). */
AM_API int am_musicnn_analyze_tracks(am_musicnn* emb, am_musicnn* pred, const float* pcm, const int64_t* offsets,
                                     int n_tracks, float* emb_out, float* moods_out, int* n_patches);

/* ------------------------------------------------------------------ Track features
 * The librosa part of analyze_track (tasks/analysis.py:344-365) for 16 kHz mono tracks, track t =
 * pcm[offsets[t], offsets[t+1]) (csrc/track_features.cu; oracle/track_features.py restates it):
 *   tempo   beat_track's tempo: 60 * 16000 / (512 * period), 0 when the onset envelope is all zero
 *   energy  np.mean(librosa.feature.rms(y))
 *   tuning  estimate_tuning of the power spectrogram; chroma_mean = mean over frames of chroma_stft(tuning)
 *   key     index into C, C#, ..., B of the key / scale block; is_major is always 0 there (the minor profile is the
 *           major one rolled by 3, so `major_max > minor_max` never holds)
 * tuning_counts / n_pitches: the tuning histogram over linspace(-0.5, 0.5, 101) and the pitches it counts.
 * An empty track gets n_frames 0 and zeros.  Device memory: about 13 bytes per sample of the call (8 of them the
 * power spectrogram); callers bound a call's size (track_features.track_features sends at most 2^26 samples). */
typedef struct am_track_feat {
  double tempo;
  double tuning;
  float energy;
  float chroma_mean[12];
  int period;
  int key;
  int is_major;
  int n_frames;
  int n_pitches;
  int tuning_counts[100];
} am_track_feat;
typedef struct am_features am_features;
AM_API int am_features_create(am_features** out);
AM_API void am_features_free(am_features* h);
/* frees every per-call buffer (the tables stay) */
AM_API int am_features_release_workspace(am_features* h);
/* tempogram (nullable): f32[n_tracks, 250], the per-lag mean of each track's normalised tempogram */
AM_API int am_features_run(am_features* h, const float* pcm, const int64_t* offsets, int n_tracks,
                           am_track_feat* out, float* tempogram);
/* the same with device-resident PCM (offsets, out and tempogram stay on the host), ordered on `stream` */
AM_API int am_features_run_dev(am_features* h, const float* pcm_dev, const int64_t* offsets, int n_tracks,
                               am_track_feat* out, float* tempogram, void* stream);

/* ------------------------------------------------------------------ K4: exact k-NN index
 * Replaces the voyager.Index object (voyager==2.1.0) used at tasks/voyager_manager.py:183,
 * 341-346,1397,1447,1580,1681 and tasks/clap_text_search.py:173,242,263,493.
 * metric: 0 cosine (rows are stored unit-normalised; distance = 1 - cos),
 *         1 euclidean (distance = squared L2, hnswlib convention), 2 inner product (1 - dot). */
typedef struct am_index am_index;
AM_API int am_knn_build(const float* X, int64_t N, int d, int metric, am_index** out);
AM_API int am_knn_build_dev(const float* X_dev, int64_t N, int d, int metric, void* stream, am_index** out);
AM_API void am_knn_free(am_index* idx);
AM_API int64_t am_knn_size(const am_index* idx);
AM_API int am_knn_dim(const am_index* idx);
AM_API int am_knn_get_vector(const am_index* idx, int64_t id, float* out /* [d] */);
/* Q f32[nq,d] -> ids i64[nq,k], dist f32[nq,k]; ascending distance, ties by lower id.
 * Exact: candidates are re-ranked with float64 accumulation.  Re-entrant. */
AM_API int am_knn_query(const am_index* idx, const float* Q, int nq, int k, int64_t* ids, float* dist);
/* mode: 0 auto, 1 force fp32 scoring pass, 2 force bf16 tensor-core filter pass */
AM_API int am_knn_query_ex(const am_index* idx, const float* Q, int nq, int k, int mode, int64_t* ids,
                    float* dist);
/* Device version of voyager_manager.py:526-617 (_filter_by_distance, with :487-524 for lists longer than `batch`):
 * ids i64[n_lists, n] are row ids in result order (rows outside [0, N) are dropped like missing vectors);
 * keep u8[n_lists, n] receives 1 for the items the reference's greedy walk keeps.  threshold / lookback are
 * config.DUPLICATE_DISTANCE_THRESHOLD_* / DUPLICATE_DISTANCE_CHECK_LOOKBACK (config.py:550-552), batch is
 * BATCH_SIZE_VECTOR_OPS (voyager_manager.py:63).  Distances are the reference's get_direct_distance (:99-140)
 * for the index metric (cosine / inner product: 1 - cos; euclidean: ||a - b||), in float64.  n <= 4096. */
AM_API int am_knn_filter_by_distance(const am_index* idx, const int64_t* ids, int n_lists, int n, float threshold,
                                     int lookback, int batch, unsigned char* keep);
/* Direct distances (voyager_manager.py:99-140, get_direct_distance for the index metric) between all pairs of
 * the n stored rows `ids`: out f32[n, n], symmetric; +inf where a row id is outside [0, N).  Serves the radius
 * walk / path scoring (voyager_manager.py:1166-1258) without per-candidate get_vector round trips.  n <= 8192. */
AM_API int am_knn_pairwise(const am_index* idx, const int64_t* ids, int n, float* out);
/* n stored rows in one device gather + one copy: out f32[n, d] */
AM_API int am_knn_get_vectors(const am_index* idx, const int64_t* ids, int n, float* out);
AM_API int am_knn_query_dev(const am_index* idx, const float* Q_dev, int nq, int k, int mode,
                     int64_t* ids_dev, float* dist_dev, void* stream);

/* ------------------------------------------------------------------ K5: k-means
 * Replaces cuml.cluster.KMeans(...).fit_predict (tasks/clustering_gpu.py:100-123).
 * init_centers may be NULL (k-means++ seeding from `seed`) or f32[k,d]. */
AM_API int am_kmeans_fit(const float* X, int64_t N, int d, int k, int n_init, int max_iter, float tol,
                  uint64_t seed, const float* init_centers, float* centers, int32_t* labels,
                  float* inertia, int* n_iter);
/* One Lloyd assignment pass on device data (multi-GPU hosts all-reduce sums/counts between
 * passes): labels i32[N], sums f32[k,d], counts f32[k], inertia f32[1] are OVERWRITTEN. */
AM_API int am_kmeans_assign_dev(const float* X_dev, int64_t N, int d, const float* centers_dev, int k,
                         int32_t* labels_dev, float* sums_dev, float* counts_dev,
                         float* inertia_dev, void* stream);

/* ------------------------------------------------------------------ PCA / DBSCAN (SURVEY 8(f4))
 * Replace cuml.decomposition.PCA / cuml.cluster.DBSCAN behind GPUPCA / GPUDBSCAN (tasks/clustering_gpu.py:151-278);
 * scikit-learn's results are the bar (its CPU classes are the reference's own fallback).
 * am_pca_moments: column means f64[d] and the covariance f64[d, d] (n - 1 normalisation), float64 accumulation on the
 * device; the d x d eigenproblem is the host's (LAPACK).  am_pca_project: Y f32[N, k] = (X - mean) components^T. */
AM_API int am_pca_moments(const float* X, int64_t N, int d, double* mean, double* cov);
AM_API int am_pca_project(const float* X, int64_t N, int d, const float* mean, const float* components, int k, float* Y);
/* Exact brute-force DBSCAN (euclidean, eps-neighbourhood includes the point itself): labels i32[N] numbered like
 * sklearn.cluster.DBSCAN (clusters in order of their lowest core index, border points take the smallest label among
 * their core neighbours, noise -1).  N <= 2^20 (the neighbourhood bit matrix is N^2 / 8 bytes). */
AM_API int am_dbscan(const float* X, int64_t N, int d, float eps, int min_samples, int32_t* labels, int* n_clusters);

/* Iterative form for Lloyd loops on device data (multi-GPU: one plan per rank over its row shard, the host all-reduces
 * sums / counts between steps; tasks/clustering_gpu.py:108-124 is the call this serves).  The plan keeps a split-bf16
 * copy of the rows so each step is one tensor-core assignment pass + one partial-sum pass (k <= 128; larger k runs on
 * CUDA cores).  X_dev must stay valid while the plan lives.  am_kmeans_plan_step is stream-ordered (no sync):
 * labels i32[N]; sums f32[k,d], counts f32[k], inertia f32[1] (each optional) are OVERWRITTEN; dist f32[N] (optional)
 * receives the squared distance of every row to its centre. */
typedef struct am_kmeans_plan am_kmeans_plan;
AM_API int am_kmeans_plan_create(const float* X_dev, int64_t N, int d, int k, void* stream, am_kmeans_plan** out);
AM_API int am_kmeans_plan_step(am_kmeans_plan* plan, const float* centers_dev, int32_t* labels_dev, float* sums_dev,
                               float* counts_dev, float* inertia_dev, float* dist_dev, void* stream);
AM_API int am_kmeans_plan_uses_tensor_cores(const am_kmeans_plan* plan);
/* diagnostic: rows the last step re-checked in exact fp32 (near-ties within the tensor-core error band); synchronises */
AM_API int am_kmeans_plan_last_recheck(am_kmeans_plan* plan, void* stream, int* n_rows);
AM_API void am_kmeans_plan_free(am_kmeans_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* AUDIOMUSE_B200_H */
