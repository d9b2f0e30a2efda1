/* nisqa_b200.h - C ABI of the B200-native NISQA predict engine (libnisqa_b200.so).
 *
 * Drop-in boundary (SURVEY.md 8b): the reference has no FFI; its seam for this path is the
 * Python function boundary
 *     NL.predict_dim(model, ds, bs, dev, num_workers)   reference nisqa/NISQA_lib.py:1441-1467
 *     NL.predict_mos(model, ds, bs, dev, num_workers)   reference nisqa/NISQA_lib.py:1420-1439
 * called from nisqaModel.predict() (reference nisqa/NISQA_model.py:54-81).  Everything below
 * that seam - get_librosa_melspec (lib:2284-2331) minus the file decode, segment_specs
 * (lib:2239-2282), Framewise/AdaptCNN/StandardCNN (lib:428-836), SelfAttention/LSTM
 * (lib:897-1040), PoolAttFF/PoolLastStepBi (lib:1099-1183) and the NISQA / NISQA_DIM
 * containers (lib:29-268) - runs inside this library as hand-written sm_100a CUDA.
 *
 * Plain C types only: pointers and sizes, no torch types.  All functions return 0 on
 * success and a negative nisqa_status on failure; nisqa_last_error() gives the message.
 * No exceptions cross the ABI.  One engine handle per GPU / rank; a handle is not
 * thread-safe.  There is NO CPU fallback: every entry point fails loudly without a device.
 */
#ifndef NISQA_B200_H
#define NISQA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NISQA_B200_ABI_VERSION 3

#if defined(__GNUC__)
#define NISQA_API __attribute__((visibility("default")))
#else
#define NISQA_API
#endif

typedef struct nisqa_engine nisqa_engine;

/* architectures of the shipped checkpoints (SURVEY.md 0.4) */
enum nisqa_arch {
  NISQA_ARCH_ADAPT_SA_ATTFF  = 0, /* nisqa.tar, nisqa_mos_only.tar: AdaptCNN + SelfAttention + PoolAttFF */
  NISQA_ARCH_STD_LSTM_LASTBI = 1  /* nisqa_tts.tar: StandardCNN + BiLSTM + PoolLastStepBi            */
};

/* pooling over time (reference lib:1066-1225).  The shipped checkpoints use ATT_FF (nisqa*.tar) and LAST_STEP_BI
 * (nisqa_tts.tar); the others are reachable through user-trained checkpoints (SURVEY.md 8f.4). */
enum nisqa_pool {
  NISQA_POOL_ATT_FF       = 0, /* PoolAttFF, h = 128 (lib:1156-1183)                  */
  NISQA_POOL_ATT          = 1, /* PoolAtt (lib:1131-1154)                             */
  NISQA_POOL_AVG          = 2, /* PoolAvg (lib:1185-1204)                             */
  NISQA_POOL_MAX          = 3, /* PoolMax (lib:1206-1225)                             */
  NISQA_POOL_LAST_STEP    = 4, /* PoolLastStep (lib:1117-1129)                        */
  NISQA_POOL_LAST_STEP_BI = 5  /* PoolLastStepBi (lib:1099-1115), BiLSTM only         */
};

/* double-ended model NISQA_DE (reference lib:272-424; train_nisqa_double_ended.yaml): time alignment of the reference
 * clip's features to the degraded clip's (Alignment, lib:1228-1285), how the alignment is applied, and the fusion of the
 * two feature streams (Fusion, lib:1380-1417).  de_align 'none' is refused (it needs equally long signals). */
enum nisqa_de_align { NISQA_DE_ALIGN_DOT = 1, NISQA_DE_ALIGN_COSINE = 2, NISQA_DE_ALIGN_DISTANCE = 3,
                      NISQA_DE_ALIGN_LUONG = 4 /* AttLuong lib:1344-1357 */, NISQA_DE_ALIGN_BAHDANAU = 5 /* AttBahdanau lib:1325-1342 */ };
enum nisqa_de_apply { NISQA_DE_APPLY_HARD = 0, NISQA_DE_APPLY_SOFT = 1 };
enum nisqa_de_fuse  { NISQA_DE_FUSE_XY_MINUS = 0 /* 'x/y/-' */, NISQA_DE_FUSE_PLUS_MINUS = 1 /* '+/-' */, NISQA_DE_FUSE_XY = 2 /* 'x/y' */ };

enum nisqa_cnn_kind { NISQA_CNN_CONV = 0, NISQA_CNN_SKIP = 1, NISQA_CNN_DFF = 2 };

enum nisqa_sample_fmt { NISQA_FMT_S16 = 0, NISQA_FMT_F32 = 1 };

/* per-clip status written to status_out; the Python wrapper maps them onto the reference's
 * ValueError messages (lib:2259-2263 "Sample too short", lib:2276-2277 "n_wins > max_length") */
enum nisqa_clip_status { NISQA_CLIP_OK = 0, NISQA_CLIP_TOO_SHORT = 1, NISQA_CLIP_TOO_LONG = 2 };

enum nisqa_status {
  NISQA_SUCCESS = 0,
  NISQA_ERR_INVALID = -1,      /* bad argument / unsupported configuration        */
  NISQA_ERR_CUDA = -2,         /* CUDA runtime error (no device, OOM, launch)     */
  NISQA_ERR_WEIGHTS = -3,      /* missing / mis-shaped tensor in load_weights     */
  NISQA_ERR_STATE = -4,        /* call order (e.g. predict before load_weights)   */
  NISQA_ERR_NCCL = -5
};

/* stages readable through nisqa_stage_dump after a predict call (parity tests) */
enum nisqa_stage {
  NISQA_STAGE_MEL_DB   = 0, /* per clip [n_mels, n_frames] row-major, clamped (lib:2330), clips concatenated */
  NISQA_STAGE_POOL1    = 1, /* [n_seg, 16, 24, W1] NCHW like the reference tensors           */
  NISQA_STAGE_POOL2    = 2, /* [n_seg, 32, 12, W2]                                           */
  NISQA_STAGE_CONV3    = 3, /* [n_seg, 64, 12, W2]                                           */
  NISQA_STAGE_POOL3    = 4, /* [n_seg, 64, 6, W3]                                            */
  NISQA_STAGE_CONV5    = 5, /* [n_seg, 64, 6, W3]                                            */
  NISQA_STAGE_CNN_FEAT = 6, /* [n_seg, 384] (adapt, index c*6+h) or [n_seg, 20] (standard)   */
  NISQA_STAGE_TD_IN    = 7, /* adapt only: LayerNorm(Linear 384->64) [n_seg, 64]             */
  NISQA_STAGE_TD_OUT   = 8  /* [n_seg, 64] (self-attention) or [n_seg, 256] (BiLSTM fwd||bwd) */
};

/* Mirrors the checkpoint 'args' the hot path consumes (SURVEY.md Appendix A). */
typedef struct nisqa_config {
  int32_t abi_version;   /* NISQA_B200_ABI_VERSION */
  int32_t arch;          /* enum nisqa_arch */
  int32_t n_out;         /* 1 (NISQA) or 5 (NISQA_DIM: mos,noi,dis,col,loud - lib:1461-1465) */
  int32_t n_fft;         /* ms_n_fft = 4096 */
  int32_t n_mels;        /* ms_n_mels = 48  */
  int32_t seg_len;       /* ms_seg_length = 15 */
  int32_t seg_hop;       /* ms_seg_hop_length (4 | 1) */
  int32_t max_segments;  /* ms_max_segments (1300 | 6000) */
  double  hop_s;         /* ms_hop_length seconds: hop = (int)(sr*hop_s), lib:2308 */
  double  win_s;         /* ms_win_length seconds: win = (int)(sr*win_s), lib:2309 */
  double  fmax;          /* ms_fmax Hz */
  int32_t sa_layers;     /* td_sa_num_layers (adapt arch), else 0 */
  int32_t max_chunk_segments; /* 0 = default; upper bound on segments processed per internal pass */
  int32_t pool;          /* enum nisqa_pool */
  int32_t pos_enc;       /* td_sa_pos_enc: add the checkpoint's positional-encoding buffer after the input LayerNorm (lib:1042-1062) */
  /* NISQA_DE (arch NISQA_ARCH_ADAPT_SA_ATTFF, n_out 1).  A double-ended engine takes its clips in PAIRS: clip 2p is the
   * degraded signal, clip 2p + 1 its reference (csv_deg / csv_ref of one dataset row, lib:2132-2156); n_clips must be
   * even; scores_out row 2p holds the pair's score, row 2p + 1 is NaN; a pair with a skipped clip scores NaN. */
  int32_t double_ended;  /* 1: NISQA_DE */
  int32_t de_align;      /* enum nisqa_de_align */
  int32_t de_align_apply;/* enum nisqa_de_apply */
  int32_t de_fuse;       /* enum nisqa_de_fuse */
  int32_t td2_layers;    /* td_2 = 'self_att' (d_model 64, one head, h 64): number of layers; 0 = td_2 'skip'.  NISQA_DE needs >= 1;
                          * NISQA / NISQA_DIM run it as a second stack behind the first (lib:114-141, 236-268) */
  int32_t td2_pos_enc;   /* td_2_sa_pos_enc */
  /* framewise model in front of the self-attention stack (arch NISQA_ARCH_ADAPT_SA_ATTFF): */
  int32_t cnn_kind;      /* enum nisqa_cnn_kind: 0 = the convolutional networks, 1 = SkipCNN (lib:504-534), 2 = DFF (lib:536-583) */
  int32_t cnn_fc;        /* cnn_fc_out_h: Linear behind the AdaptCNN (lib:682-684, 708-709), of SkipCNN (0 = none: 720 features),
                          * hidden width of DFF; a multiple of 64 */
  int32_t de_fuse_dim;   /* NISQA_DE: Linear(fused features -> de_fuse_dim) behind the fusion (lib:1399-1401, 1414-1415); 0 = none;
                          * a multiple of 64 */
} nisqa_config;

/* One state_dict entry, passed straight through: name as in the checkpoint
 * ("cnn.model.conv1.weight", ...), fp32 host data, up to 4 dims. */
typedef struct nisqa_tensor {
  const char*  name;
  const float* data;
  int32_t      ndim;
  int64_t      dims[4];
} nisqa_tensor;

NISQA_API int  nisqa_create(nisqa_engine** out, int device, const nisqa_config* cfg);
NISQA_API void nisqa_destroy(nisqa_engine* e);
NISQA_API const char* nisqa_last_error(const nisqa_engine* e);

/* replaces model.load_state_dict(checkpoint['model_state_dict'], strict=True), model:1023:
 * folds eval-mode BatchNorm into the convolutions, repacks to the kernel layouts, uploads. */
NISQA_API int  nisqa_load_weights(nisqa_engine* e, const nisqa_tensor* tensors, int n);

/* replaces the body of predict_dim / predict_mos for n_clips clips given as mono PCM in HOST
 * memory (already channel-selected / mono-mixed by the caller, lib:2298-2304).
 *   pcm[i]         : n_samples[i] samples of sample_fmt
 *   sample_rate[i] : native rate of clip i (ms_sr=None path, lib:2304)
 *   scores_out     : [n_clips, n_out] fp32 (NaN rows for clips whose status != OK)
 *   n_segments_out : [n_clips] int32 - n_wins as returned by segment_specs (lib:2282)
 *   status_out     : [n_clips] int32 - enum nisqa_clip_status
 * Synchronous: results are valid in host memory on return. */
NISQA_API int  nisqa_predict_pcm(nisqa_engine* e, int n_clips,
                       const void* const* pcm, const int64_t* n_samples,
                       const int32_t* sample_rate, int sample_fmt,
                       float* scores_out, int32_t* n_segments_out, int32_t* status_out);

/* Asynchronous form of nisqa_predict_pcm for streams of batches (what the reference gets from
 * DataLoader prefetching, lib:1425-1430): returns as soon as the copies and kernels are enqueued;
 * up to six submissions are in flight (their uploads run ahead on the copy stream, their kernels
 * rotate over three compute lanes), so the host->device copy of batch k+1 overlaps the kernels
 * of batch k.  n_segments_out / status_out are valid on return (host arithmetic); scores_out and the
 * PCM buffers must stay alive until nisqa_wait(ticket) returns.  Submitting a seventh batch first waits for the oldest one. */
NISQA_API int  nisqa_submit_pcm(nisqa_engine* e, int n_clips,
                                const void* const* pcm, const int64_t* n_samples,
                                const int32_t* sample_rate, int sample_fmt,
                                float* scores_out, int32_t* n_segments_out, int32_t* status_out,
                                int64_t* ticket);
NISQA_API int  nisqa_wait(nisqa_engine* e, int64_t ticket);
/* Abandon every submission still in flight (error paths of the caller: a later batch failed on the host side and
 * the loop is being unwound): waits until the device is idle, then forgets the tickets WITHOUT writing their
 * scores - after it returns the scores_out / PCM buffers of those submissions may be freed. */
NISQA_API int  nisqa_drain(nisqa_engine* e);

/* Same computation with the packed PCM already resident in device memory (clips laid back
 * to back, clip i starting at element offset pcm_offsets[i]); scores stay on the device
 * (scores_dev [n_clips, n_out]).  Asynchronous on the engine stream unless sync != 0.
 * Used by bench.py for the "inputs resident in HBM" throughput figure. */
NISQA_API int  nisqa_predict_pcm_device(nisqa_engine* e, int n_clips,
                              const void* pcm_dev, const int64_t* pcm_offsets,
                              const int64_t* n_samples, const int32_t* sample_rate,
                              int sample_fmt, float* scores_dev,
                              int32_t* n_segments_out, int32_t* status_out, int sync);

/* Copy an intermediate of the LAST predict call to host memory (parity tests).  Only valid
 * when that call fitted in one internal pass.  Returns the number of floats written (>=0)
 * or a negative status; with out == NULL returns the required count. */
NISQA_API int64_t nisqa_stage_dump(nisqa_engine* e, int stage, float* out, int64_t cap);

/* Pure host arithmetic (no device work): frames / segments / status for a clip length,
 * exactly as lib:2308 + librosa's frame count + lib:2257-2277. */
NISQA_API int  nisqa_segment_counts(const nisqa_config* cfg, int64_t n_samples, int32_t sample_rate,
                          int32_t* n_frames, int32_t* n_segments, int32_t* status);

/* Host copy of the engine's mel filterbank for a sample rate: dense [n_mels, n_fft/2+1]. */
NISQA_API int  nisqa_mel_filterbank(nisqa_engine* e, int32_t sample_rate, float* out, int64_t cap);

/* Single exchange step of the multi-GPU path (SURVEY.md 8e): gather the per-rank score rows
 * onto every rank with one ncclAllGather on the engine stream.
 *   nccl_comm : ncclComm_t of the caller (one rank per GPU)
 *   local_dev : [max_rows, n_out] fp32 device rows of this rank (padded to max_rows)
 *   global_dev: [world, max_rows, n_out] fp32 device buffer */
NISQA_API int  nisqa_gather_nccl(nisqa_engine* e, void* nccl_comm /* NULL: the engine's own */,
                       const float* local_dev, int max_rows, float* global_dev);
/* Engine-owned communicator: rank 0 calls nisqa_nccl_unique_id (128 bytes), the caller ships
 * the id to every rank (torch.distributed broadcast), every rank calls nisqa_nccl_init. */
NISQA_API int  nisqa_nccl_unique_id(nisqa_engine* e, void* id128);
NISQA_API int  nisqa_nccl_init(nisqa_engine* e, int world, int rank, const void* id128);
/* Streaming form of the exchange: once a target [world, rows, n_out] device buffer is set, every
 * nisqa_submit_pcm / nisqa_predict_pcm_device call over exactly `rows` clips ends with the
 * ncclAllGather of its score rows, enqueued on the call's own compute lane (no host sync).
 * global_dev == NULL switches it off. */
NISQA_API int  nisqa_set_gather_target(nisqa_engine* e, float* global_dev, int rows);

/* ---- native WAV ingest (SURVEY.md 8f.1; replaces lb.load + channel pick, lib:2298-2306) -----------
 * Host-only, thread-safe, no engine handle: probe the header, then decode straight into caller-owned
 * (ideally pinned) memory.  kind_out / out_fmt use enum nisqa_sample_fmt: S16 when the clip can be
 * delivered as int16 without loss (PCM16, mono or channel pick), else F32 (libsndfile conversion,
 * float32 mean over channels when ms_channel < 0).  Any failure is what the reference reports as
 * "Could not load file". */
NISQA_API int     nisqa_wav_probe(const char* path, int32_t ms_channel, int32_t* sample_rate,
                                  int64_t* n_frames, int32_t* channels, int32_t* kind_out);
NISQA_API int64_t nisqa_wav_decode(const char* path, int32_t ms_channel, int32_t out_fmt, void* dst,
                                   int64_t cap_frames);
/* whole-batch forms: one call per batch, files spread over n_threads native threads; status[i] per
 * file, return value = number of files that failed (or a negative status for bad arguments) */
NISQA_API int     nisqa_wav_probe_batch(int n, const char* const* paths, int32_t ms_channel, int n_threads,
                                        int32_t* sample_rate, int64_t* n_frames, int32_t* kind,
                                        int32_t* status);
NISQA_API int     nisqa_wav_decode_batch(int n, const char* const* paths, int32_t ms_channel, int32_t out_fmt,
                                         void* base, const int64_t* elem_offsets, const int64_t* cap_frames,
                                         int n_threads, int32_t* status);

/* ---- sample-rate conversion of the ingest (reference lib:2300-2304 with ms_sr != None: librosa 0.8.1
 * resample(res_type='kaiser_best', fix=True) = resampy's band-limited sinc interpolation).  Host side, no
 * engine handle.  The interpolation table (resampy's kaiser_best half window, num_table samples per zero
 * crossing) is set once; the output has ceil(n * sr_new / sr_orig) samples. */
NISQA_API int     nisqa_resample_set_filter(const double* half_window, int64_t n, int32_t num_table);
NISQA_API int64_t nisqa_resample_out_len(int64_t n, int32_t sr_orig, int32_t sr_new);
NISQA_API int64_t nisqa_resample_f32(const float* x, int64_t n, int32_t sr_orig, int32_t sr_new, float* y,
                                     int64_t cap);

/* The same conversion ON THE DEVICE (csrc/resample_gpu.cu; bit-identical to nisqa_resample_f32: float64 weights, the
 * float32 accumulator rounded after every addition, resampy's sequential time register reproduced per clip).
 * nisqa_resample_device converts one host clip (S16 samples are scaled by 1/32768 first, like the ingest) and copies the
 * result back - the parity hook; returns the number of samples written or a negative status.
 * nisqa_predict_pcm_resampled is nisqa_predict_pcm for checkpoints with ms_sr != None: every clip is converted to
 * target_sr on the device (clips already at target_sr are only copied) and the predict path runs on the converted PCM
 * where it lies, in HBM (reference lib:2300-2304 followed by the rest of get_librosa_melspec). */
NISQA_API int     nisqa_resample_device(nisqa_engine* e, const void* x, int64_t n, int sample_fmt, int32_t sr_orig,
                                        int32_t sr_new, float* y, int64_t cap);
NISQA_API int     nisqa_predict_pcm_resampled(nisqa_engine* e, int n_clips, const void* const* pcm,
                                              const int64_t* n_samples, const int32_t* sample_rate, int sample_fmt,
                                              int32_t target_sr, float* scores_out, int32_t* n_segments_out,
                                              int32_t* status_out);

/* bookkeeping for bench.py */
NISQA_API int64_t nisqa_kernel_launches(const nisqa_engine* e);   /* total kernels launched so far      */
NISQA_API void*   nisqa_stream(const nisqa_engine* e);            /* cudaStream_t of compute lane 0 */
/* Passes rotate over several compute lanes (streams with private workspaces).  nisqa_join makes
 * lane 0's stream wait for everything enqueued so far on the other lanes, so that an event recorded
 * on nisqa_stream() afterwards covers all outstanding work. */
NISQA_API int     nisqa_join(nisqa_engine* e);
/* average device time (ms) of the named kernel group during the last predict call, measured
 * with CUDA events on the engine stream when profiling was enabled; <0 if unknown.
 * groups: "frontend", "cnn", "td", "pool" */
NISQA_API int    nisqa_set_profiling(nisqa_engine* e, int on);
/* options (any other name is rejected with NISQA_ERR_INVALID, "unknown option"):
 *   "keep_pool1"  1 = also write the pool1 activations so that NISQA_STAGE_POOL1 can be dumped (default 0: the fused
 *                 conv1 + conv2 kernel, csrc/conv12.cu, keeps them in shared memory).  Scores are unchanged.
 *   "keep_td_out" standard architecture: 1 = also store the per-step BiLSTM outputs so that
 *                 NISQA_STAGE_TD_OUT can be dumped (default 0: only the final states are needed, lib:1107-1115).
 *   "fe_ppc"      frame pairs per front-end CTA (0 = kernel default). */
NISQA_API int    nisqa_set_option(nisqa_engine* e, const char* name, int value);
NISQA_API double nisqa_group_ms(const nisqa_engine* e, const char* group);

#ifdef __cplusplus
}
#endif
#endif /* NISQA_B200_H */
