// engine.cu - C-ABI of libnisqa_b200.so (include/nisqa_b200.h) and the host runtime around the
// kernels: checkpoint tensor repacking (BatchNorm folding, k-major linears), per-sample-rate
// front-end tables (periodic Hann, Slaney mel filterbank as band-major CSR - restating
// librosa.filters.mel in double precision), pass planning (exact frame / segment counts,
// reference nisqa/NISQA_lib.py:2308-2309, 2257-2277), device workspaces and launches.
//
// There is no CPU fallback: without a usable CUDA device nisqa_create fails.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/nisqa_b200.h"
#include "common.cuh"

namespace nisqa {
// frontend.cu
void launch_frontend(cudaStream_t, const void*, int, const ClipDesc*, int, int,
                     const FbTables*, const float2*, float*, unsigned*, int, int, int);
void launch_seg_table(cudaStream_t, const ClipDesc*, int, const int*, const unsigned*, int, int,
                      int*, float*, int*);
void launch_mel_dump(cudaStream_t, const float*, const ClipDesc*, int, const unsigned*, float*);
// conv1.cu
void launch_conv1(cudaStream_t, int, const float*, const int*, const float*, const float*,
                  const float*, void*, void*, int);
void launch_nhwc_to_nchw(cudaStream_t, const float*, float*, long long, int, int);
// conv_split.cu
size_t split_plane_bytes(int std_mode, int layer, int n_seg);
void launch_conv_split(cudaStream_t, int, int, const void*, const void*, const void*, const float*, float,
                       void*, void*, float*, int);
void launch_unsplit(cudaStream_t, int, int, const void*, const void*, float*, int);
// conv12.cu
void launch_conv12(cudaStream_t, int, const float*, const int*, const float*, const float*, const float*, const void*,
                   const float*, float, void*, void*, int);
#ifdef NISQA_TC_TIMING
int pipe_timing_read(long long*, int, int);
int c12_timing_read(long long*, int, int);
#endif
// td.cu
struct SaLayerParams {
  const float* WoT; const float* bo; const float* W1T; const float* b1; const float* W2T;
  const float* b2; const float* ln1_g; const float* ln1_b; const float* ln2_g; const float* ln2_b;
};
struct PoolHeadParams { const float* W1T; const float* b1; const float* w2; const float* b2; const float* w3; const float* b3; };
struct LstmParams { const float* w_ih; const float* w_hh; const float* b; const float* w_pool; };
void launch_fc20(cudaStream_t, const float*, const float*, const float*, float*, int);
void launch_lstm_batched(cudaStream_t, const float*, const ClipDesc*, const int*, int, const LstmParams&, float*, float*, float, float*);
void launch_pool_final(cudaStream_t, const float*, const float*, const ClipDesc*, int, const PoolHeadParams&, int, int, float*);
// td_tiled.cu
struct ResampleClip { long long in_off, out_off, time_off; int n_in, n_out, n_fix, copy; double ratio; };
void launch_resample(cudaStream_t, const void*, int, const ResampleClip*, int, int, double*, const double*, int, int, float*);
bool resample_table(std::vector<double>*, int*);
struct DeAlignParams { const float* wT; const float* b; const float* wqT; const float* bq; const float* wyT; const float* by; const float* v; };
void launch_de_align(cudaStream_t, const float*, const ClipDesc*, int, const int*, int, int, int, int, const DeAlignParams&, float*);
void launch_de_finalize(cudaStream_t, const ClipDesc*, int, int, float*);
void launch_seg_feats(cudaStream_t, const float*, const int*, const float*, const float*, int, float*);
void launch_linear_tile(cudaStream_t, const float*, int, const float*, const float*, int, float*, int, int, int, int);
void launch_td_in(cudaStream_t, const float*, const float*, int, const float*, const float*, const float*,
                  const float*, const float*, const float*, const int*, const ClipDesc*, float*, float*, int);
struct PoolSimpleParams { const float* a1; const float* a1b; const float* w3; const float* b3; };
void launch_pool_simple(cudaStream_t, const float*, int, const ClipDesc*, int, int, const PoolSimpleParams&, int, int, float*);
void launch_td_sa(cudaStream_t, const float*, const float*, const ClipDesc*, int, const int*, int, const SaLayerParams&,
                  float*, const float*, const float*, float*, const PoolHeadParams&, int, float*);
}  // namespace nisqa

using namespace nisqa;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // reserve; a (re)allocated buffer is zero-filled on `st` (fp16 plane pairs rely on never-written
  // padding rows / columns being zero)
  cudaError_t reserve_zeroed(size_t bytes, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    cudaError_t e = reserve(bytes);
    if (e != cudaSuccess) return e;
    return cudaMemsetAsync(p, 0, cap, st);
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostBuf {  // pinned
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct FbEntry {
  int sr = 0, hop = 0, win = 0;
  std::vector<float> dense;      // [n_mels][n_bins] host copy (nisqa_mel_filterbank)
  DevBuf window, band_start, band_k0, weights, wtab;
  int n_mag = 0;
};

struct ClipPlan {
  int hop, win, n_frames, n_seg, status, fb_id;
  int run;     // processed by the pass: status OK and, in a double-ended engine, its partner's status OK too
};

struct Ticket {          // one asynchronous nisqa_submit_pcm call
  bool active = false;
  int64_t id = 0;
  size_t bytes = 0;
  float* user_scores = nullptr;
  HostBuf pinned;
  DevBuf scores;         // device scores of this submission (calls in flight do not share one)
  cudaEvent_t done = nullptr;
};

// A compute lane: everything one in-flight pass needs - its own stream, host->device staging and
// activation workspaces.  Passes rotate over the lanes, so the kernels of consecutive passes /
// submissions run on different streams: wave tails and the small low-occupancy kernels of one
// pass are filled with CTAs of another (+8..12 % throughput measured, tools/two_engines.py), and
// the upload of the next pass (copy stream) overlaps compute.
#ifndef NISQA_LANES
#define NISQA_LANES 3
#endif
constexpr int kLanes = NISQA_LANES;
constexpr int kStages = 6;     // staging slots / submissions in flight (uploads run ahead of the lanes)
struct Lane {
  cudaStream_t stream = nullptr;
  DevBuf mel, segtab, feats, xa, xb, qkv, qkv2, logits, feats20, tdout, partial, fused, td2in, ffa, ffb;
  DevBuf planes[7];        // planes[l]: fp16 hi | lo plane pair feeding conv layer l (3..6; 2: pool1, keep_pool1 only), conv_split.cu
  size_t plane_bytes[7] = {0, 0, 0, 0, 0, 0, 0};   // offset of the lo plane inside planes[l] (half of the allocation)
  void release() {
    for (auto& b : planes) b.release();
    DevBuf* all[] = {&mel, &segtab, &feats, &xa, &xb, &qkv, &qkv2, &logits, &feats20, &tdout, &partial, &fused, &td2in, &ffa, &ffb};
    for (auto* b : all) b->release();
    if (stream) cudaStreamDestroy(stream);
  }
};
// Host->device staging of one pass: pinned tables, device tables, packed PCM, and the two events that
// order it (copied: upload finished on the copy stream; done: the pass's kernels finished on its lane).
struct Stage {
  cudaEvent_t ev_copied = nullptr, ev_done = nullptr;
  bool busy = false;
  int lane = 0;
  HostBuf h_tables;
  DevBuf pcm, clips, prefixes, clipmax;
  void release() {
    DevBuf* all[] = {&pcm, &clips, &prefixes, &clipmax};
    for (auto* b : all) b->release();
    h_tables.release();
    if (ev_copied) cudaEventDestroy(ev_copied);
    if (ev_done) cudaEventDestroy(ev_done);
  }
};

struct TimerSlot {
  std::string name;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
  double ms = 0.0;
  int launches = 0;
};

}  // namespace

struct nisqa_engine {
  nisqa_config cfg;
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  bool weights_loaded = false;
  bool profiling = false;
  int fe_ppc = 0;          // frame pairs per front-end CTA (0: kernel default)
  int keep_pool1 = 0;      // also write pool1 to the plane pair planes[2] (conv12_kernel keeps it on chip; only the stage dump reads it)
  bool last_pool1 = false; // the last pass wrote pool1
  int keep_td_out = 0;     // standard arch: also write the per-step LSTM outputs [n_seg][256] (only the stage dump reads them)
  std::vector<TimerSlot> timers;

  // weights arena (device) + offsets
  DevBuf warena;
  DevBuf rs_raw, rs_out, rs_clips, rs_times, rs_win;   // device resampler of the ingest (resample_gpu.cu)
  HostBuf rs_host;
  int rs_nwin = 0, rs_num_table = 0;
  std::map<std::string, size_t> woff;   // float offsets into warena
  float pool_bias_std = 0.f;
  float tc_scale[8] = {1, 1, 1, 1, 1, 1, 1, 1};   // 2^-S of the fp16 weight pre-scale, per conv layer

  // front-end tables
  std::vector<FbEntry*> fbs;
  DevBuf fb_table;       // FbTables[]
  DevBuf tw4096;         // float2[6144] (twiddle tables of the front-end)

  // per-pass state lives in the lanes; `stream` aliases lane 0's stream (nisqa_stream)
  Lane lanes[kLanes];
  Stage stages[kStages];
  int last_stage = 0;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t cur_stream = nullptr;     // stream of the pass being enqueued (kernel timers)
  HostBuf h_scores;
  int last_lane = 0;
  int64_t pass_counter = 0;
  Ticket tickets[kStages];
  int64_t next_ticket = 1;
  DevBuf scores, dump, dump_nhwc;     // stage dumps: the NCHW result, and the channels-last activations it is converted from

  // description of the last pass (stage dumps)
  std::vector<ClipDesc> last_clips;
  int last_n_seg = 0, last_n_frames = 0, last_passes = 0;
  const float* last_td_in = nullptr;
  const float* last_td_out = nullptr;

  // engine-owned NCCL communicator (multi-GPU gather, SURVEY.md 8e)
  void* nccl_comm = nullptr;
  int nccl_world = 1, nccl_rank = 0;
  float* gather_dst = nullptr;      // when set: every asynchronous / device-path call ends with an
  int gather_rows = 0;              // ncclAllGather of its [gather_rows, n_out] scores on its own lane

  ~nisqa_engine() {
    for (auto* f : fbs) { f->window.release(); f->band_start.release(); f->band_k0.release(); f->weights.release(); f->wtab.release(); delete f; }
    DevBuf* all[] = {&warena, &fb_table, &tw4096, &scores, &dump, &dump_nhwc, &rs_raw, &rs_out, &rs_clips, &rs_times, &rs_win};
    rs_host.release();
    for (auto* b : all) b->release();
    h_scores.release();
    for (auto& tk : tickets) { tk.pinned.release(); tk.scores.release(); if (tk.done) cudaEventDestroy(tk.done); }
    if (copy_stream) cudaStreamDestroy(copy_stream);
    for (auto& l : lanes) l.release();
    for (auto& g : stages) g.release();
    stream = nullptr;
    for (auto& t : timers) for (auto& e : t.ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  }
};

namespace {

int fail(nisqa_engine* e, int code, const std::string& msg) {
  if (e) e->err = msg;
  return code;
}
#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess)                                                                \
      return fail(e, NISQA_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
  } while (0)

// ---------------------------------------------------------------- timing of kernel groups
struct Scope {
  nisqa_engine* e; TimerSlot* slot = nullptr; cudaEvent_t stop = nullptr;
  Scope(nisqa_engine* e_, const char* name, int n_launch = 1) : e(e_) {
    e->launches += n_launch;
    if (!e->profiling) return;
    for (auto& t : e->timers) if (t.name == name) slot = &t;
    if (!slot) { e->timers.push_back(TimerSlot()); slot = &e->timers.back(); slot->name = name; }
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    cudaEventRecord(a, e->cur_stream);
    slot->ev.push_back({a, b});
    slot->launches += n_launch;
    stop = b;
  }
  ~Scope() { if (stop) cudaEventRecord(stop, e->cur_stream); }
};

void collect_timers(nisqa_engine* e) {
  for (auto& t : e->timers) {
    for (auto& ev : t.ev) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) t.ms += ms;
      cudaEventDestroy(ev.first); cudaEventDestroy(ev.second);
    }
    t.ev.clear();
  }
}

// ---------------------------------------------------------------- host arithmetic (a2, a6)
void plan_clip(const nisqa_config& c, int64_t n_samples, int sr, ClipPlan* p) {
  // reference lib:2308-2309: int(sr * seconds) in double precision, truncation
  p->hop = (int)((double)sr * c.hop_s);
  p->win = (int)((double)sr * c.win_s);
  p->n_frames = 0; p->n_seg = 0; p->status = NISQA_CLIP_TOO_SHORT; p->fb_id = -1;
  if (p->hop < 1 || p->win < 1 || p->win > c.n_fft || n_samples < 1) return;
  // librosa.stft(center=True): frames = 1 + (n + 2*(n_fft/2) - n_fft) / hop = 1 + n / hop
  const int64_t frames = 1 + n_samples / p->hop;
  const int64_t n_wins = frames - (c.seg_len - 1);          // lib:2257
  p->n_frames = (int)std::min<int64_t>(frames, INT32_MAX);
  if (n_wins < 1) return;                                    // lib:2258-2263
  const int64_t n_seg = (c.seg_hop > 1) ? (n_wins + c.seg_hop - 1) / c.seg_hop : n_wins;  // lib:2271-2273
  p->n_seg = (int)std::min<int64_t>(n_seg, INT32_MAX);
  if (c.max_segments > 0 && n_seg > c.max_segments) { p->status = NISQA_CLIP_TOO_LONG; return; }  // lib:2276-2277
  p->status = NISQA_CLIP_OK;
}

// ---------------------------------------------------------------- librosa.filters.mel in double
double hz_to_mel(double f) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = (min_log_hz - 0.0) / f_sp;
  const double logstep = log(6.4) / 27.0;
  if (f >= min_log_hz) return min_log_mel + log(f / min_log_hz) / logstep;
  return (f - 0.0) / f_sp;
}
double mel_to_hz(double m) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = (min_log_hz - 0.0) / f_sp;
  const double logstep = log(6.4) / 27.0;
  if (m >= min_log_mel) return min_log_hz * exp(logstep * (m - min_log_mel));
  return 0.0 + f_sp * m;
}
void np_linspace(double start, double stop, int num, std::vector<double>& y) {
  y.resize(num);
  const double step = (stop - start) / (double)(num - 1);
  for (int i = 0; i < num; ++i) { volatile double t = (double)i * step; y[i] = t + start; }
  y[num - 1] = stop;
}

int build_fb(nisqa_engine* e, int sr, int hop, int win, int* id_out) {
  for (size_t i = 0; i < e->fbs.size(); ++i)
    if (e->fbs[i]->sr == sr) { *id_out = (int)i; return 0; }
  const nisqa_config& c = e->cfg;
  const int n_bins = c.n_fft / 2 + 1, n_mels = c.n_mels;
  FbEntry* fb = new FbEntry();
  fb->sr = sr; fb->hop = hop; fb->win = win;
  std::vector<double> fftfreqs, mels, mel_f(n_mels + 2);
  np_linspace(0.0, (double)sr / 2, n_bins, fftfreqs);
  np_linspace(hz_to_mel(0.0), hz_to_mel(c.fmax), n_mels + 2, mels);
  for (int i = 0; i < n_mels + 2; ++i) mel_f[i] = mel_to_hz(mels[i]);
  fb->dense.assign((size_t)n_mels * n_bins, 0.f);
  std::vector<int> band_start(n_mels + 1, 0), band_k0(n_mels, 0);
  std::vector<float> wts;
  for (int i = 0; i < n_mels; ++i) {
    const double fd0 = mel_f[i + 1] - mel_f[i], fd1 = mel_f[i + 2] - mel_f[i + 1];
    const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
    int k0 = -1, k1 = -1;
    for (int k = 0; k < n_bins; ++k) {
      const double lower = -(mel_f[i] - fftfreqs[k]) / fd0;
      const double upper = (mel_f[i + 2] - fftfreqs[k]) / fd1;
      const float tri = (float)std::max(0.0, std::min(lower, upper));   // float32 triangle ...
      const float w = (float)((double)tri * enorm);                      // ... then `weights *= enorm`
      fb->dense[(size_t)i * n_bins + k] = w;
      if (w != 0.f) { if (k0 < 0) k0 = k; k1 = k; }
    }
    band_start[i] = (int)wts.size();
    band_k0[i] = k0 < 0 ? 0 : k0;
    if (k0 >= 0) for (int k = k0; k <= k1; ++k) wts.push_back(fb->dense[(size_t)i * n_bins + k]);
    while (wts.size() % 32) wts.push_back(0.f);     // rows padded to the warp width (frontend mel_bands)
  }
  band_start[n_mels] = (int)wts.size();
  if (wts.empty()) wts.push_back(0.f);
  // scipy.signal.get_window('hann', win, fftbins=True): periodic Hann in float64 -> float32
  std::vector<float> window((size_t)(win + 1023) / 1024 * 1024, 0.f);   // zero-padded to the FFT sub-length
  for (int n = 0; n < win; ++n) window[n] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * (double)n / (double)win));
  if (win == 1) window[0] = 1.f;
  // fused window x residue twiddle table of the pipelined front-end: wt[r][n] = hann[n] * e^{-2 pi i r n / 4096}
  std::vector<float2> wtab(4 * 1024, make_float2(0.f, 0.f));
  for (int r = 0; r < 4; ++r)
    for (int nn = 0; nn < win && nn < 1024; ++nn) {
      const double wv = (win == 1) ? 1.0 : 0.5 - 0.5 * cos(2.0 * M_PI * (double)nn / (double)win);
      const float wf = (float)wv;                                   // the float32 window the reference multiplies with
      const double a = -2.0 * M_PI * (double)(((long)r * nn) & 4095) / 4096.0;
      wtab[r * 1024 + nn] = make_float2((float)((double)wf * cos(a)), (float)((double)wf * sin(a)));
    }
  int n_mag = 0;
  for (int i = 0; i < n_mels; ++i)
    for (int k = 0; k < n_bins; ++k)
      if (fb->dense[(size_t)i * n_bins + k] != 0.f) n_mag = std::max(n_mag, k + 1);
  fb->n_mag = n_mag;
  CK(fb->wtab.reserve(wtab.size() * sizeof(float2)));
  CK(cudaMemcpy(fb->wtab.p, wtab.data(), wtab.size() * sizeof(float2), cudaMemcpyHostToDevice));
  CK(fb->window.reserve(window.size() * 4));
  CK(fb->band_start.reserve(band_start.size() * 4));
  CK(fb->band_k0.reserve(band_k0.size() * 4));
  CK(fb->weights.reserve(wts.size() * 4));
  CK(cudaMemcpy(fb->window.p, window.data(), window.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(fb->band_start.p, band_start.data(), band_start.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(fb->band_k0.p, band_k0.data(), band_k0.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(fb->weights.p, wts.data(), wts.size() * 4, cudaMemcpyHostToDevice));
  e->fbs.push_back(fb);
  // refresh the device table of FbTables
  std::vector<FbTables> tab(e->fbs.size());
  for (size_t i = 0; i < e->fbs.size(); ++i) {
    tab[i].window = e->fbs[i]->window.as<float>();
    tab[i].band_start = e->fbs[i]->band_start.as<int>();
    tab[i].band_k0 = e->fbs[i]->band_k0.as<int>();
    tab[i].weights = e->fbs[i]->weights.as<float>();
    tab[i].wtab = e->fbs[i]->wtab.as<float2>();
    tab[i].n_mag = e->fbs[i]->n_mag;
    tab[i].pad_ = 0;
  }
  CK(cudaDeviceSynchronize());      // the table may be in use by passes in flight on any lane
  CK(e->fb_table.reserve(tab.size() * sizeof(FbTables) + 64 * sizeof(FbTables)));
  CK(cudaMemcpy(e->fb_table.p, tab.data(), tab.size() * sizeof(FbTables), cudaMemcpyHostToDevice));
  *id_out = (int)e->fbs.size() - 1;
  return 0;
}

// ---------------------------------------------------------------- weight repacking
struct TensorView { const float* d; int nd; int64_t dims[4]; int64_t numel; };

struct Packer {
  nisqa_engine* e;
  std::map<std::string, TensorView> t;
  std::vector<float> arena;
  std::string missing;
  const TensorView* get(const std::string& name, std::initializer_list<int64_t> shape) {
    auto it = t.find(name);
    if (it == t.end()) { if (missing.empty()) missing = "missing tensor " + name; return nullptr; }
    const TensorView& v = it->second;
    bool ok = v.nd == (int)shape.size();
    int i = 0;
    for (int64_t s : shape) { if (ok && v.dims[i] != s) ok = false; ++i; }
    if (!ok) { if (missing.empty()) missing = "bad shape for tensor " + name; return nullptr; }
    return &v;
  }
  size_t alloc(const std::string& key, size_t n) {
    size_t off = (arena.size() + 63) / 64 * 64;     // 256-byte aligned blocks
    arena.resize(off + n, 0.f);
    e->woff[key] = off;
    return off;
  }
};

// BatchNorm-folded conv weights go to `wf` as [cin][9][cout]; the folded bias goes to the arena as conv<idx>.b
bool pack_conv(Packer& P, int idx, int cin, int cout, std::vector<float>& wf) {
  char nm[96];
  auto name = [&](const char* fmt) { snprintf(nm, sizeof nm, fmt, idx); return std::string(nm); };
  const TensorView* w = P.get(name("cnn.model.conv%d.weight"), {cout, cin, 3, 3});
  const TensorView* b = P.get(name("cnn.model.conv%d.bias"), {cout});
  const TensorView* g = P.get(name("cnn.model.bn%d.weight"), {cout});
  const TensorView* be = P.get(name("cnn.model.bn%d.bias"), {cout});
  const TensorView* mu = P.get(name("cnn.model.bn%d.running_mean"), {cout});
  const TensorView* var = P.get(name("cnn.model.bn%d.running_var"), {cout});
  if (!w || !b || !g || !be || !mu || !var) return false;
  wf.assign((size_t)cin * 9 * cout, 0.f);
  const size_t bo = P.alloc(name("conv%d.b"), cout);
  for (int co = 0; co < cout; ++co) {
    // eval-mode BatchNorm2d (eps 1e-5) folded into the convolution (SURVEY.md Appendix A)
    const double s = (double)g->d[co] / sqrt((double)var->d[co] + 1e-5);
    P.arena[bo + co] = (float)(((double)b->d[co] - (double)mu->d[co]) * s + (double)be->d[co]);
    for (int ci = 0; ci < cin; ++ci)
      for (int tap = 0; tap < 9; ++tap)
        wf[((size_t)ci * 9 + tap) * cout + co] = (float)((double)w->d[((size_t)co * cin + ci) * 9 + tap] * s);
  }
  return true;
}

// dst[k][j] = src[j][perm(k)] for a [n_out][n_in] PyTorch Linear weight
void pack_linear_T(Packer& P, size_t off, const TensorView* w, int n_out, int n_in, float scale = 1.f) {
  for (int k = 0; k < n_in; ++k)
    for (int j = 0; j < n_out; ++j) P.arena[off + (size_t)k * n_out + j] = w->d[(size_t)j * n_in + k] * scale;
}

int pack_weights(nisqa_engine* e, const nisqa_tensor* tensors, int n) {
  Packer P; P.e = e;
  for (int i = 0; i < n; ++i) {
    if (!tensors[i].name || !tensors[i].data) continue;
    TensorView v; v.d = tensors[i].data; v.nd = tensors[i].ndim; v.numel = 1;
    for (int d = 0; d < 4; ++d) { v.dims[d] = d < v.nd ? tensors[i].dims[d] : 1; v.numel *= v.dims[d]; }
    P.t[tensors[i].name] = v;
  }
  e->woff.clear();
  const int cin[7] = {0, 1, 16, 32, 64, 64, 64}, cout[7] = {0, 16, 32, 64, 64, 64, 64};
  const bool conv_net = e->cfg.cnn_kind == NISQA_CNN_CONV;
  if (!conv_net) {
    // SkipCNN / DFF (lib:504-583): the BatchNorm2d(1) in front as a scalar affine map (applied by seg_feats_kernel, so
    // that the Linear layers see what the reference's see), Linear layers k-major, DFF's BatchNorm1d folded into them
    const bool dff = e->cfg.cnn_kind == NISQA_CNN_DFF;
    const std::string p = "cnn.model.";
    const std::string bn = dff ? "bn1." : "bn.";
    const TensorView* g = P.get(p + bn + "weight", {1});
    const TensorView* be = P.get(p + bn + "bias", {1});
    const TensorView* mu = P.get(p + bn + "running_mean", {1});
    const TensorView* var = P.get(p + bn + "running_var", {1});
    if (!g || !be || !mu || !var) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
    const double a = (double)g->d[0] / sqrt((double)var->d[0] + 1e-5);
    size_t o = P.alloc("ff.bn", 2);
    P.arena[o] = (float)a; P.arena[o + 1] = (float)((double)be->d[0] - (double)mu->d[0] * a);
    const int H = e->cfg.cnn_fc;
    auto pack_lin = [&](const std::string& wname, const std::string& bnname, int n_in, int n_in_pad, int n_out, const std::string& key) -> bool {
      const TensorView* w = P.get(p + wname + ".weight", {n_out, n_in});
      const TensorView* b = P.get(p + wname + ".bias", {n_out});
      if (!w || !b) return false;
      std::vector<double> sc(n_out, 1.0), sh(n_out, 0.0);
      if (!bnname.empty()) {            // eval-mode BatchNorm1d (eps 1e-5) folded into the Linear in front of it
        const TensorView* g2 = P.get(p + bnname + ".weight", {n_out});
        const TensorView* b2 = P.get(p + bnname + ".bias", {n_out});
        const TensorView* m2 = P.get(p + bnname + ".running_mean", {n_out});
        const TensorView* v2 = P.get(p + bnname + ".running_var", {n_out});
        if (!g2 || !b2 || !m2 || !v2) return false;
        for (int j = 0; j < n_out; ++j) {
          sc[j] = (double)g2->d[j] / sqrt((double)v2->d[j] + 1e-5);
          sh[j] = (double)b2->d[j] - (double)m2->d[j] * sc[j];
        }
      }
      const size_t ow = P.alloc(key + ".wT", (size_t)n_in_pad * n_out), ob = P.alloc(key + ".b", n_out);
      for (int k = 0; k < n_in; ++k)
        for (int j = 0; j < n_out; ++j) P.arena[ow + (size_t)k * n_out + j] = (float)((double)w->d[(size_t)j * n_in + k] * sc[j]);
      for (int j = 0; j < n_out; ++j) P.arena[ob + j] = (float)((double)b->d[j] * sc[j] + sh[j]);
      return true;
    };
    bool ok = true;
    if (dff) {
      ok = pack_lin("lin1", "bn2", 720, 768, H, "ff1") && pack_lin("lin2", "bn3", H, H, H, "ff2") &&
           pack_lin("lin3", "bn4", H, H, H, "ff3") && pack_lin("lin4", "bn5", H, H, H, "ff4");
    } else if (H > 0) {
      ok = pack_lin("linear", "", 720, 768, H, "ff1");
    }
    if (!ok) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
  }
  // conv1 runs on FFMA with the fp32 weights; conv2..conv6 on tcgen05 with [tap][ci/8][hi co | lo co][8], the fp16
  // two-term split of w * 2^S (conv_split.cu)
  std::vector<float> wf;
  for (int i = 1; conv_net && i <= 6; ++i) {
    if (!pack_conv(P, i, cin[i], cout[i], wf)) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
    if (i == 1) {
      const size_t o = P.alloc("conv1.w", wf.size());
      memcpy(&P.arena[o], wf.data(), wf.size() * 4);
      continue;
    }
    char k2[32];
    snprintf(k2, sizeof k2, "conv%d.wtc", i);
    const int ci_n = cin[i], co_n = cout[i];
    float wmax = 0.f;
    for (float w : wf) wmax = std::max(wmax, fabsf(w));
    int S = 0;
    while (S < 14 && wmax * (float)(2 << S) <= 1024.f) ++S;        // max|w| * 2^S <= 1024
    e->tc_scale[i] = 1.0f / (float)(1 << S);
    const size_t n_half = (size_t)9 * 2 * ci_n * co_n;
    const size_t dst = P.alloc(k2, (n_half + 1) / 2);              // fp16 payload inside the float arena
    for (int tap = 0; tap < 9; ++tap)
      for (int ci = 0; ci < ci_n; ++ci)
        for (int co = 0; co < co_n; ++co) {
          const float w = wf[((size_t)ci * 9 + tap) * co_n + co] * (float)(1 << S);
          const __half hi = __float2half_rn(w);
          const __half lo = __float2half_rn(w - __half2float(hi));
          __half* base = reinterpret_cast<__half*>(&P.arena[dst]) + (size_t)tap * 2 * ci_n * co_n;
          // per 16-byte K chunk: rows [0,co_n) = hi, rows [co_n, 2 co_n) = lo  (one N = 2*C_out operand)
          const size_t off = ((size_t)(ci / 8) * (2 * co_n) + co) * 8 + (ci & 7);
          base[off] = hi;
          base[off + (size_t)co_n * 8] = lo;
        }
  }

  if (e->cfg.arch == NISQA_ARCH_ADAPT_SA_ATTFF) {
    const std::string td = "time_dependency.model.";
    // one SelfAttention stack (lib:945-1040): Linear(in -> 64) + LayerNorm + `layers` encoder layers.  `kp` prefixes the
    // arena keys ("" = time_dependency, "2" = time_dependency_2 of the double-ended model)
    auto pack_sa_stack = [&](const std::string& ck, const std::string& kp, int in_dim, int layers, bool cnn_order) -> bool {
      const TensorView* lw = P.get(ck + "linear.weight", {64, in_dim});
      const TensorView* lb = P.get(ck + "linear.bias", {64});
      const TensorView* ng = P.get(ck + "norm1.weight", {64});
      const TensorView* nb = P.get(ck + "norm1.bias", {64});
      if (!lw || !lb || !ng || !nb) return false;
      size_t o = P.alloc("lin" + kp + ".wT", (size_t)((in_dim + 63) / 64 * 64) * 64);      // (rows beyond in_dim stay zero)
      if (cnn_order) {
        // engine feature order k' = h*64 + c  <->  reference view(-1, 64*6) order c*6 + h (lib:706)
        for (int h = 0; h < 6; ++h)
          for (int c = 0; c < 64; ++c)
            for (int j = 0; j < 64; ++j) P.arena[o + ((size_t)h * 64 + c) * 64 + j] = lw->d[(size_t)j * 384 + c * 6 + h];
      } else {
        pack_linear_T(P, o, lw, 64, in_dim);
      }
      o = P.alloc("lin" + kp + ".b", 64); memcpy(&P.arena[o], lb->d, 256);
      o = P.alloc("ln" + kp + "0.g", 64); memcpy(&P.arena[o], ng->d, 256);
      o = P.alloc("ln" + kp + "0.b", 64); memcpy(&P.arena[o], nb->d, 256);
      for (int l = 0; l < layers; ++l) {
        char pf[96]; snprintf(pf, sizeof pf, "layers.%d.", l);
        char key[64];
        const std::string p = ck + pf;
        const TensorView* iw = P.get(p + "self_attn.in_proj_weight", {192, 64});
        const TensorView* ib = P.get(p + "self_attn.in_proj_bias", {192});
        const TensorView* ow = P.get(p + "self_attn.out_proj.weight", {64, 64});
        const TensorView* ob = P.get(p + "self_attn.out_proj.bias", {64});
        const TensorView* w1 = P.get(p + "linear1.weight", {64, 64});
        const TensorView* b1 = P.get(p + "linear1.bias", {64});
        const TensorView* w2 = P.get(p + "linear2.weight", {64, 64});
        const TensorView* b2 = P.get(p + "linear2.bias", {64});
        const TensorView* g1 = P.get(p + "norm1.weight", {64});
        const TensorView* e1 = P.get(p + "norm1.bias", {64});
        const TensorView* g2 = P.get(p + "norm2.weight", {64});
        const TensorView* e2 = P.get(p + "norm2.bias", {64});
        if (!iw || !ib || !ow || !ob || !w1 || !b1 || !w2 || !b2 || !g1 || !e1 || !g2 || !e2) return false;
        auto K = [&](const char* s2) { snprintf(key, sizeof key, "sa%s%d.%s", kp.c_str(), l, s2); return std::string(key); };
        o = P.alloc(K("qkvT"), 3 * 4096);
        for (int part = 0; part < 3; ++part) {
          const float sc = part == 0 ? 0.125f : 1.f;      // q * 1/sqrt(64): exact power of two
          for (int k = 0; k < 64; ++k)
            for (int j = 0; j < 64; ++j)
              P.arena[o + part * 4096 + k * 64 + j] = iw->d[(size_t)(part * 64 + j) * 64 + k] * sc;
        }
        o = P.alloc(K("qkvb"), 192);
        for (int j = 0; j < 192; ++j) P.arena[o + j] = ib->d[j] * (j < 64 ? 0.125f : 1.f);
        o = P.alloc(K("woT"), 4096); pack_linear_T(P, o, ow, 64, 64);
        o = P.alloc(K("bo"), 64); memcpy(&P.arena[o], ob->d, 256);
        o = P.alloc(K("w1T"), 4096); pack_linear_T(P, o, w1, 64, 64);
        o = P.alloc(K("b1"), 64); memcpy(&P.arena[o], b1->d, 256);
        o = P.alloc(K("w2T"), 4096); pack_linear_T(P, o, w2, 64, 64);
        o = P.alloc(K("b2"), 64); memcpy(&P.arena[o], b2->d, 256);
        o = P.alloc(K("ln1g"), 64); memcpy(&P.arena[o], g1->d, 256);
        o = P.alloc(K("ln1b"), 64); memcpy(&P.arena[o], e1->d, 256);
        o = P.alloc(K("ln2g"), 64); memcpy(&P.arena[o], g2->d, 256);
        o = P.alloc(K("ln2b"), 64); memcpy(&P.arena[o], e2->d, 256);
      }
      return true;
    };
    auto pack_pos_enc = [&](const std::string& ck, const std::string& key) -> int {
      auto it = P.t.find(ck + "pos_encoder.pe");                  // registered buffer [max_len, 1, 64] (lib:1051-1058)
      if (it == P.t.end() || it->second.nd != 3 || it->second.dims[1] != 1 || it->second.dims[2] != 64)
        return fail(e, NISQA_ERR_WEIGHTS, "missing tensor " + ck + "pos_encoder.pe");
      if (e->cfg.max_segments > 0 && it->second.dims[0] < e->cfg.max_segments)
        return fail(e, NISQA_ERR_WEIGHTS, "positional encoding shorter than ms_max_segments");
      const size_t o2 = P.alloc(key, (size_t)it->second.numel);
      memcpy(&P.arena[o2], it->second.d, (size_t)it->second.numel * 4);
      return 0;
    };
    // framewise features feeding the first stack: 384 (AdaptCNN, engine order), 720 (SkipCNN without Linear: padded to 768
    // with zero rows) or cnn_fc_out_h
    const int feat_dim = e->cfg.cnn_fc > 0 ? e->cfg.cnn_fc : (conv_net ? 384 : 720);
    if (conv_net && e->cfg.cnn_fc > 0) {
      // AdaptCNN's optional Linear (lib:682-684, 708-709): k-major, rows in the engine's feature order h*64 + c
      const int H = e->cfg.cnn_fc;
      const TensorView* w = P.get("cnn.model.fc.weight", {H, 384});
      const TensorView* b = P.get("cnn.model.fc.bias", {H});
      if (!w || !b) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
      const size_t ow = P.alloc("ffc.wT", (size_t)384 * H), ob = P.alloc("ffc.b", H);
      for (int h = 0; h < 6; ++h)
        for (int c = 0; c < 64; ++c)
          for (int j = 0; j < H; ++j) P.arena[ow + ((size_t)h * 64 + c) * H + j] = w->d[(size_t)j * 384 + c * 6 + h];
      memcpy(&P.arena[ob], b->d, (size_t)H * 4);
    }
    if (!pack_sa_stack(td, "", feat_dim, e->cfg.sa_layers, conv_net && e->cfg.cnn_fc == 0)) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
    if (e->cfg.double_ended || e->cfg.td2_layers > 0) {
      // time_dependency_2: behind the fusion of the double-ended model (input 192 / 128), or a second stack behind the
      // first one in NISQA / NISQA_DIM (lib:114-141, 236-268; input 64)
      const std::string td2 = "time_dependency_2.model.";
      int fdim = !e->cfg.double_ended ? 64 : (e->cfg.de_fuse == NISQA_DE_FUSE_XY_MINUS ? 192 : 128);
      if (e->cfg.double_ended && e->cfg.de_fuse_dim > 0) {        // Fusion.lin_fusion (lib:1399-1401)
        const int D = e->cfg.de_fuse_dim;
        const TensorView* w = P.get("fuse.lin_fusion.weight", {D, fdim});
        const TensorView* b = P.get("fuse.lin_fusion.bias", {D});
        if (!w || !b) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
        const size_t ow = P.alloc("defuse.wT", (size_t)fdim * D), ob = P.alloc("defuse.b", D);
        pack_linear_T(P, ow, w, D, fdim);
        memcpy(&P.arena[ob], b->d, (size_t)D * 4);
        fdim = D;
      }
      if (!pack_sa_stack(td2, "2", fdim, e->cfg.td2_layers, false)) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
      if (e->cfg.td2_pos_enc) { int rc = pack_pos_enc(td2, "pe2"); if (rc) return rc; }
      if (e->cfg.de_align == NISQA_DE_ALIGN_LUONG) {            // AttLuong: W = Linear(y_dim -> q_dim), lib:1348-1351
        const TensorView* w = P.get("align.att.W.weight", {64, 64});
        const TensorView* b = P.get("align.att.W.bias", {64});
        if (!w || !b) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
        size_t o = P.alloc("de.wT", 4096); pack_linear_T(P, o, w, 64, 64);
        o = P.alloc("de.b", 64); memcpy(&P.arena[o], b->d, 256);
      }
      if (e->cfg.de_align == NISQA_DE_ALIGN_BAHDANAU) {         // AttBahdanau: Wq, Wy (-> att_dim 128), v, lib:1329-1337
        const TensorView* wq = P.get("align.att.Wq.weight", {128, 64});
        const TensorView* bq = P.get("align.att.Wq.bias", {128});
        const TensorView* wy = P.get("align.att.Wy.weight", {128, 64});
        const TensorView* by = P.get("align.att.Wy.bias", {128});
        const TensorView* v = P.get("align.att.v.weight", {1, 128});
        if (!wq || !bq || !wy || !by || !v) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
        size_t o = P.alloc("de.wqT", 64 * 128); pack_linear_T(P, o, wq, 128, 64);
        o = P.alloc("de.bq", 128); memcpy(&P.arena[o], bq->d, 512);
        o = P.alloc("de.wyT", 64 * 128); pack_linear_T(P, o, wy, 128, 64);
        o = P.alloc("de.by", 128); memcpy(&P.arena[o], by->d, 512);
        o = P.alloc("de.v", 128); memcpy(&P.arena[o], v->d, 512);
      }
    }
    const int nh = e->cfg.n_out;
    auto head_prefix = [&](int h) {
      char pf[64];
      if (nh == 1) snprintf(pf, sizeof pf, "pool.model.");
      else snprintf(pf, sizeof pf, "pool_layers.%d.model.", h);   // head order mos,noi,dis,col,loud (lib:1461-1465)
      return std::string(pf);
    };
    if (e->cfg.pos_enc) { int rc = pack_pos_enc(td, "pe"); if (rc) return rc; }
    if (e->cfg.pool == NISQA_POOL_ATT_FF) {
    const size_t oW1 = P.alloc("pool.w1T", (size_t)nh * 64 * 128), ob1 = P.alloc("pool.b1", nh * 128),
                 ow2 = P.alloc("pool.w2", nh * 128), ob2 = P.alloc("pool.b2", nh),
                 ow3 = P.alloc("pool.w3", nh * 64), ob3 = P.alloc("pool.b3", nh);
    for (int h = 0; h < nh; ++h) {
      const std::string p = head_prefix(h);
      const TensorView* w1 = P.get(p + "linear1.weight", {128, 64});
      const TensorView* b1 = P.get(p + "linear1.bias", {128});
      const TensorView* w2 = P.get(p + "linear2.weight", {1, 128});
      const TensorView* b2 = P.get(p + "linear2.bias", {1});
      const TensorView* w3 = P.get(p + "linear3.weight", {1, 64});
      const TensorView* b3 = P.get(p + "linear3.bias", {1});
      if (!w1 || !b1 || !w2 || !b2 || !w3 || !b3) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
      pack_linear_T(P, oW1 + (size_t)h * 64 * 128, w1, 128, 64);
      memcpy(&P.arena[ob1 + h * 128], b1->d, 512);
      memcpy(&P.arena[ow2 + h * 128], w2->d, 512);
      P.arena[ob2 + h] = b2->d[0];
      memcpy(&P.arena[ow3 + h * 64], w3->d, 256);
      P.arena[ob3 + h] = b3->d[0];
    }
    } else {
      // PoolAtt: linear1 (64 -> 1 attention logit) + linear2 (64 -> 1); PoolAvg / PoolMax / PoolLastStep: linear (64 -> 1)
      const bool att = e->cfg.pool == NISQA_POOL_ATT;
      const size_t oa1 = P.alloc("pool.a1", nh * 64), oa1b = P.alloc("pool.a1b", nh),
                   ow3 = P.alloc("pool.w3", nh * 64), ob3 = P.alloc("pool.b3", nh);
      for (int h = 0; h < nh; ++h) {
        const std::string p = head_prefix(h);
        const TensorView* a1 = att ? P.get(p + "linear1.weight", {1, 64}) : nullptr;
        const TensorView* a1b = att ? P.get(p + "linear1.bias", {1}) : nullptr;
        const TensorView* w3 = P.get(p + (att ? "linear2.weight" : "linear.weight"), {1, 64});
        const TensorView* b3 = P.get(p + (att ? "linear2.bias" : "linear.bias"), {1});
        if ((att && (!a1 || !a1b)) || !w3 || !b3) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
        if (att) { memcpy(&P.arena[oa1 + h * 64], a1->d, 256); P.arena[oa1b + h] = a1b->d[0]; }
        memcpy(&P.arena[ow3 + h * 64], w3->d, 256);
        P.arena[ob3 + h] = b3->d[0];
      }
    }
  } else {
    const TensorView* fw = P.get("cnn.model.fc_out.weight", {20, 768});
    const TensorView* fb = P.get("cnn.model.fc_out.bias", {20});
    if (!fw || !fb) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
    size_t o = P.alloc("fc.wT", 768 * 20);
    // engine order k' = (h*2 + w)*64 + c  <->  reference view order c*12 + h*2 + w (lib:830)
    for (int hw = 0; hw < 12; ++hw)
      for (int c = 0; c < 64; ++c)
        for (int j = 0; j < 20; ++j) P.arena[o + ((size_t)hw * 64 + c) * 20 + j] = fw->d[(size_t)j * 768 + c * 12 + hw];
    o = P.alloc("fc.b", 32); memcpy(&P.arena[o], fb->d, 80);
    const std::string p = "time_dependency.model.lstm.";
    const size_t owi = P.alloc("lstm.wih", 2 * 512 * 20), owh = P.alloc("lstm.whh", 2 * 512 * 128),
                 obb = P.alloc("lstm.b", 2 * 512);
    for (int d = 0; d < 2; ++d) {
      const std::string sfx = d ? "_reverse" : "";
      const TensorView* wi = P.get(p + "weight_ih_l0" + sfx, {512, 20});
      const TensorView* wh = P.get(p + "weight_hh_l0" + sfx, {512, 128});
      const TensorView* bi = P.get(p + "bias_ih_l0" + sfx, {512});
      const TensorView* bh = P.get(p + "bias_hh_l0" + sfx, {512});
      if (!wi || !wh || !bi || !bh) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
      memcpy(&P.arena[owi + (size_t)d * 512 * 20], wi->d, 512 * 20 * 4);
      memcpy(&P.arena[owh + (size_t)d * 512 * 128], wh->d, 512 * 128 * 4);
      for (int g = 0; g < 512; ++g) P.arena[obb + d * 512 + g] = bi->d[g] + bh->d[g];
    }
    const TensorView* pw = P.get("pool.model.linear.weight", {1, 256});      // every pooling module of this arch: Linear(256 -> 1)
    const TensorView* pb = P.get("pool.model.linear.bias", {1});
    if (!pw || !pb) return fail(e, NISQA_ERR_WEIGHTS, P.missing);
    o = P.alloc("lastbi.w", 256); memcpy(&P.arena[o], pw->d, 1024);
    e->pool_bias_std = pb->d[0];
    o = P.alloc("pool.w3", 256); memcpy(&P.arena[o], pw->d, 1024);
    o = P.alloc("pool.b3", 1); P.arena[o] = pb->d[0];
    P.alloc("pool.a1", 1); P.alloc("pool.a1b", 1);
  }
  // conv1 is stored as [tap][16]: same as the generic [ci=1][tap][cout] packing.
  CK(e->warena.reserve(P.arena.size() * 4));
  CK(cudaMemcpy(e->warena.p, P.arena.data(), P.arena.size() * 4, cudaMemcpyHostToDevice));
  return 0;
}

const float* W(nisqa_engine* e, const std::string& key) {
  return e->warena.as<float>() + e->woff.at(key);
}

// ---------------------------------------------------------------- one pass over a run of clips
struct PassInput {
  int n_clips;
  const ClipPlan* plan;               // [n_clips]
  const int64_t* n_samples;           // [n_clips]
  // exactly one of the two sources:
  const void* const* host_pcm;        // per-clip host pointers, or
  const void* dev_pcm; const int64_t* dev_off;   // packed device buffer + element offsets
  int fmt;
  float* scores_dev_out;              // device destination [n_clips][n_out]
  int slot;                           // compute lane
  int stage;                          // staging slot
};

int lane_allgather(nisqa_engine* e, const float* src, float* dst, size_t count, cudaStream_t st);

int run_pass(nisqa_engine* e, const PassInput& in) {
  const nisqa_config& c = e->cfg;
  const int n = in.n_clips;
  const int std_mode = c.arch == NISQA_ARCH_STD_LSTM_LASTBI;
  const size_t esz = in.fmt == NISQA_FMT_F32 ? 4 : 2;
  // ---- tables
  std::vector<ClipDesc>& cl = e->last_clips;
  cl.assign(n, ClipDesc());
  std::vector<int> pair_prefix(n + 1, 0), seg_prefix(n + 1, 0), qt_prefix(n + 1, 0), qt64_prefix(n + 1, 0), by_len(n + 1, 0);
  long long pcm_elems = 0;
  int n_frames = 0, n_seg = 0, n_pairs = 0, n_qt = 0, n_qt64 = 0, Q = 1, max_pairs = 0, max_span = 0, max_n_seg = 0;
  for (int i = 0; i < n; ++i) {
    const ClipPlan& p = in.plan[i];
    ClipDesc& d = cl[i];
    const bool ok = p.run != 0;
    d.n_samples = (int)in.n_samples[i];
    d.fb_id = ok ? p.fb_id : 0;
    d.hop = p.hop; d.win = p.win;
    d.s0 = (c.n_fft - p.win) / 2 - c.n_fft / 2;      // pad_center lpad minus the reflect pad
    d.n_frames = ok ? p.n_frames : 0;
    d.n_seg = ok ? p.n_seg : 0;
    d.frame_off = n_frames; d.seg_off = n_seg; d.pair_off = n_pairs;
    if (in.host_pcm) { d.pcm_off = pcm_elems; pcm_elems += ((long long)in.n_samples[i] + 15) / 16 * 16; }
    else d.pcm_off = in.dev_off[i];
    pair_prefix[i] = n_pairs; seg_prefix[i] = n_seg; qt_prefix[i] = n_qt; qt64_prefix[i] = n_qt64;
    n_frames += d.n_frames; n_seg += d.n_seg;
    n_pairs += (d.n_frames + 1) / 2;
    max_pairs = std::max(max_pairs, (d.n_frames + 1) / 2);
    n_qt += (d.n_seg + 127) / 128;
    n_qt64 += (d.n_seg + 63) / 64;
    max_n_seg = std::max(max_n_seg, d.n_seg);
    if (ok) { Q = std::max(Q, (p.win + 1023) / 1024); max_span = std::max(max_span, p.hop + p.win); }
  }
  pair_prefix[n] = n_pairs; seg_prefix[n] = n_seg; qt_prefix[n] = n_qt; qt64_prefix[n] = n_qt64;
  for (int i = 0; i < n; ++i) by_len[i] = i;          // clips by decreasing length (batched BiLSTM groups)
  std::stable_sort(by_len.begin(), by_len.begin() + n, [&](int a, int b) { return cl[a].n_seg > cl[b].n_seg; });
  e->last_n_seg = n_seg; e->last_n_frames = n_frames;
  const int n_out = c.n_out;

  float* scores = in.scores_dev_out;
  Lane& LN = e->lanes[in.slot];
  Stage& SG = e->stages[in.stage];
  cudaStream_t st = LN.stream, cs = e->copy_stream;
  e->cur_stream = st;
  // the staging slot (pinned tables, device tables, PCM buffer) is reused every kStages-th pass; the
  // lane's activation workspaces are protected by stream order alone
  if (SG.busy) { CK(cudaEventSynchronize(SG.ev_done)); SG.busy = false; }
  SG.lane = in.slot;

  // ---- upload tables (one pinned block: ClipDesc[n] | 4 prefix arrays | clips by length)
  const size_t tb_clips = (size_t)n * sizeof(ClipDesc);
  const size_t tb_pref = (size_t)(n + 1) * 4;
  CK(SG.h_tables.reserve(tb_clips + 5 * tb_pref));
  char* ht = SG.h_tables.as<char>();
  memcpy(ht, cl.data(), tb_clips);
  memcpy(ht + tb_clips, pair_prefix.data(), tb_pref);
  memcpy(ht + tb_clips + tb_pref, seg_prefix.data(), tb_pref);
  memcpy(ht + tb_clips + 2 * tb_pref, qt_prefix.data(), tb_pref);
  memcpy(ht + tb_clips + 3 * tb_pref, qt64_prefix.data(), tb_pref);
  memcpy(ht + tb_clips + 4 * tb_pref, by_len.data(), tb_pref);
  CK(SG.clips.reserve(tb_clips));
  CK(SG.prefixes.reserve(5 * tb_pref));
  CK(SG.clipmax.reserve((size_t)n * 4));
  CK(cudaMemcpyAsync(SG.clips.p, ht, tb_clips, cudaMemcpyHostToDevice, cs));
  CK(cudaMemcpyAsync(SG.prefixes.p, ht + tb_clips, 5 * tb_pref, cudaMemcpyHostToDevice, cs));
  CK(cudaMemsetAsync(SG.clipmax.p, 0, (size_t)n * 4, cs));
  const ClipDesc* d_clips = SG.clips.as<ClipDesc>();
  unsigned* d_clipmax = SG.clipmax.as<unsigned>();
  const int* d_pair = SG.prefixes.as<int>();
  (void)d_pair;
  e->last_lane = in.slot;
  e->last_stage = in.stage;
  const int* d_seg = d_pair + (n + 1);
  const int* d_qt = d_pair + 2 * (n + 1);
  const int* d_qt64 = d_pair + 3 * (n + 1);
  const int* d_by_len = d_pair + 4 * (n + 1);

  if (n_seg == 0) {   // nothing valid in this pass: NaN scores
    CK(cudaEventRecord(SG.ev_copied, cs));
    CK(cudaStreamWaitEvent(st, SG.ev_copied, 0));
    CK(cudaMemsetAsync(scores, 0xFF, (size_t)n * n_out * 4, st));
  } else {
    // ---- PCM (copy stream), then hand over to the compute stream
    const void* d_pcm = in.dev_pcm;
    if (in.host_pcm) {
      CK(SG.pcm.reserve((size_t)pcm_elems * esz));
      // clips that are back to back in host memory with the same 16-element alignment as the
      // device packing travel as ONE copy (a pinned batch buffer becomes a single large DMA)
      for (int i = 0; i < n;) {
        if (cl[i].n_frames <= 0) { ++i; continue; }
        const char* h0 = static_cast<const char*>(in.host_pcm[i]);
        const long long o0 = cl[i].pcm_off;
        size_t bytes = (size_t)in.n_samples[i] * esz;
        int j = i + 1;
        while (j < n && cl[j].n_frames > 0 &&
               static_cast<const char*>(in.host_pcm[j]) == h0 + (size_t)(cl[j].pcm_off - o0) * esz) {
          bytes = (size_t)(cl[j].pcm_off - o0) * esz + (size_t)in.n_samples[j] * esz;
          ++j;
        }
        CK(cudaMemcpyAsync(SG.pcm.as<char>() + (size_t)o0 * esz, h0, bytes, cudaMemcpyHostToDevice, cs));
        i = j;
      }
      d_pcm = SG.pcm.p;
    }
    CK(cudaEventRecord(SG.ev_copied, cs));
    CK(cudaStreamWaitEvent(st, SG.ev_copied, 0));
    // ---- workspaces
    const int FEAT = std_mode ? 768 : 384;
    CK(LN.mel.reserve((size_t)n_frames * kMels * 4));
    CK(LN.segtab.reserve((size_t)n_seg * 12));
    const bool conv_net = c.cnn_kind == NISQA_CNN_CONV;
    const bool keep_pool1 = conv_net && e->keep_pool1;
    e->last_pool1 = keep_pool1;
    for (int l = keep_pool1 ? 2 : 3; conv_net && l <= 6; ++l) {
      // the lo plane sits at a fixed offset of the ALLOCATION (not of this pass's n_seg): the zero rows /
      // columns of both planes must stay where they were when the buffer was cleared
      CK(LN.planes[l].reserve_zeroed(2 * split_plane_bytes(std_mode, l, n_seg), st));
      LN.plane_bytes[l] = (LN.planes[l].cap / 2) & ~(size_t)1023;
    }
    CK(LN.feats.reserve((size_t)n_seg * FEAT * 4));
    int* seg_frame0 = LN.segtab.as<int>();
    float* seg_thr = reinterpret_cast<float*>(seg_frame0 + n_seg);
    int* seg_clip = seg_frame0 + 2 * (size_t)n_seg;

    { Scope s(e, "frontend");
      launch_frontend(st, d_pcm, in.fmt == NISQA_FMT_F32, d_clips, n, max_pairs,
                      e->fb_table.as<FbTables>(), e->tw4096.as<float2>(), LN.mel.as<float>(),
                      d_clipmax, Q, max_span, e->fe_ppc); }
    { Scope s(e, "seg_table");
      launch_seg_table(st, d_clips, n, d_seg, d_clipmax, c.seg_hop, n_seg,
                       seg_frame0, seg_thr, seg_clip); }
    auto plane_hi = [&](int l) { return LN.planes[l].as<char>(); };
    auto plane_lo = [&](int l) { return LN.planes[l].as<char>() + LN.plane_bytes[l]; };
    const float* sa_in = LN.feats.as<float>();       // rows fed to the first self-attention stack
    int sa_nk = 6;                                   // ... in 64-wide chunks
    if (!conv_net) {
      // SkipCNN / DFF (lib:504-583): BN + flatten (+ Linear layers), no convolution
      Scope s(e, "framewise", 5);
      const int H = c.cnn_fc;
      CK(LN.ffa.reserve((size_t)n_seg * std::max(768, H) * 4));
      launch_seg_feats(st, LN.mel.as<float>(), seg_frame0, seg_thr, W(e, "ff.bn"), n_seg, LN.ffa.as<float>());
      sa_in = LN.ffa.as<float>(); sa_nk = 12;
      if (H > 0) {
        CK(LN.ffb.reserve((size_t)n_seg * H * 4));
        const bool dff = c.cnn_kind == NISQA_CNN_DFF;
        launch_linear_tile(st, LN.ffa.as<float>(), 768, W(e, "ff1.wT"), W(e, "ff1.b"), dff, LN.ffb.as<float>(), H, n_seg, 768, H);
        sa_in = LN.ffb.as<float>(); sa_nk = H / 64;
        if (dff) {
          float* pp2[2] = {LN.ffa.as<float>(), LN.ffb.as<float>()};
          const char* keys[3] = {"ff2", "ff3", "ff4"};
          for (int l = 0; l < 3; ++l)       // ffb -> ffa -> ffb -> ffa
            launch_linear_tile(st, pp2[(l + 1) & 1], H, W(e, std::string(keys[l]) + ".wT"), W(e, std::string(keys[l]) + ".b"), 1,
                               pp2[l & 1], H, n_seg, H, H);
          sa_in = LN.ffa.as<float>();
        }
      }
    } else {
      if (keep_pool1) {     // (not a "conv*" scope: the cnn group and the per-kernel tables count the product path only)
        Scope s(e, "pool1_dump");
        launch_conv1(st, std_mode, LN.mel.as<float>(), seg_frame0, seg_thr, W(e, "conv1.w"), W(e, "conv1.b"),
                     plane_hi(2), plane_lo(2), n_seg);
      }
      { Scope s(e, "conv12");
        launch_conv12(st, std_mode, LN.mel.as<float>(), seg_frame0, seg_thr, W(e, "conv1.w"), W(e, "conv1.b"),
                      W(e, "conv2.wtc"), W(e, "conv2.b"), e->tc_scale[2], plane_hi(3), plane_lo(3), n_seg); }
      for (int l = 3; l <= 6; ++l) {
        char nm[16], kt[24], kb[24];
        snprintf(nm, sizeof nm, "conv%d", l);
        snprintf(kt, sizeof kt, "conv%d.wtc", l); snprintf(kb, sizeof kb, "conv%d.b", l);
        Scope s(e, nm);
        launch_conv_split(st, std_mode, l, plane_hi(l), plane_lo(l), W(e, kt), W(e, kb), e->tc_scale[l],
                          l < 6 ? plane_hi(l + 1) : nullptr, l < 6 ? plane_lo(l + 1) : nullptr,
                          l == 6 ? LN.feats.as<float>() : nullptr, n_seg);
      }
    }

    if (conv_net && c.cnn_fc > 0) {      // AdaptCNN's Linear behind conv6 (lib:708-709)
      Scope s(e, "framewise");
      CK(LN.ffb.reserve((size_t)n_seg * c.cnn_fc * 4));
      launch_linear_tile(st, LN.feats.as<float>(), 384, W(e, "ffc.wT"), W(e, "ffc.b"), 0, LN.ffb.as<float>(), c.cnn_fc, n_seg, 384, c.cnn_fc);
      sa_in = LN.ffb.as<float>(); sa_nk = c.cnn_fc / 64;
    }
    if (!std_mode) {
      CK(LN.xa.reserve((size_t)n_seg * 64 * 4));
      CK(LN.xb.reserve((size_t)n_seg * 64 * 4));
      CK(LN.qkv.reserve((size_t)n_seg * 192 * 4));
      CK(LN.logits.reserve((size_t)n_seg * n_out * 4));
      CK(LN.tdout.reserve((size_t)n_seg * 64 * 4));
      const bool attff = c.pool == NISQA_POOL_ATT_FF;
      PoolHeadParams H = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
      if (attff) {
        H.W1T = W(e, "pool.w1T"); H.b1 = W(e, "pool.b1"); H.w2 = W(e, "pool.w2"); H.b2 = W(e, "pool.b2");
      }
      H.w3 = W(e, "pool.w3"); H.b3 = W(e, "pool.b3");
      e->last_td_in = LN.tdout.as<float>();
      const float* cur = LN.tdout.as<float>();
      float* pp[2] = {LN.xa.as<float>(), LN.xb.as<float>()};
      // Linear+LN (+positional encoding, +QKV of layer 0) | per layer: attention + out_proj + FFN + LNs (+ next QKV, or
      // the PoolAttFF logits behind the last layer) | per-clip pooling.  qkv ping-pongs between two buffers: a layer's
      // CTAs read keys / values of rows whose next-layer projection other CTAs are already writing.
      CK(LN.qkv2.reserve((size_t)n_seg * 192 * 4));
      float* qk[2] = {LN.qkv.as<float>(), LN.qkv2.as<float>()};
      const bool de = c.double_ended != 0;
      // one SelfAttention stack; `kp` = "" (time_dependency) or "2" (time_dependency_2); the stack that feeds the pooling
      // module computes the PoolAttFF logits behind its last layer
      auto sa_stack = [&](const std::string& kp, const float* in_rows, int nk, int layers, bool pos_enc, bool feeds_pool,
                          float* x0) -> const float* {
        auto key = [&](int l, const char* s2) { char k[40]; snprintf(k, sizeof k, "sa%s%d.%s", kp.c_str(), l, s2); return std::string(k); };
        auto params = [&](int l) {
          SaLayerParams P;
          P.WoT = W(e, key(l, "woT")); P.bo = W(e, key(l, "bo")); P.W1T = W(e, key(l, "w1T")); P.b1 = W(e, key(l, "b1"));
          P.W2T = W(e, key(l, "w2T")); P.b2 = W(e, key(l, "b2")); P.ln1_g = W(e, key(l, "ln1g")); P.ln1_b = W(e, key(l, "ln1b"));
          P.ln2_g = W(e, key(l, "ln2g")); P.ln2_b = W(e, key(l, "ln2b"));
          return P;
        };
        { Scope s(e, "lin_ln");
          launch_td_in(st, in_rows, W(e, "lin" + kp + ".wT"), nk, W(e, "lin" + kp + ".b"), W(e, "ln" + kp + "0.g"), W(e, "ln" + kp + "0.b"),
                       W(e, key(0, "qkvT")), W(e, key(0, "qkvb")), pos_enc ? W(e, kp.empty() ? "pe" : "pe2") : nullptr, seg_clip, d_clips,
                       x0, qk[0], n_seg); }
        const float* cur2 = x0;
        for (int l = 0; l < layers; ++l) {
          const bool last = l + 1 == layers;
          Scope s(e, "sa_layer");
          launch_td_sa(st, cur2, qk[l & 1], d_clips, n, d_qt64, n_qt64, params(l), pp[l & 1],
                       last ? nullptr : W(e, key(l + 1, "qkvT")), last ? nullptr : W(e, key(l + 1, "qkvb")),
                       qk[(l + 1) & 1], H, (feeds_pool && attff) ? n_out : 0, LN.logits.as<float>());
          cur2 = pp[l & 1];
        }
        return cur2;
      };
      const bool td2_single = !de && c.td2_layers > 0;      // NISQA / NISQA_DIM with td_2 = 'self_att'
      cur = sa_stack("", sa_in, sa_nk, c.sa_layers, c.pos_enc != 0, !de && !td2_single, LN.tdout.as<float>());
      if (td2_single) {
        CK(LN.td2in.reserve((size_t)n_seg * 64 * 4));
        cur = sa_stack("2", cur, 1, c.td2_layers, c.td2_pos_enc != 0, true, LN.td2in.as<float>());
      }
      if (de) {
        // NISQA_DE (lib:404-424): align the reference clip's rows to the degraded clip's, fuse, second time-dependency stack
        const int nf = c.de_fuse == NISQA_DE_FUSE_XY_MINUS ? 3 : 2;
        CK(LN.fused.reserve((size_t)n_seg * 64 * nf * 4));
        CK(LN.td2in.reserve((size_t)n_seg * 64 * 4));
        CK(cudaMemsetAsync(LN.fused.p, 0, (size_t)n_seg * 64 * nf * 4, st));      // rows of the reference clips stay zero
        DeAlignParams AP = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
        if (c.de_align == NISQA_DE_ALIGN_LUONG) { AP.wT = W(e, "de.wT"); AP.b = W(e, "de.b"); }
        if (c.de_align == NISQA_DE_ALIGN_BAHDANAU) {
          AP.wqT = W(e, "de.wqT"); AP.bq = W(e, "de.bq"); AP.wyT = W(e, "de.wyT"); AP.by = W(e, "de.by"); AP.v = W(e, "de.v");
        }
        { Scope s(e, "de_align");
          launch_de_align(st, cur, d_clips, n, d_qt64, n_qt64, c.de_align, c.de_align_apply == NISQA_DE_APPLY_SOFT, c.de_fuse,
                          AP, LN.fused.as<float>()); }
        const float* td2_rows = LN.fused.as<float>();
        int td2_nk = nf;
        if (c.de_fuse_dim > 0) {         // Fusion.lin_fusion (lib:1414-1415)
          Scope s(e, "de_align");
          CK(LN.ffa.reserve((size_t)n_seg * c.de_fuse_dim * 4));
          launch_linear_tile(st, LN.fused.as<float>(), 64 * nf, W(e, "defuse.wT"), W(e, "defuse.b"), 0, LN.ffa.as<float>(), c.de_fuse_dim,
                             n_seg, 64 * nf, c.de_fuse_dim);
          td2_rows = LN.ffa.as<float>(); td2_nk = c.de_fuse_dim / 64;
        }
        cur = sa_stack("2", td2_rows, td2_nk, c.td2_layers, c.td2_pos_enc != 0, true, LN.td2in.as<float>());
      }
      e->last_td_out = cur;
      { Scope s(e, "pool");
        if (attff) launch_pool_final(st, cur, LN.logits.as<float>(), d_clips, n, H, n_out, max_n_seg, scores);
        else {
          PoolSimpleParams Q = {W(e, "pool.a1"), W(e, "pool.a1b"), W(e, "pool.w3"), W(e, "pool.b3")};
          launch_pool_simple(st, cur, 64, d_clips, n, c.pool, Q, n_out, max_n_seg, scores);
        }
        if (de) launch_de_finalize(st, d_clips, n, n_out, scores); }
    } else {
      CK(LN.feats20.reserve((size_t)n_seg * 20 * 4));
      CK(LN.tdout.reserve((size_t)n_seg * 256 * 4));
      CK(LN.partial.reserve((size_t)n * 2 * 4));
      { Scope s(e, "fc_out"); launch_fc20(st, LN.feats.as<float>(), W(e, "fc.wT"), W(e, "fc.b"), LN.feats20.as<float>(), n_seg); }
      LstmParams L;
      L.w_ih = W(e, "lstm.wih"); L.w_hh = W(e, "lstm.whh"); L.b = W(e, "lstm.b"); L.w_pool = W(e, "lastbi.w");
      const bool lastbi = c.pool == NISQA_POOL_LAST_STEP_BI;
      const bool keep = e->keep_td_out || !lastbi;        // the other pooling modules read every step's output
      { Scope s(e, "lstm", 2);
        launch_lstm_batched(st, LN.feats20.as<float>(), d_clips, d_by_len, n, L, keep ? LN.tdout.as<float>() : nullptr,
                            LN.partial.as<float>(), e->pool_bias_std, lastbi ? scores : nullptr); }
      if (!lastbi) {
        Scope s(e, "pool");
        PoolSimpleParams Q = {W(e, "pool.a1"), W(e, "pool.a1b"), W(e, "pool.w3"), W(e, "pool.b3")};
        launch_pool_simple(st, LN.tdout.as<float>(), 256, d_clips, n, c.pool, Q, 1, max_n_seg, scores);
      }
      e->last_td_in = nullptr;
      e->last_td_out = keep ? LN.tdout.as<float>() : nullptr;
    }
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(SG.ev_done, st));
  SG.busy = true;
  return 0;
}

int predict_common(nisqa_engine* e, int n_clips, const void* const* host_pcm, const void* dev_pcm,
                   const int64_t* dev_off, const int64_t* n_samples, const int32_t* sample_rate,
                   int fmt, float* scores_host, float* scores_dev, int32_t* n_seg_out,
                   int32_t* status_out, int sync, int64_t* ticket_out = nullptr) {
  if (!e) return NISQA_ERR_INVALID;
  if (!e->weights_loaded) return fail(e, NISQA_ERR_STATE, "nisqa_load_weights has not been called");
  if (n_clips < 0 || (n_clips > 0 && (!n_samples || !sample_rate)))
    return fail(e, NISQA_ERR_INVALID, "null argument");
  if (fmt != NISQA_FMT_S16 && fmt != NISQA_FMT_F32) return fail(e, NISQA_ERR_INVALID, "sample_fmt");
  CK(cudaSetDevice(e->device));
  for (auto& t : e->timers) { t.ms = 0.0; t.launches = 0; }
  std::vector<ClipPlan> plan(n_clips);
  for (int i = 0; i < n_clips; ++i) {
    if (n_samples[i] > (int64_t)INT32_MAX) return fail(e, NISQA_ERR_INVALID, "clip longer than 2^31 samples");
    plan_clip(e->cfg, n_samples[i], sample_rate[i], &plan[i]);
    if (plan[i].status == NISQA_CLIP_OK) {
      int rc = build_fb(e, sample_rate[i], plan[i].hop, plan[i].win, &plan[i].fb_id);
      if (rc) return rc;
    }
    plan[i].run = plan[i].status == NISQA_CLIP_OK;
    if (n_seg_out) n_seg_out[i] = plan[i].n_seg;
    if (status_out) status_out[i] = plan[i].status;
  }
  const int unit = e->cfg.double_ended ? 2 : 1;      // clips travel in (degraded, reference) pairs through a double-ended engine
  if (e->cfg.double_ended) {
    if (n_clips & 1) return fail(e, NISQA_ERR_INVALID, "a double-ended engine takes clips in (degraded, reference) pairs: n_clips must be even");
    for (int i = 0; i < n_clips; i += 2)
      if (!plan[i].run || !plan[i + 1].run) plan[i].run = plan[i + 1].run = 0;      // the pair scores NaN
  }
  // segments per internal pass: 131072 segments keep ~8 GB of activation planes per compute lane (sized for the
  // 180 GB of a B200) and give the BiLSTM >= 128 clips per launch at configs[3]; one 64-clip batch is 15 808
  const int max_seg = e->cfg.max_chunk_segments > 0 ? e->cfg.max_chunk_segments : 131072;
  float* scores_all = scores_dev;
  if (!scores_all) {
    DevBuf& sb = ticket_out ? e->tickets[e->next_ticket % kStages].scores : e->scores;
    CK(sb.reserve((size_t)std::max(n_clips, 1) * e->cfg.n_out * 4));
    scores_all = sb.as<float>();
  }
  const int64_t first_pass = e->pass_counter;
  int i0 = 0;
  e->last_passes = 0;
  while (i0 < n_clips) {
    int i1 = i0; long long segs = 0;
    while (i1 < n_clips) {
      long long s = 0;
      for (int u = 0; u < unit; ++u) s += plan[i1 + u].run ? plan[i1 + u].n_seg : 0;
      if (i1 > i0 && (segs + s > max_seg || i1 - i0 >= 32768)) break;      // (clips ride in grid.y of the front-end: < 65536)
      segs += s; i1 += unit;
    }
    PassInput in;
    in.n_clips = i1 - i0; in.plan = plan.data() + i0; in.n_samples = n_samples + i0;
    in.host_pcm = host_pcm ? host_pcm + i0 : nullptr;
    in.dev_pcm = dev_pcm; in.dev_off = dev_off ? dev_off + i0 : nullptr;
    in.fmt = fmt;
    in.scores_dev_out = scores_all + (size_t)i0 * e->cfg.n_out;
    in.slot = e->profiling ? 0 : (int)(e->pass_counter % kLanes);
    in.stage = (int)(e->pass_counter % kStages);
    ++e->pass_counter;
    int rc = run_pass(e, in);
    if (rc) return rc;
    ++e->last_passes;
    i0 = i1;
  }
  // the lane of the last pass collects: it waits for the other lanes this call used
  const int n_pass = (int)(e->pass_counter - first_pass);
  cudaStream_t fin = e->lanes[e->last_lane].stream;
  if (n_pass == 0) fin = e->lanes[0].stream;
  for (int k = 0; k < kStages && n_pass > 1; ++k)      // passes of this call that ran on other lanes
    if (e->stages[k].busy && e->stages[k].lane != e->last_lane) CK(cudaStreamWaitEvent(fin, e->stages[k].ev_done, 0));
  if (e->gather_dst && e->nccl_comm && n_clips == e->gather_rows && (ticket_out || scores_dev)) {
    // the path's single exchange step, enqueued behind this call's kernels on its own lane
    int rc = lane_allgather(e, scores_all, e->gather_dst, (size_t)n_clips * e->cfg.n_out, fin);
    if (rc) return rc;
    CK(cudaEventRecord(e->stages[e->last_stage].ev_done, fin));
  }
  if (ticket_out) {
    // asynchronous completion: scores land in the ticket's pinned block; nisqa_wait hands them over
    Ticket& tk = e->tickets[e->next_ticket % kStages];
    tk.bytes = (size_t)n_clips * e->cfg.n_out * 4;
    tk.user_scores = scores_host;
    CK(tk.pinned.reserve(std::max<size_t>(tk.bytes, 16)));
    if (tk.bytes) CK(cudaMemcpyAsync(tk.pinned.p, scores_all, tk.bytes, cudaMemcpyDeviceToHost, fin));
    if (!tk.done) CK(cudaEventCreateWithFlags(&tk.done, cudaEventDisableTiming));
    CK(cudaEventRecord(tk.done, fin));
    tk.active = true;
    tk.id = e->next_ticket++;
    *ticket_out = tk.id;
    return 0;
  }
  if (scores_host && n_clips > 0) {
    const size_t bytes = (size_t)n_clips * e->cfg.n_out * 4;
    CK(e->h_scores.reserve(bytes));
    CK(cudaMemcpyAsync(e->h_scores.p, scores_all, bytes, cudaMemcpyDeviceToHost, fin));
    CK(cudaStreamSynchronize(fin));
    memcpy(scores_host, e->h_scores.p, bytes);
  }
  if (sync || scores_host || e->profiling) CK(cudaStreamSynchronize(fin));
  if (e->profiling) collect_timers(e);
  return 0;
}

int finish_ticket(nisqa_engine* e, Ticket& tk) {
  if (!tk.active) return 0;
  CK(cudaEventSynchronize(tk.done));
  if (tk.bytes && tk.user_scores) memcpy(tk.user_scores, tk.pinned.p, tk.bytes);
  tk.active = false;
  return 0;
}

}  // namespace

// ======================================================================== C ABI
extern "C" {

int nisqa_create(nisqa_engine** out, int device, const nisqa_config* cfg) {
  if (!out || !cfg) return NISQA_ERR_INVALID;
  *out = nullptr;
  nisqa_engine* e = new nisqa_engine();
  e->cfg = *cfg; e->device = device;
  *out = e;     // returned even on failure so that nisqa_last_error() can be read
  if (cfg->abi_version != NISQA_B200_ABI_VERSION) return fail(e, NISQA_ERR_INVALID, "abi_version mismatch");
  if (cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF && cfg->arch != NISQA_ARCH_STD_LSTM_LASTBI)
    return fail(e, NISQA_ERR_INVALID, "unsupported architecture");
  if (cfg->n_fft != kNfft || cfg->n_mels != kMels || cfg->seg_len != kSegLen)
    return fail(e, NISQA_ERR_INVALID, "engine is built for n_fft=4096, n_mels=48, seg_length=15");
  if (cfg->n_out != 1 && cfg->n_out != 5) return fail(e, NISQA_ERR_INVALID, "n_out must be 1 or 5");
  if (cfg->arch == NISQA_ARCH_STD_LSTM_LASTBI && cfg->n_out != 1) return fail(e, NISQA_ERR_INVALID, "n_out");
  if (cfg->seg_hop < 1 || cfg->hop_s <= 0 || cfg->win_s <= 0 || cfg->fmax <= 0)
    return fail(e, NISQA_ERR_INVALID, "bad front-end parameters");
  if (cfg->arch == NISQA_ARCH_ADAPT_SA_ATTFF && (cfg->sa_layers < 1 || cfg->sa_layers > 8))
    return fail(e, NISQA_ERR_INVALID, "sa_layers");
  if (cfg->pool < NISQA_POOL_ATT_FF || cfg->pool > NISQA_POOL_LAST_STEP_BI ||
      (cfg->arch == NISQA_ARCH_ADAPT_SA_ATTFF && cfg->pool == NISQA_POOL_LAST_STEP_BI) ||
      (cfg->arch == NISQA_ARCH_STD_LSTM_LASTBI && (cfg->pool == NISQA_POOL_ATT_FF || cfg->pool == NISQA_POOL_ATT)))
    return fail(e, NISQA_ERR_INVALID, "pooling module not available for this architecture");
  if (cfg->pos_enc && cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF) return fail(e, NISQA_ERR_INVALID, "pos_enc needs the self-attention architecture");
  if (cfg->cnn_kind < NISQA_CNN_CONV || cfg->cnn_kind > NISQA_CNN_DFF || cfg->cnn_fc < 0 || cfg->cnn_fc % 64 != 0 || cfg->cnn_fc > 8192 ||
      (cfg->cnn_kind == NISQA_CNN_DFF && cfg->cnn_fc == 0) || (cfg->cnn_fc != 0 && cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF) ||
      (cfg->cnn_kind != NISQA_CNN_CONV && cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF) ||
      cfg->de_fuse_dim < 0 || cfg->de_fuse_dim % 64 != 0 || cfg->de_fuse_dim > 8192 || (cfg->de_fuse_dim != 0 && !cfg->double_ended))
    return fail(e, NISQA_ERR_INVALID, "cnn_kind / cnn_fc: SkipCNN and DFF feed the self-attention architecture; cnn_fc_out_h a multiple of 64");
  if (cfg->td2_layers < 0 || cfg->td2_layers > 8 || (cfg->td2_layers > 0 && cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF))
    return fail(e, NISQA_ERR_INVALID, "td_2 = 'self_att' needs the self-attention architecture (td2_layers 0..8)");
  if (cfg->double_ended) {
    if (cfg->arch != NISQA_ARCH_ADAPT_SA_ATTFF || cfg->n_out != 1)
      return fail(e, NISQA_ERR_INVALID, "NISQA_DE: AdaptCNN + self-attention, one output");
    if (cfg->de_align < NISQA_DE_ALIGN_DOT || cfg->de_align > NISQA_DE_ALIGN_BAHDANAU)
      return fail(e, NISQA_ERR_INVALID, "de_align: dot, cosine, distance, luong or bahd");
    if (cfg->de_align_apply != NISQA_DE_APPLY_HARD && cfg->de_align_apply != NISQA_DE_APPLY_SOFT)
      return fail(e, NISQA_ERR_INVALID, "de_align_apply");
    if (cfg->de_fuse < NISQA_DE_FUSE_XY_MINUS || cfg->de_fuse > NISQA_DE_FUSE_XY) return fail(e, NISQA_ERR_INVALID, "de_fuse");
    if (cfg->td2_layers < 1 || cfg->td2_layers > 8) return fail(e, NISQA_ERR_INVALID, "td_2 must be a self-attention stack (td2_layers 1..8)");
  }
  int count = 0;
  CK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(e, NISQA_ERR_CUDA, "no such CUDA device (there is no CPU fallback)");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(e, NISQA_ERR_CUDA, "libnisqa_b200 is compiled for sm_100a only");
  CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
  for (auto& l : e->lanes) CK(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
  for (auto& g : e->stages) {
    CK(cudaEventCreateWithFlags(&g.ev_copied, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&g.ev_done, cudaEventDisableTiming));
  }
  e->stream = e->lanes[0].stream;
  e->cur_stream = e->stream;
  // twiddles laid out per lane so that every warp load is coalesced:
  //   tw1[r-1][j][lane] = W_4096^(r*(lane+32j)),  tw2[q][lane] = W_1024^(lane*q)
  std::vector<float2> tw(6 * 1024);     // tw1 [3][32][32], tw2 [32][32], then tw2 again as (x, y, -y, x) float4 [32][32]
  auto w4096 = [](long k) {
    const double a = -2.0 * M_PI * (double)(k & 4095) / 4096.0;
    return make_float2((float)cos(a), (float)sin(a));
  };
  for (int r = 1; r <= 3; ++r)
    for (int j = 0; j < 32; ++j)
      for (int l = 0; l < 32; ++l) tw[((r - 1) * 32 + j) * 32 + l] = w4096((long)r * (l + 32 * j));
  for (int q = 0; q < 32; ++q)
    for (int l = 0; l < 32; ++l) {
      const float2 t = w4096(4L * l * q);
      tw[3 * 1024 + q * 32 + l] = t;
      tw[4 * 1024 + 2 * (q * 32 + l)] = t;
      tw[4 * 1024 + 2 * (q * 32 + l) + 1] = make_float2(-t.y, t.x);
    }
  CK(e->tw4096.reserve(tw.size() * sizeof(float2)));
  CK(cudaMemcpy(e->tw4096.p, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice));
  return 0;
}

void nisqa_destroy(nisqa_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  delete e;
}

const char* nisqa_last_error(const nisqa_engine* e) { return e ? e->err.c_str() : "null engine"; }

int nisqa_load_weights(nisqa_engine* e, const nisqa_tensor* tensors, int n) {
  if (!e || !tensors || n <= 0) return NISQA_ERR_INVALID;
  if (!e->stream) return fail(e, NISQA_ERR_STATE, "engine was not created successfully");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  int rc = pack_weights(e, tensors, n);
  if (rc) return rc;
  e->weights_loaded = true;
  return 0;
}

int nisqa_predict_pcm(nisqa_engine* e, int n_clips, const void* const* pcm, const int64_t* n_samples,
                      const int32_t* sample_rate, int sample_fmt, float* scores_out,
                      int32_t* n_segments_out, int32_t* status_out) {
  if (!e) return NISQA_ERR_INVALID;
  if (n_clips > 0 && (!pcm || !scores_out)) return fail(e, NISQA_ERR_INVALID, "null argument");
  for (auto& tk : e->tickets) { int rc = finish_ticket(e, tk); if (rc) return rc; }
  return predict_common(e, n_clips, pcm, nullptr, nullptr, n_samples, sample_rate, sample_fmt,
                        scores_out, nullptr, n_segments_out, status_out, 1);
}

int nisqa_submit_pcm(nisqa_engine* e, int n_clips, const void* const* pcm, const int64_t* n_samples,
                     const int32_t* sample_rate, int sample_fmt, float* scores_out,
                     int32_t* n_segments_out, int32_t* status_out, int64_t* ticket) {
  if (!e || !ticket) return NISQA_ERR_INVALID;
  if (n_clips > 0 && (!pcm || !scores_out)) return fail(e, NISQA_ERR_INVALID, "null argument");
  if (e->profiling) return fail(e, NISQA_ERR_STATE, "profiling needs the synchronous entry points");
  int rc = finish_ticket(e, e->tickets[e->next_ticket % kStages]);      // at most kStages submissions in flight
  if (rc) return rc;
  return predict_common(e, n_clips, pcm, nullptr, nullptr, n_samples, sample_rate, sample_fmt,
                        scores_out, nullptr, n_segments_out, status_out, 0, ticket);
}

int nisqa_wait(nisqa_engine* e, int64_t ticket) {
  if (!e) return NISQA_ERR_INVALID;
  CK(cudaSetDevice(e->device));
  // tickets complete in submission order: finish everything up to and including `ticket`
  for (int64_t id = ticket - kStages; id <= ticket; ++id)
    for (auto& tk : e->tickets)
      if (tk.active && tk.id == id) { int rc = finish_ticket(e, tk); if (rc) return rc; }
  return 0;
}

int nisqa_drain(nisqa_engine* e) {
  if (!e || !e->stream) return NISQA_ERR_INVALID;
  cudaSetDevice(e->device);
  // abandon every submission in flight: wait for the device, deliver nothing (the caller's score / PCM buffers
  // may already be gone - that is what this call is for)
  cudaError_t err = cudaDeviceSynchronize();
  for (auto& tk : e->tickets) { tk.active = false; tk.user_scores = nullptr; }
  for (auto& g : e->stages) g.busy = false;
  if (err != cudaSuccess) return fail(e, NISQA_ERR_CUDA, std::string("cudaDeviceSynchronize: ") + cudaGetErrorString(err));
  return 0;
}

int nisqa_predict_pcm_device(nisqa_engine* e, int n_clips, const void* pcm_dev, const int64_t* pcm_offsets,
                             const int64_t* n_samples, const int32_t* sample_rate, int sample_fmt,
                             float* scores_dev, int32_t* n_segments_out, int32_t* status_out, int sync) {
  if (!e) return NISQA_ERR_INVALID;
  if (n_clips > 0 && (!pcm_dev || !pcm_offsets || !scores_dev)) return fail(e, NISQA_ERR_INVALID, "null argument");
  return predict_common(e, n_clips, nullptr, pcm_dev, pcm_offsets, n_samples, sample_rate, sample_fmt,
                        nullptr, scores_dev, n_segments_out, status_out, sync);
}


// ---- device resampler of the ingest (SURVEY.md 8f.2): host clips at their own rates -> packed float32 PCM at
// `target` Hz in e->rs_out (clip i at element offset offs[i], n_fix[i] samples), on lane 0's stream (synchronised).
static int resample_to_device(nisqa_engine* e, int n_clips, const void* const* pcm, const int64_t* n_samples,
                              const int32_t* sample_rate, int fmt, int32_t target, std::vector<int64_t>* offs,
                              std::vector<int64_t>* n_fix) {
  if (fmt != NISQA_FMT_S16 && fmt != NISQA_FMT_F32) return fail(e, NISQA_ERR_INVALID, "sample_fmt");
  if (target <= 0) return fail(e, NISQA_ERR_INVALID, "target sample rate");
  CK(cudaSetDevice(e->device));
  cudaStream_t st = e->lanes[0].stream;
  if (!e->rs_nwin) {
    std::vector<double> win;
    int num_table = 0;
    if (!resample_table(&win, &num_table))
      return fail(e, NISQA_ERR_STATE, "nisqa_resample_set_filter has not been called (the interpolation table)");
    CK(e->rs_win.reserve(win.size() * 8));
    CK(cudaMemcpy(e->rs_win.p, win.data(), win.size() * 8, cudaMemcpyHostToDevice));
    e->rs_nwin = (int)win.size(); e->rs_num_table = num_table;
  }
  const size_t esz = fmt == NISQA_FMT_F32 ? 4 : 2;
  std::vector<ResampleClip> rc(n_clips);
  offs->assign(n_clips, 0); n_fix->assign(n_clips, 0);
  long long in_elems = 0, out_elems = 0, t_entries = 0;
  int max_fix = 0;
  for (int i = 0; i < n_clips; ++i) {
    if (n_samples[i] < 0 || n_samples[i] > (int64_t)INT32_MAX / 4 || sample_rate[i] <= 0)
      return fail(e, NISQA_ERR_INVALID, "resample: clip length / sample rate");
    ResampleClip& c = rc[i];
    c.n_in = (int)n_samples[i];
    c.copy = sample_rate[i] == target;
    c.ratio = (double)target / (double)sample_rate[i];
    c.n_out = c.copy ? c.n_in : (int)((double)c.n_in * c.ratio);                      // resampy: int(shape * ratio)
    c.n_fix = c.copy ? c.n_in : (int)ceil((double)c.n_in * c.ratio);                  // librosa fix_length
    if (!c.copy && c.n_out < 1) return fail(e, NISQA_ERR_INVALID, "resample: signal too short for the target rate");
    c.in_off = in_elems; in_elems += ((long long)c.n_in + 15) / 16 * 16;
    c.out_off = out_elems; out_elems += ((long long)c.n_fix + 15) / 16 * 16;
    c.time_off = t_entries; t_entries += (c.n_fix + 255) / 256 + 1;
    (*offs)[i] = c.out_off; (*n_fix)[i] = c.n_fix;
    max_fix = std::max(max_fix, c.n_fix);
  }
  if (n_clips == 0) return 0;
  CK(e->rs_raw.reserve((size_t)std::max<long long>(in_elems, 16) * esz));
  CK(e->rs_out.reserve((size_t)std::max<long long>(out_elems, 16) * 4));
  CK(e->rs_times.reserve((size_t)t_entries * 8));
  CK(e->rs_clips.reserve(rc.size() * sizeof(ResampleClip)));
  CK(e->rs_host.reserve(rc.size() * sizeof(ResampleClip)));
  memcpy(e->rs_host.p, rc.data(), rc.size() * sizeof(ResampleClip));
  CK(cudaMemcpyAsync(e->rs_clips.p, e->rs_host.p, rc.size() * sizeof(ResampleClip), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < n_clips; ++i)
    if (rc[i].n_in > 0)
      CK(cudaMemcpyAsync(e->rs_raw.as<char>() + (size_t)rc[i].in_off * esz, pcm[i], (size_t)rc[i].n_in * esz, cudaMemcpyHostToDevice, st));
  e->launches += 2;
  launch_resample(st, e->rs_raw.p, fmt == NISQA_FMT_F32, e->rs_clips.as<ResampleClip>(), n_clips, max_fix, e->rs_times.as<double>(),
                  e->rs_win.as<double>(), e->rs_nwin, e->rs_num_table, e->rs_out.as<float>());
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));
  return 0;
}

int nisqa_resample_device(nisqa_engine* e, const void* x, int64_t n, int sample_fmt, int32_t sr_orig, int32_t sr_new,
                          float* y, int64_t cap) {
  if (!e || !x || !y) return NISQA_ERR_INVALID;
  std::vector<int64_t> offs, n_fix;
  const void* ptrs[1] = {x};
  int rc = resample_to_device(e, 1, ptrs, &n, &sr_orig, sample_fmt, sr_new, &offs, &n_fix);
  if (rc) return rc;
  if (n_fix[0] > cap) return fail(e, NISQA_ERR_INVALID, "resample: output buffer too small");
  CK(cudaMemcpy(y, e->rs_out.as<float>() + offs[0], (size_t)n_fix[0] * 4, cudaMemcpyDeviceToHost));
  return (int)n_fix[0];
}

int nisqa_predict_pcm_resampled(nisqa_engine* e, int n_clips, const void* const* pcm, const int64_t* n_samples,
                                const int32_t* sample_rate, int sample_fmt, int32_t target_sr,
                                float* scores_out, int32_t* n_segments_out, int32_t* status_out) {
  if (!e) return NISQA_ERR_INVALID;
  if (n_clips > 0 && (!pcm || !n_samples || !sample_rate || !scores_out)) return fail(e, NISQA_ERR_INVALID, "null argument");
  std::vector<int64_t> offs, n_fix;
  int rc = resample_to_device(e, n_clips, pcm, n_samples, sample_rate, sample_fmt, target_sr, &offs, &n_fix);
  if (rc) return rc;
  std::vector<int32_t> srs(n_clips, target_sr);
  // the converted clips are ordinary float32 PCM resident in HBM: the device entry of the predict path takes over
  return predict_common(e, n_clips, nullptr, e->rs_out.p, offs.data(), n_fix.data(), srs.data(), NISQA_FMT_F32,
                        scores_out, nullptr, n_segments_out, status_out, 1);
}

int64_t nisqa_stage_dump(nisqa_engine* e, int stage, float* out, int64_t cap) {
  if (!e) return NISQA_ERR_INVALID;
  if (e->last_passes != 1) return fail(e, NISQA_ERR_STATE, "stage dump needs a predict call that ran in one pass");
  cudaSetDevice(e->device);
  Lane& LN = e->lanes[e->last_lane];
  Stage& SG = e->stages[e->last_stage];
  const int std_mode = e->cfg.arch == NISQA_ARCH_STD_LSTM_LASTBI;
  const int W1 = std_mode ? 8 : 7, W2 = std_mode ? 4 : 5, W3 = std_mode ? 2 : 3;
  const int64_t ns = e->last_n_seg;
  if (e->cfg.cnn_kind != NISQA_CNN_CONV && stage >= NISQA_STAGE_POOL1 && stage <= NISQA_STAGE_CNN_FEAT)
    return fail(e, NISQA_ERR_INVALID, "stage not available: this checkpoint has no convolutional framewise model");
  int64_t count = 0;
  const float* src = nullptr;
  int hw = 0, ch = 0;    // NHWC -> NCHW conversion when ch > 0
  int plane_layer = 0;   // the stage lives in the plane pair feeding this conv layer
  switch (stage) {
    case NISQA_STAGE_MEL_DB: count = (int64_t)e->last_n_frames * kMels; break;
    case NISQA_STAGE_POOL1: plane_layer = 2; hw = 24 * W1; ch = 16; break;
    case NISQA_STAGE_POOL2: plane_layer = 3; hw = 12 * W2; ch = 32; break;
    case NISQA_STAGE_CONV3: plane_layer = 4; hw = 12 * W2; ch = 64; break;
    case NISQA_STAGE_POOL3: plane_layer = 5; hw = 6 * W3; ch = 64; break;
    case NISQA_STAGE_CONV5: plane_layer = 6; hw = 6 * W3; ch = 64; break;
    case NISQA_STAGE_CNN_FEAT:
      if (std_mode) { src = LN.feats20.as<float>(); count = ns * 20; }
      else { src = LN.feats.as<float>(); hw = 6; ch = 64; }     // [h][c] -> c*6+h
      break;
    case NISQA_STAGE_TD_IN:
      if (std_mode || !e->last_td_in) return fail(e, NISQA_ERR_INVALID, "stage not available for this architecture");
      src = e->last_td_in; count = ns * 64; break;
    case NISQA_STAGE_TD_OUT:
      if (!e->last_td_out) return fail(e, NISQA_ERR_STATE, "the per-step BiLSTM outputs were not kept: nisqa_set_option(\"keep_td_out\", 1) before the predict call");
      src = e->last_td_out; count = ns * (std_mode ? 256 : 64); break;
    default: return fail(e, NISQA_ERR_INVALID, "unknown stage");
  }
  if (ch > 0) count = ns * hw * ch;
  if (!out) return count;
  if (stage == NISQA_STAGE_POOL1 && !e->last_pool1)
    return fail(e, NISQA_ERR_STATE, "pool1 was not kept (conv12_kernel holds it in shared memory only): nisqa_set_option(\"keep_pool1\", 1) before the predict call");
  if (cap < count) return fail(e, NISQA_ERR_INVALID, "stage dump buffer too small");
  if (count == 0) return 0;
  cudaStream_t st = LN.stream;
  if (stage == NISQA_STAGE_MEL_DB) {
    CK(e->dump.reserve((size_t)count * 4));
    launch_mel_dump(st, LN.mel.as<float>(), SG.clips.as<ClipDesc>(), (int)e->last_clips.size(),
                    SG.clipmax.as<unsigned>(), e->dump.as<float>());
    src = e->dump.as<float>();
  } else if (ch > 0) {
    if (plane_layer) {
      CK(e->dump_nhwc.reserve((size_t)count * 4));
      launch_unsplit(st, std_mode, plane_layer, LN.planes[plane_layer].as<char>(),
                     LN.planes[plane_layer].as<char>() + LN.plane_bytes[plane_layer], e->dump_nhwc.as<float>(), (int)ns);
      src = e->dump_nhwc.as<float>();
    }
    CK(e->dump.reserve((size_t)count * 4));
    launch_nhwc_to_nchw(st, src, e->dump.as<float>(), ns, hw, ch);
    src = e->dump.as<float>();
  }
  if (!src) return fail(e, NISQA_ERR_STATE, "stage was not produced");
  CK(cudaMemcpyAsync(out, src, (size_t)count * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return count;
}

int nisqa_segment_counts(const nisqa_config* cfg, int64_t n_samples, int32_t sample_rate,
                         int32_t* n_frames, int32_t* n_segments, int32_t* status) {
  if (!cfg) return NISQA_ERR_INVALID;
  ClipPlan p;
  plan_clip(*cfg, n_samples, sample_rate, &p);
  if (n_frames) *n_frames = p.n_frames;
  if (n_segments) *n_segments = p.n_seg;
  if (status) *status = p.status;
  return 0;
}

int nisqa_mel_filterbank(nisqa_engine* e, int32_t sample_rate, float* out, int64_t cap) {
  if (!e || !out) return NISQA_ERR_INVALID;
  if (!e->stream) return fail(e, NISQA_ERR_STATE, "engine was not created successfully");
  CK(cudaSetDevice(e->device));
  const int hop = (int)((double)sample_rate * e->cfg.hop_s), win = (int)((double)sample_rate * e->cfg.win_s);
  if (hop < 1 || win < 1 || win > e->cfg.n_fft) return fail(e, NISQA_ERR_INVALID, "unsupported sample rate");
  int id = -1;
  int rc = build_fb(e, sample_rate, hop, win, &id);
  if (rc) return rc;
  const std::vector<float>& d = e->fbs[id]->dense;
  if (cap < (int64_t)d.size()) return fail(e, NISQA_ERR_INVALID, "buffer too small");
  memcpy(out, d.data(), d.size() * 4);
  return 0;
}

int64_t nisqa_kernel_launches(const nisqa_engine* e) { return e ? e->launches : 0; }
void* nisqa_stream(const nisqa_engine* e) { return e ? (void*)e->stream : nullptr; }

int nisqa_join(nisqa_engine* e) {
  if (!e || !e->stream) return NISQA_ERR_INVALID;
  CK(cudaSetDevice(e->device));
  for (auto& g : e->stages)
    if (g.busy && g.lane != 0) CK(cudaStreamWaitEvent(e->stream, g.ev_done, 0));
  return 0;
}

int nisqa_set_option(nisqa_engine* e, const char* name, int value) {
  if (!e || !name) return NISQA_ERR_INVALID;
  if (strcmp(name, "fe_ppc") == 0) { e->fe_ppc = value; return 0; }
  if (strcmp(name, "keep_pool1") == 0) { e->keep_pool1 = value != 0; return 0; }
  if (strcmp(name, "keep_td_out") == 0) { e->keep_td_out = value != 0; return 0; }
  return fail(e, NISQA_ERR_INVALID, std::string("unknown option ") + name);
}

int nisqa_set_profiling(nisqa_engine* e, int on) {
  if (!e) return NISQA_ERR_INVALID;
  e->profiling = on != 0;
  return 0;
}

double nisqa_group_ms(const nisqa_engine* e, const char* group) {
  if (!e || !group) return -1.0;
  const std::string g(group);
  double total = 0.0; bool found = false;
  for (const auto& t : e->timers) {
    const bool cnn = t.name.compare(0, 4, "conv") == 0;
    const bool td = t.name == "lin_ln" || t.name == "qkv" || t.name == "sa_layer" || t.name == "fc_out" || t.name == "lstm";
    const bool match = t.name == g || (g == "cnn" && cnn) || (g == "td" && td) ||
                       (g == "frontend" && t.name == "seg_table");
    if (match) { total += t.ms; found = true; }
  }
  return found ? total : -1.0;
}

}  // extern "C"

// ------------------------------------------------------------------ NCCL (resolved at run time)
// The single exchange step of the multi-GPU path.  libnccl is bound with dlopen/dlsym so that
// the library has no link-time NCCL dependency (the torch-bundled libnccl.so.2 that is already
// in the process is reused when present).
struct NcclId { char internal[128]; };   // ncclUniqueId (passed by value to ncclCommInitRank)
namespace {
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi* nccl_api(std::string* why) {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { api.lib = dlopen(nm, RTLD_NOW | RTLD_NOLOAD); if (api.lib) break; }
    if (!api.lib) for (const char* nm : names) { api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
    if (api.lib) {
      api.GetUniqueId = (int (*)(void*))dlsym(api.lib, "ncclGetUniqueId");
      api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(api.lib, "ncclCommInitRank");
      api.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(api.lib, "ncclAllGather");
      api.CommDestroy = (int (*)(void*))dlsym(api.lib, "ncclCommDestroy");
      api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
    }
  }
  if (!api.lib || !api.GetUniqueId || !api.CommInitRank || !api.AllGather) {
    if (why) *why = "libnccl.so.2 could not be loaded (dlopen/dlsym)";
    return nullptr;
  }
  return &api;
}
}  // namespace

namespace {
int lane_allgather(nisqa_engine* e, const float* src, float* dst, size_t count, cudaStream_t st) {
  std::string why;
  NcclApi* a = nccl_api(&why);
  if (!a) return fail(e, NISQA_ERR_NCCL, why);
  int rc = a->AllGather(src, dst, count, /*ncclFloat32*/ 7, e->nccl_comm, st);
  if (rc) return fail(e, NISQA_ERR_NCCL, std::string("ncclAllGather: ") + (a->GetErrorString ? a->GetErrorString(rc) : "error"));
  e->launches += 1;
  return 0;
}
}  // namespace

extern "C" {

int nisqa_set_gather_target(nisqa_engine* e, float* global_dev, int rows) {
  if (!e || rows < 0) return NISQA_ERR_INVALID;
  e->gather_dst = global_dev; e->gather_rows = global_dev ? rows : 0;
  return 0;
}

int nisqa_nccl_unique_id(nisqa_engine* e, void* id128) {
  if (!e || !id128) return NISQA_ERR_INVALID;
  std::string why;
  NcclApi* a = nccl_api(&why);
  if (!a) return fail(e, NISQA_ERR_NCCL, why);
  int rc = a->GetUniqueId(id128);
  if (rc) return fail(e, NISQA_ERR_NCCL, std::string("ncclGetUniqueId: ") + (a->GetErrorString ? a->GetErrorString(rc) : "error"));
  return 0;
}

int nisqa_nccl_init(nisqa_engine* e, int world, int rank, const void* id128) {
  if (!e || !id128 || world < 1 || rank < 0 || rank >= world) return NISQA_ERR_INVALID;
  std::string why;
  NcclApi* a = nccl_api(&why);
  if (!a) return fail(e, NISQA_ERR_NCCL, why);
  CK(cudaSetDevice(e->device));
  NcclId id; memcpy(&id, id128, sizeof id);
  void* comm = nullptr;
  int rc = a->CommInitRank(&comm, world, id, rank);
  if (rc) return fail(e, NISQA_ERR_NCCL, std::string("ncclCommInitRank: ") + (a->GetErrorString ? a->GetErrorString(rc) : "error"));
  e->nccl_comm = comm; e->nccl_world = world; e->nccl_rank = rank;
  return 0;
}

int nisqa_gather_nccl(nisqa_engine* e, void* nccl_comm, const float* local_dev, int max_rows, float* global_dev) {
  if (!e || !local_dev || !global_dev || max_rows < 0) return NISQA_ERR_INVALID;
  std::string why;
  NcclApi* a = nccl_api(&why);
  if (!a) return fail(e, NISQA_ERR_NCCL, why);
  void* comm = nccl_comm ? nccl_comm : e->nccl_comm;
  if (!comm) return fail(e, NISQA_ERR_STATE, "no NCCL communicator: call nisqa_nccl_init or pass one");
  CK(cudaSetDevice(e->device));
  for (auto& g : e->stages)                 // the rows may have been produced on any lane
    if (g.busy && g.lane != 0) CK(cudaStreamWaitEvent(e->stream, g.ev_done, 0));
  const size_t count = (size_t)max_rows * e->cfg.n_out;
  int rc = a->AllGather(local_dev, global_dev, count, /*ncclFloat32*/ 7, comm, e->stream);
  if (rc) return fail(e, NISQA_ERR_NCCL, std::string("ncclAllGather: ") + (a->GetErrorString ? a->GetErrorString(rc) : "error"));
  e->launches += 1;
  CK(cudaStreamSynchronize(e->stream));
  return 0;
}

}  // extern "C"

#ifdef NISQA_TC_TIMING
extern "C" __attribute__((visibility("default"))) int nisqa_debug_pipe_timing(long long* host, int n, int reset) {
  return nisqa::pipe_timing_read(host, n, reset);
}
extern "C" __attribute__((visibility("default"))) int nisqa_debug_c12_timing(long long* host, int n, int reset) {
  return nisqa::c12_timing_read(host, n, reset);
}
#endif
