// engine.cu -- host runtime + C-ABI (include/sigdigger_b200.h) of the B200 analyzer engine.
//
// One engine = one channel plan applied to a batch of S independent IQ streams on one GPU.
// feed(): main PSD over every psd_size frame (four-step FFT, two kernels), channeliser forward FFT
// over half-overlapping windows with a compacting bin scatter, per-channel IFFT + cross-fade, and
// the inspector chains.  Everything is queued on one CUDA stream; results are read back on demand.
//
// This file replaces, for the hot path only, suscan's analyzer object as the reference drives it:
// suscan_analyzer_new/destroy (Suscan/Analyzer.cpp:608,636), open/set_inspector_config
// (Suscan/Analyzer.cpp:459-495), and the PSD / SAMPLES payloads (Suscan/Messages/PSDMessage.cpp:26-39,
// include/Suscan/Messages/SamplesMessage.h:33-59).  No CPU fallback exists: without a device the
// constructor fails with an error string.
#include "../../include/sigdigger_b200.h"
#include "sdb_internal.h"
#include "host_design.h"

#include <algorithm>
#include <map>
#include <string>
#include <vector>
#include <cstdio>
#include <cstring>

static thread_local std::string g_err;
static int fail(const std::string &m) { g_err = m; return -1; }
#define CK(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { \
  g_err = std::string(#expr) + ": " + cudaGetErrorString(e__); return -1; } } while (0)
#define CKP(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { \
  g_err = std::string(#expr) + ": " + cudaGetErrorString(e__); return nullptr; } } while (0)

extern "C" const char *sdb_last_error(void) { return g_err.c_str(); }
int sdb_set_error(const char *m) { g_err = m ? m : ""; return -1; }     // other units of the library (tv_kernels.cu)

extern "C" int sdb_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

static bool is_pow2(unsigned v) { return v && !(v & (v - 1)); }
static int ilog2u(unsigned v) { int l = 0; while ((1u << l) < v) ++l; return l; }

struct Channel {
  sdb_channel_params p;
  unsigned center, size, width, halfw, halfsz;
  bool has_insp;
  sdb_inspector_config cfg;
  int spect_kind = 0; unsigned spect_size = 0, est_mask = 0;   // SPEC U
};

struct TimedSpan { int family; cudaEvent_t a, b; };
enum { FAM_COLS = 0, FAM_ROWS_PSD, FAM_ROWS_CHAN, FAM_CHAN_IFFT, FAM_INSPECTOR, FAM_COUNT };
static const char *kFamNames[FAM_COUNT] = { "fft_cols", "fft_rows_psd", "fft_rows_chan", "chan_ifft",
                                            "inspector" };

struct sdb_engine {
  sdb_engine_params prm;
  double samp_rate;
  cudaStream_t stream = nullptr;
  uint64_t launches = 0;
  bool committed = false, first_feed = true, timing = false, chains_fresh = true;
  std::vector<Channel> channels;
  std::map<unsigned, float2 *> tw;     // twiddle tables by size
  std::vector<void *> allocs;

  unsigned Np = 0, W = 0;               // PSD size, channeliser window
  SdbFourStep fs_psd{}, fs_st{};
  bool psd_small = false;
  float *d_window = nullptr;
  float2 *d_scratch = nullptr; int chunk_windows = 1; size_t l2_pinned_bytes = 0; int sm_count = 0;
  // The PSD transforms run on their own stream, concurrently with the channeliser transforms of the same
  // group of streams (feed_device): the two kernel chains fill each other's launch gaps and partial waves,
  // and both read the same input region while it is still in L2.
  cudaStream_t psd_stream = nullptr; cudaEvent_t ev_feed = nullptr;
  float2 *d_xin = nullptr;              // staging for host feeds
  float2 *d_hist = nullptr;             // [S][W/2]
  float *d_psd = nullptr; size_t max_frames = 0, last_frames = 0;
  // channeliser
  int *d_binmap = nullptr; int n_bins = 0; unsigned ka_mask = 0;
  float2 *d_cspec = nullptr; size_t max_hops = 0;
  std::vector<SdbChannelDev> h_chans; SdbChannelDev *d_chans = nullptr;
  struct Group { int size; int len; int *d_ids; int any_precise; };
  std::vector<Group> groups;
  float2 *d_tails = nullptr; size_t tail_stride = 0;
  float *d_lo_phase = nullptr;
  // channel streams are double-buffered: the (latency-bound, 1-CTA-per-32-chains) inspector kernel of feed i
  // runs on its own stream while the FFT kernels of feed i+1 fill the other buffer
  float2 *d_chanb[2] = { nullptr, nullptr }; size_t chan_stride = 0;
  cudaStream_t insp_stream = nullptr;
  cudaEvent_t ev_chan[2] = { nullptr, nullptr }, ev_insp[2] = { nullptr, nullptr };
  bool ev_insp_valid[2] = { false, false };
  unsigned feed_index = 0; int last_buf = 0;
  uint64_t n_fed = 0; std::vector<float2> last_x_tail;
  // DC removal (SDB_FLAG_DC_REMOVE, SPEC R): per-stream estimate, the estimate the current block is corrected with,
  // run sums, and the corrected float32 copy of the block the rest of the path reads
  float2 *d_dc_state = nullptr, *d_dc_cur = nullptr, *d_xdc = nullptr; double2 *d_dc_part = nullptr;   // samples fed so far; (engines without channels keep no history)
  // Host-buffer pipeline: results and input staging are double-buffered by feed parity so that the H2D
  // copy of feed i+1 and the D2H reads of feed i-1 overlap the kernels of feed i (three copy/compute
  // streams).  d_psd / d_soft / d_hard / d_counts always point at the buffers of the latest feed.
  float *d_psdb[2] = { nullptr, nullptr };
  float2 *d_softb[2] = { nullptr, nullptr }; uint8_t *d_hardb[2] = { nullptr, nullptr };
  uint32_t *d_countsb[2] = { nullptr, nullptr };
  unsigned long long *d_sym_off[2] = { nullptr, nullptr };   // packed read-out: start of every chain, 16-symbol aligned
  float2 *d_xinb[2] = { nullptr, nullptr };
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  cudaEvent_t ev_psd_ready[2] = { nullptr, nullptr }, ev_psd_read[2] = { nullptr, nullptr },
              ev_sym_read[2] = { nullptr, nullptr }, ev_h2d[2] = { nullptr, nullptr }, ev_xfree[2] = { nullptr, nullptr };
  bool psd_read_valid[2] = { false, false }, sym_read_valid[2] = { false, false }, xfree_valid[2] = { false, false };
  unsigned host_feeds = 0;
  size_t last_hops = 0;
  // chains
  SdbChainCfg *d_cfg = nullptr; std::vector<SdbChainCfg> h_cfg;
  SdbChainState *d_state = nullptr;
  float *d_pool = nullptr; size_t pool_stride = 0;
  int *d_chain_map = nullptr; int insp_ctas = 0; std::vector<int> h_chain_map;
  float *d_taps = nullptr;
  float2 *d_soft = nullptr; uint8_t *d_hard = nullptr; uint32_t *d_counts = nullptr; size_t sym_cap = 0;
  // channel detector on the main PSD (SPEC K; chdet_kernels.cu)
  struct sdb_chdet *chdet = nullptr; bool cd_enabled = false;
  float cd_alpha = 0, cd_gamma = 0, cd_snr = 0; unsigned cd_min_bins = 1;
  // inspector spectrum sources / estimators (SPEC U)
  std::map<unsigned, float *> bh_windows;
  std::vector<SdbSpectCfg> h_spect; SdbSpectCfg *d_spectcfg = nullptr;
  float *d_spect = nullptr; size_t spect_stride = 0; int spect_max_ns = 0;
  uint32_t *d_spect_size = nullptr; float *d_est = nullptr; int *d_est_valid = nullptr;
  // timing
  std::vector<TimedSpan> spans;
  double fam_ms[FAM_COUNT] = {0}; uint64_t fam_n[FAM_COUNT] = {0};

  template <typename T> T *dalloc(size_t n)
  {
    void *p = nullptr;
    if (n == 0) n = 1;
    if (cudaMalloc(&p, n * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    allocs.push_back(p);
    return (T *) p;
  }
  const float2 *twiddle(unsigned n)
  {
    auto it = tw.find(n);
    if (it != tw.end()) return it->second;
    std::vector<float2> h;
    sdbh::twiddle_fill(n, h);
    float2 *d = dalloc<float2>(n);
    if (!d) return nullptr;
    cudaMemcpy(d, h.data(), n * sizeof(float2), cudaMemcpyHostToDevice);
    tw[n] = d;
    return d;
  }
  void span_begin(int fam, cudaStream_t on = nullptr)
  {
    if (!timing) return;
    TimedSpan s; s.family = fam;
    cudaEventCreate(&s.a); cudaEventCreate(&s.b);
    cudaEventRecord(s.a, on ? on : stream);
    spans.push_back(s);
  }
  void span_end(cudaStream_t on = nullptr)
  {
    if (!timing) return;
    cudaEventRecord(spans.back().b, on ? on : stream);
  }
  // make the main stream wait for everything queued on the inspector stream
  cudaError_t join()
  {
    if (!insp_stream) return cudaSuccess;
    const int b = last_buf;
    if (ev_insp_valid[b]) return cudaStreamWaitEvent(stream, ev_insp[b], 0);
    return cudaSuccess;
  }
  void collect_spans()
  {
    for (auto &s : spans) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) { fam_ms[s.family] += ms; fam_n[s.family]++; }
      cudaEventDestroy(s.a); cudaEventDestroy(s.b);
    }
    spans.clear();
  }
};

static bool make_four_step(sdb_engine *e, unsigned N, SdbFourStep *fs)
{
  int l = ilog2u(N), l1 = l / 2;
  if (N == 32768 || N == 16384 || N == 8192) l1 = l - 8;        // SPEC F.5: N1 x 256 on the register-butterfly passes
  fs->N = (int) N; fs->N1 = 1 << l1; fs->N2 = (int) N / fs->N1;
  fs->twN1 = e->twiddle(fs->N1); fs->twN2 = e->twiddle(fs->N2); fs->twN = e->twiddle(N);
  fs->twPQ = nullptr;
  if (!(fs->twN1 && fs->twN2 && fs->twN)) return false;
  if (N == 65536) {
    // the product the kernels used to form per output (two table look-ups + one complex multiply), tabulated
    // once with the same arithmetic (SPEC F.1: one rounded product + one fused multiply-add per component)
    auto it = e->tw.find(0x10000u | 1u);
    if (it != e->tw.end()) { fs->twPQ = it->second; return true; }
    std::vector<float2> c, f, pq((size_t) 65536);
    sdbh::twiddle_fill(256, c); sdbh::twiddle_fill(65536, f);
    for (unsigned k1 = 0; k1 < 256; ++k1)
      for (unsigned n2 = 0; n2 < 256; ++n2) {
        const unsigned p = n2 * k1;
        const float2 a = c[p >> 8], b = f[p & 255];
        pq[(size_t) k1 * 256 + n2].x = fmaf(a.x, b.x, -(a.y * b.y));
        pq[(size_t) k1 * 256 + n2].y = fmaf(a.x, b.y, a.y * b.x);
      }
    float2 *d = e->dalloc<float2>(65536);
    if (!d) return false;
    cudaMemcpy(d, pq.data(), 65536 * sizeof(float2), cudaMemcpyHostToDevice);
    e->tw[0x10000u | 1u] = d;
    fs->twPQ = d;
  }
  if (N == 32768 || N == 16384 || N == 8192) {
    // SPEC F.5: N1 x 256, inter-pass twiddle [k1][n2] = W_N1^(p >> 8) x W_N^(p & 255), p = n2 k1
    const unsigned N1 = N / 256;
    auto it = e->tw.find(N | 1u);
    if (it != e->tw.end()) { fs->twPQ = it->second; return true; }
    std::vector<float2> c, f, pq((size_t) N);
    sdbh::twiddle_fill(N1, c); sdbh::twiddle_fill(N, f);
    for (unsigned k1 = 0; k1 < N1; ++k1)
      for (unsigned n2 = 0; n2 < 256; ++n2) {
        const unsigned p = n2 * k1;
        const float2 a = c[p >> 8], b = f[p & 255];
        pq[(size_t) k1 * 256 + n2].x = fmaf(a.x, b.x, -(a.y * b.y));
        pq[(size_t) k1 * 256 + n2].y = fmaf(a.x, b.y, a.y * b.x);
      }
    float2 *d = e->dalloc<float2>(N);
    if (!d) return false;
    cudaMemcpy(d, pq.data(), (size_t) N * sizeof(float2), cudaMemcpyHostToDevice);
    e->tw[N | 1u] = d;
    fs->twPQ = d;
  }
  return true;
}

extern "C" sdb_engine_t *sdb_engine_new(const sdb_engine_params *p, double samp_rate)
{
  if (!p) { g_err = "null params"; return nullptr; }
  if (sdb_device_count() <= 0) { g_err = "no CUDA device: sigdigger_b200 has no CPU fallback"; return nullptr; }
  if (p->n_streams < 1) { g_err = "n_streams must be >= 1"; return nullptr; }
  if (p->psd_size && (!is_pow2(p->psd_size) || p->psd_size < 16 || p->psd_size > (1u << 20))) {
    g_err = "psd_size must be a power of two in [16, 2^20]"; return nullptr;
  }
  unsigned W = p->st_window_size ? p->st_window_size : p->psd_size;
  if (!is_pow2(W) || W < 64 || W > (1u << 20)) { g_err = "st_window_size must be a power of two in [64, 2^20]"; return nullptr; }
  if (p->input_format < SDB_FORMAT_FLOAT32 || p->input_format > SDB_FORMAT_SIGNED16) {
    g_err = "unknown input_format"; return nullptr;
  }
  CKP(cudaSetDevice(p->device));
  sdb_engine *e = new sdb_engine();
  e->prm = *p; e->samp_rate = samp_rate; e->Np = p->psd_size; e->W = W;
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_err = "cudaStreamCreate failed"; delete e; return nullptr;
  }
  return e;
}

extern "C" void sdb_engine_destroy(sdb_engine_t *e)
{
  if (!e) return;
  cudaSetDevice(e->prm.device);
  cudaStreamSynchronize(e->stream);
  if (e->insp_stream) cudaStreamSynchronize(e->insp_stream);
  e->collect_spans();
  if (e->l2_pinned_bytes) { cudaCtxResetPersistingL2Cache(); cudaGetLastError(); }
  if (e->chdet) sdb_chdet_destroy(e->chdet);
  for (void *p : e->allocs) cudaFree(p);
  for (int i = 0; i < 2; ++i) {
    if (e->ev_chan[i]) cudaEventDestroy(e->ev_chan[i]);
    if (e->ev_insp[i]) cudaEventDestroy(e->ev_insp[i]);
  }
  if (e->insp_stream) cudaStreamDestroy(e->insp_stream);
  if (e->psd_stream) { cudaStreamSynchronize(e->psd_stream); cudaStreamDestroy(e->psd_stream); }
  if (e->ev_feed) cudaEventDestroy(e->ev_feed);
  if (e->h2d_stream) { cudaStreamSynchronize(e->h2d_stream); cudaStreamDestroy(e->h2d_stream); }
  if (e->d2h_stream) { cudaStreamSynchronize(e->d2h_stream); cudaStreamDestroy(e->d2h_stream); }
  for (int i = 0; i < 2; ++i)
    for (cudaEvent_t ev : { e->ev_psd_ready[i], e->ev_psd_read[i], e->ev_sym_read[i], e->ev_h2d[i], e->ev_xfree[i] })
      if (ev) cudaEventDestroy(ev);
  cudaStreamDestroy(e->stream);
  delete e;
}

extern "C" int sdb_inspector_config_default(sdb_inspector_config *c, int insp_class, float fs)
{
  if (!c) return fail("null config");
  memset(c, 0, sizeof(*c));
  c->insp_class = insp_class; c->fs = fs;
  c->agc_enabled = 1; c->agc_gain_db = 0.0f;
  c->costas_order = insp_class == SDB_INSP_PSK ? 2 : 0;
  c->bits_per_symbol = insp_class == SDB_INSP_PSK ? 2 : 1;
  c->loop_bw = fs * 1e-3f; c->offset = 0.0f;
  c->mf_type = 0; c->mf_rolloff = 0.35f;
  c->clock_type = 1; c->baud = fs * 0.25f; c->clock_gain = 1.0f; c->clock_phase = 0.0f; c->clock_running = 1;
  c->audio_cutoff = 5000.0f; c->audio_volume = 1.0f; c->audio_sample_rate = 44100;
  c->audio_demod = SDB_AUDIO_FM; c->agc_ts = 0.1f;
  c->eq_type = 0; c->eq_rate = 1e-3f; c->eq_locked = 0;
  return 0;
}

extern "C" int sdb_engine_open_channel(sdb_engine_t *e, const sdb_channel_params *p, sdb_channel_info *info)
{
  if (!e || !p) return fail("null argument");
  if (e->committed) return fail("engine already committed");
  if (!(p->guard >= 1.0f) || !(p->bw > 0.0f) || p->bw > 6.28318530717958647692f * 1.0001f)
    return fail("invalid channel: guard >= 1 and 0 < bw <= 2 pi required");   // INVALID_CHANNEL
  if (!(p->f0 >= 0.0f) || p->f0 >= 6.28318530717958647692f) return fail("invalid channel: f0 must be in [0, 2 pi)");
  Channel c;
  c.p = *p; c.has_insp = false;
  sdbh::channel_geometry(e->W, p->f0, p->bw, p->guard, &c.center, &c.size, &c.width);
  c.halfw = c.width >> 1; c.halfsz = c.size >> 1;
  if (c.size > 16384) return fail("channel size > 16384 bins not supported by the shared-memory IFFT");
  memset(&c.cfg, 0, sizeof(c.cfg));
  e->channels.push_back(c);
  if (info) { info->center = c.center; info->size = c.size; info->width = c.width;
              info->decimation = (float) e->W / (float) c.size; }
  return (int) e->channels.size() - 1;
}

// channel geometry without an engine (su_specttuner_open_channel computes it before any transform exists)
extern "C" int sdb_channel_geometry(uint32_t window_size, const sdb_channel_params *p, sdb_channel_info *info)
{
  if (!p || !info) return fail("null argument");
  if (!is_pow2(window_size) || window_size < 64) return fail("window size must be a power of two >= 64");
  if (!(p->guard >= 1.0f) || !(p->bw > 0.0f) || p->bw > 6.28318530717958647692f * 1.0001f)
    return fail("invalid channel: bw must be in (0, 2 pi], guard >= 1");
  if (!(p->f0 >= 0.0f) || p->f0 >= 6.28318530717958647692f) return fail("invalid channel: f0 must be in [0, 2 pi)");
  unsigned center, size, width;
  sdbh::channel_geometry(window_size, p->f0, p->bw, p->guard, &center, &size, &width);
  info->center = center; info->size = size; info->width = width;
  info->decimation = (float) window_size / (float) size;
  return 0;
}

extern "C" int sdb_engine_set_inspector(sdb_engine_t *e, int handle, const sdb_inspector_config *cfg)
{
  if (!e || !cfg) return fail("null argument");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");   // WRONG_HANDLE
  if (e->committed) return fail("engine already committed");
  if (cfg->insp_class < SDB_INSP_PSK || cfg->insp_class > SDB_INSP_RAW) return fail("wrong kind");
  Channel &c = e->channels[handle];
  c.cfg = *cfg; c.has_insp = true;
  c.cfg.fs = (float) (e->samp_rate * (double) c.size / (double) e->W);
  return 0;
}

struct sdb_chdet;
cudaError_t sdb_chdet_feed_stream(sdb_chdet *d, const float *psd_dev, uint32_t frames, size_t stream_stride,
                                  cudaStream_t stream, uint64_t *launch_counter);

extern "C" int sdb_engine_set_channel_detector(sdb_engine_t *e, float alpha, float beta, float gamma, float snr,
                                               uint32_t min_bins)
{
  (void) beta;
  if (!e) return fail("null argument");
  if (e->committed) return fail("engine already committed");
  if (!e->prm.psd_size) return fail("the channel detector needs the main PSD");
  if (e->prm.flags & SDB_FLAG_PSD_SHIFT_DB) return fail("the channel detector needs a linear PSD");
  if (!(snr > 0.0f) || !(alpha >= 0.0f && alpha <= 1.0f) || !(gamma >= 0.0f && gamma <= 1.0f))
    return fail("detector parameters out of range");
  e->cd_enabled = true; e->cd_alpha = alpha; e->cd_gamma = gamma; e->cd_snr = snr; e->cd_min_bins = min_bins ? min_bins : 1;
  return 0;
}

extern "C" long sdb_engine_read_channels(sdb_engine_t *e, uint32_t stream, double center_freq,
                                         sdb_detected_channel *out, size_t cap, uint32_t *total)
{
  if (!e) return fail("null argument");
  if (!e->committed || !e->chdet) return fail("channel detector not enabled");
  if (stream >= e->prm.n_streams) return fail("stream out of range");
  CK(cudaSetDevice(e->prm.device));
  CK(cudaStreamSynchronize(e->psd_stream ? e->psd_stream : e->stream));
  CK(cudaStreamSynchronize(e->stream));
  const long n = sdb_chdet_read(e->chdet, stream, e->samp_rate, center_freq, out, cap, total);
  if (n < 0) return fail("channel read failed");
  return n;
}

extern "C" int sdb_chdet_read_all(struct sdb_chdet *d, double samp_rate, const double *centers, sdb_detected_channel *out,
                                  size_t cap, uint32_t *counts);
// all streams at once: centers[S] (host), out[S][cap], counts[S]
extern "C" int sdb_engine_read_all_channels(sdb_engine_t *e, const double *centers, sdb_detected_channel *out, size_t cap,
                                            uint32_t *counts)
{
  if (!e || !centers || !out || !counts) return fail("null argument");
  if (!e->committed || !e->chdet) return fail("channel detector not enabled");
  CK(cudaSetDevice(e->prm.device));
  CK(cudaStreamSynchronize(e->psd_stream ? e->psd_stream : e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (sdb_chdet_read_all(e->chdet, e->samp_rate, centers, out, cap, counts)) return fail("channel read failed");
  return 0;
}

static const char *kSpectNames[SDB_SPECTSRC_COUNT] = { "none", "psd", "cyclo", "fmspect", "timediff", "abstimediff",
                                                      "exp_2", "exp_4", "exp_8", "fac" };
static const char *kEstNames[SDB_ESTIMATOR_COUNT] = { "baud-fac", "baud-nonlinear" };
extern "C" const char *sdb_spectsrc_name(int id) { return id >= 0 && id < SDB_SPECTSRC_COUNT ? kSpectNames[id] : nullptr; }
extern "C" const char *sdb_estimator_name(int id) { return id >= 0 && id < SDB_ESTIMATOR_COUNT ? kEstNames[id] : nullptr; }

extern "C" int sdb_engine_set_spectrum_source(sdb_engine_t *e, int handle, int spectsrc_id, uint32_t size)
{
  if (!e) return fail("null argument");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");
  if (e->committed) return fail("engine already committed");
  if (spectsrc_id < 0 || spectsrc_id >= SDB_SPECTSRC_COUNT) return fail("unknown spectrum source");
  if (!is_pow2(size) || size < 64 || size > 4096) return fail("spectrum size must be a power of two in [64, 4096]");
  Channel &c = e->channels[handle];
  if (c.spect_size && c.spect_size != size && c.est_mask) return fail("spectrum size already fixed by an estimator");
  c.spect_kind = spectsrc_id; c.spect_size = size;
  return 0;
}

extern "C" int sdb_engine_set_estimator(sdb_engine_t *e, int handle, int estimator_id, int enabled)
{
  if (!e) return fail("null argument");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");
  if (e->committed) return fail("engine already committed");
  if (estimator_id < 0 || estimator_id >= SDB_ESTIMATOR_COUNT) return fail("unknown estimator");
  Channel &c = e->channels[handle];
  if (enabled) c.est_mask |= 1u << estimator_id; else c.est_mask &= ~(1u << estimator_id);
  return 0;
}

extern "C" int sdb_engine_read_spectrum(sdb_engine_t *e, int handle, float *out, uint32_t *sizes)
{
  if (!e || !out || !sizes) return fail("null argument");
  if (!e->committed) return fail("engine not committed");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");
  if (!e->d_spect || e->h_spect[handle].kind == 0) return fail("no spectrum source on this channel");
  CK(cudaSetDevice(e->prm.device));
  CK(cudaStreamSynchronize(e->insp_stream));
  const unsigned S = e->prm.n_streams; const int K = (int) e->channels.size();
  const SdbSpectCfg &q = e->h_spect[handle];
  CK(cudaMemcpy2D(out, (size_t) q.ns * sizeof(float), e->d_spect + q.out_off, e->spect_stride * sizeof(float),
                  (size_t) q.ns * sizeof(float), S, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(sizes, sizeof(uint32_t), e->d_spect_size + handle, (size_t) K * sizeof(uint32_t), sizeof(uint32_t), S,
                  cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int sdb_engine_read_estimate(sdb_engine_t *e, int handle, int estimator_id, float *values, int32_t *valid)
{
  if (!e || !values || !valid) return fail("null argument");
  if (!e->committed) return fail("engine not committed");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");
  if (estimator_id < 0 || estimator_id >= SDB_ESTIMATOR_COUNT) return fail("unknown estimator");
  if (!e->d_est || !(e->h_spect[handle].est_mask & (1u << estimator_id))) return fail("estimator not enabled on this channel");
  CK(cudaSetDevice(e->prm.device));
  CK(cudaStreamSynchronize(e->insp_stream));
  const unsigned S = e->prm.n_streams; const int K = (int) e->channels.size();
  const size_t pitch = (size_t) K * 2 * sizeof(float), off = (size_t) handle * 2 + estimator_id;
  CK(cudaMemcpy2D(values, sizeof(float), e->d_est + off, pitch, sizeof(float), S, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(valid, sizeof(int32_t), e->d_est_valid + off, pitch, sizeof(int32_t), S, cudaMemcpyDeviceToHost));
  return 0;
}

// sdb_inspector_config -> SdbChainCfg (SPEC X; same derivations as the inspector constructors)
static bool build_chain_cfg(const Channel &ch, SdbChainCfg &c, std::vector<float> &taps_pool)
{
  const sdb_inspector_config &g = ch.cfg;
  memset(&c, 0, sizeof(c));
  c.cls = ch.has_insp ? g.insp_class : SDB_INSP_RAW;
  if (c.cls == SDB_INSP_RAW) return true;
  const float fs = g.fs;
  float bnor = g.baud / fs;
  if (bnor > 1.0f) bnor = 1.0f;
  if (!(bnor > 0.0f)) bnor = 1e-6f;
  const float T = 1.0f / bnor;
  c.bnor = bnor;
  c.gain2 = 2.0f * d_db_to_mag(g.agc_gain_db);
  c.dl_size = c.mh_size = 1;

  if (c.cls == SDB_INSP_AUDIO) {
    float tau = g.agc_ts * fs;
    if (tau < 2.0f) tau = 2.0f;
    if (g.agc_enabled) {
      sdbh::AgcDesign d = sdbh::agc_from_tau(tau, 1.0f);
      c.have_agc = 1; c.knee = d.knee; c.gain_slope = d.gain_slope; c.fixed_gain = d.fixed_gain;
      c.hang_max = d.hang_max; c.dl_size = d.dl_size; c.mh_size = d.mh_size;
      c.far_ = d.far_; c.faf = d.faf; c.sar = d.sar; c.saf = d.saf;
    }
    if (sdbh::butter_lp(4, sdbh::clampf(2.0f * g.audio_cutoff / fs, 1e-4f, 0.95f), c.alpf_b, c.alpf_a))
      c.alpf_n = 5;
    c.audio_demod = (int) g.audio_demod; c.audio_squelch = g.audio_squelch;
    c.audio_volume = g.audio_volume;
    c.dc_alpha = (float) (1.0 - exp(-1.0 / (0.05 * (double) fs)));
    c.sq_alpha = (float) (1.0 - exp(-1.0 / (0.01 * (double) fs)));
    c.sq_thr = g.audio_squelch_level;
    c.rs_step = (double) g.audio_sample_rate / (double) fs;
    float fo = g.audio_demod == SDB_AUDIO_USB ? g.offset : -g.offset;
    c.lo_omega = 3.14159265358979323846f * (2.0f * fo / fs);
    return true;
  }

  if (g.agc_enabled) {
    sdbh::AgcDesign d = sdbh::agc_from_tau(T, 1.0f);
    c.have_agc = 1; c.knee = d.knee; c.gain_slope = d.gain_slope; c.fixed_gain = d.fixed_gain;
    c.hang_max = d.hang_max; c.dl_size = d.dl_size; c.mh_size = d.mh_size;
    c.far_ = d.far_; c.faf = d.faf; c.sar = d.sar; c.saf = d.saf;
  }
  c.af_n = 1; c.af_b[0] = 1.0f; c.af_a[0] = 1.0f;
  switch (c.cls) {
    case SDB_INSP_PSK:
      if (g.costas_order > 0) {
        if (g.costas_order > 3) return false;
        c.have_costas = 1; c.costas_kind = (int) g.costas_order;
        float loop = 2.0f * g.loop_bw / fs;
        c.c_a = 3.14159265358979323846f * loop;
        c.c_b = 0.5f * c.c_a * c.c_a;
        // arm filter "order 3" = 2-pole Butterworth (Tasks/CostasRecoveryTask.cpp:41)
        if (!sdbh::butter_lp(2, sdbh::clampf(2.0f * bnor, 1e-3f, 0.95f), c.af_b, c.af_a)) return false;
        c.af_n = 3;
      } else {
        c.have_lo = 1;
        c.lo_omega = 3.14159265358979323846f * (2.0f * g.offset / fs);
      }
      break;
    case SDB_INSP_FSK: {
      float s, co;
      d_sincosf(g.fsk_phase, &s, &co);
      c.fsk_rot_re = co; c.fsk_rot_im = s;
      c.fsk_quad_demod = g.fsk_quad_demod;
      break;
    }
    case SDB_INSP_ASK:
      if (g.ask_use_pll) {
        float fc = 3.14159265358979323846f * (2.0f * g.loop_bw / fs);
        float dinv = 1.0f / (1.0f + 2.0f * 0.707f * fc + fc * fc);
        c.have_pll = 1;
        c.pll_alpha = 4.0f * fc * fc * dinv;
        c.pll_beta = 4.0f * 0.707f * fc * dinv;
      } else {
        c.have_lo = 1;
        c.lo_omega = 3.14159265358979323846f * (2.0f * g.offset / fs);
      }
      c.ask_channel = (int) g.ask_channel;
      break;
    default:
      return false;
  }
  if (g.mf_type == 1) {
    std::vector<float> h;
    unsigned n = sdbh::mf_span(T);
    sdbh::taps_rrc(h, n, T, g.mf_rolloff);
    c.have_mf = 1; c.mf_n = (int) n; c.mf_off = (int) taps_pool.size();
    taps_pool.insert(taps_pool.end(), h.begin(), h.end());
  }
  c.clock_type = (int) g.clock_type; c.clock_running = g.clock_running;
  c.clk_gain = g.clock_gain; c.clk_alpha = 2e-1f; c.clk_beta = 6e-4f * c.clk_alpha;
  c.smp_period = 1.0f / bnor; c.smp_phase0 = g.clock_phase * c.smp_period;
  if (c.cls == SDB_INSP_ASK) { c.dec_mode = 1; c.dec_min = 0.0f; c.dec_h = 1.0f - 0.0f; }
  else { c.dec_mode = 0; c.dec_min = -3.14159265358979323846f;
         c.dec_h = 3.14159265358979323846f - (-3.14159265358979323846f); }
  c.dec_intervals = 1 << g.bits_per_symbol;
  c.eq_type = (int) g.eq_type; c.eq_locked = g.eq_locked; c.eq_mu = g.eq_rate;
  if (g.eq_type > 1) return false;
  return true;
}

extern "C" int sdb_engine_commit(sdb_engine_t *e)
{
  if (!e) return fail("null engine");
  if (e->committed) return fail("already committed");
  CK(cudaSetDevice(e->prm.device));
  const unsigned S = e->prm.n_streams, W = e->W, Np = e->Np;
  const int K = (int) e->channels.size();
  size_t max_feed = e->prm.max_feed;
  if (max_feed == 0) return fail("max_feed must be > 0");
  if (max_feed % (W / 2)) return fail("max_feed must be a multiple of st_window_size / 2");
  if (Np && max_feed % Np) return fail("max_feed must be a multiple of psd_size");

  // ---- PSD plan
  if (Np) {
    std::vector<float> w;
    if (e->prm.psd_window != SDB_WINDOW_NONE) {
      sdbh::window_fill(w, Np, e->prm.psd_window);
      e->d_window = e->dalloc<float>(Np);
      if (!e->d_window) return fail("out of device memory");
      CK(cudaMemcpy(e->d_window, w.data(), Np * sizeof(float), cudaMemcpyHostToDevice));
    }
    e->psd_small = Np <= 4096;
    if (e->psd_small) { if (!e->twiddle(Np)) return fail("out of device memory"); }
    else if (!make_four_step(e, Np, &e->fs_psd)) return fail("out of device memory");
    e->max_frames = max_feed / Np;
    for (int i = 0; i < 2; ++i) {
      e->d_psdb[i] = e->dalloc<float>((size_t) S * e->max_frames * Np);
      if (!e->d_psdb[i]) return fail("out of device memory (psd)");
    }
    e->d_psd = e->d_psdb[0];
    if (e->cd_enabled) {
      e->chdet = sdb_chdet_new(e->prm.device, Np, S, e->cd_alpha, e->cd_gamma, e->cd_snr, e->cd_min_bins);
      if (!e->chdet) return fail("out of device memory (channel detector)");
    }
  }
  // ---- four-step scratch: one window per SM, pinned in L2
  {
    unsigned big = std::max(Np > 4096 ? Np : 0u, K > 0 ? W : 0u);
    if (big) {
      size_t scratch_mb = 64;
      if (const char *env = getenv("SDB_SCRATCH_MB")) { long v = atol(env); if (v >= 1 && v <= 4096) scratch_mb = (size_t) v; }
      size_t cw = (scratch_mb << 20) / ((size_t) big * sizeof(float2));
      if (cw < 1) cw = 1;
      if ((big == 65536 || big == 32768 || big == 16384 || big == 8192) && !getenv("SDB_SCRATCH_MB")) {
        // 65536 path: 16 (pass A, 4 CTAs/SM) and 8 (pass B, 2 CTAs/SM) CTAs per window, all of equal duration:
        // one window per SM is exactly 4 waves of either kernel.  148 SMs -> 148 windows -> 77.6 MB, inside
        // the 82.9 MB of L2 that can be set aside for persisting lines on B200.
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->prm.device) == cudaSuccess && sms > 0 &&
            (size_t) sms * 65536 * sizeof(float2) <= (100u << 20))
          cw = (size_t) sms * (65536 / big);          // the same 77.6 MB: two 32768-point windows per SM, ...
        e->sm_count = sms;
      }
      if (const char *env = getenv("SDB_CHUNK_WINDOWS")) { long v = atol(env); if (v >= 1 && v <= 65536) cw = (size_t) v; }
      e->chunk_windows = (int) cw;
      e->d_scratch = e->dalloc<float2>((size_t) e->chunk_windows * big);
      if (!e->d_scratch) return fail("out of device memory (scratch)");
      if (Np > 4096 && K > 0 && Np == W && !getenv("SDB_NO_PSD_STREAM")) {
        CK(cudaStreamCreateWithFlags(&e->psd_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&e->ev_feed, cudaEventDisableTiming));
      }
      // Pin the scratch in L2.  Without this the streamed input and output evict it between the two passes
      // and every window costs two extra HBM round trips (ncu: 266 MB of DRAM traffic per 148-window chunk
      // against 116 MB algorithmic, profiles/r01_l2.md).  Accesses of the transform streams inside the window
      // are "persisting" (a set-aside part of L2 that normal traffic cannot evict); the kernels additionally
      // mark their one-shot outputs as streaming (st.global.cs).
      if ((big == 65536 || big == 32768 || big == 16384 || big == 8192) && !getenv("SDB_NO_L2_PIN")) {   // the set-aside is device-wide: only the big plans claim it
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, e->prm.device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, e->prm.device);
        const size_t bytes = (size_t) e->chunk_windows * big * sizeof(float2);
        if (max_persist > 0 && max_window > 0) {
          const size_t set_aside = std::min(bytes, (size_t) max_persist);
          if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside) == cudaSuccess) {
            cudaStreamAttrValue av{};
            av.accessPolicyWindow.base_ptr = e->d_scratch;
            av.accessPolicyWindow.num_bytes = std::min(bytes, (size_t) max_window);
            av.accessPolicyWindow.hitRatio = (float) std::min(1.0, (double) set_aside / (double) av.accessPolicyWindow.num_bytes);
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            if (cudaStreamSetAttribute(e->stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess)
              e->l2_pinned_bytes = set_aside;
            if (e->psd_stream) cudaStreamSetAttribute(e->psd_stream, cudaStreamAttributeAccessPolicyWindow, &av);
          }
          cudaGetLastError();   // the pin is an optimisation: never fail the commit because of it
        }
      }
    }
  }
  // ---- channeliser plan
  e->max_hops = max_feed / (W / 2);
  if (K > 0) {
    if (!make_four_step(e, W, &e->fs_st)) return fail("out of device memory");
    std::vector<int> binmap(W, -1);
    std::vector<char> need(W, 0);
    for (auto &c : e->channels)
      for (unsigned i = 0; i < 2 * c.halfw; ++i) need[(c.center + W - c.halfw + i) % W] = 1;
    int nb = 0;
    e->ka_mask = 0;
    // bin k = k1 + N1 (ka + 16 kb): N1 = 256 (F.4) or W / 256 (F.5); the generic passes ignore the mask
    const unsigned ka_shift = W == 32768 ? 7u : (W == 16384 ? 6u : (W == 8192 ? 5u : 8u));
    for (unsigned b = 0; b < W; ++b) if (need[b]) { binmap[b] = nb++; e->ka_mask |= 1u << ((b >> ka_shift) & 15u); }
    e->n_bins = nb;
    e->d_binmap = e->dalloc<int>(W);
    if (!e->d_binmap) return fail("out of device memory");
    CK(cudaMemcpy(e->d_binmap, binmap.data(), W * sizeof(int), cudaMemcpyHostToDevice));
    e->d_cspec = e->dalloc<float2>((size_t) S * e->max_hops * nb);
    e->d_hist = e->dalloc<float2>((size_t) S * (W / 2));
    if (!e->d_cspec || !e->d_hist) return fail("out of device memory (cspec)");
    CK(cudaMemset(e->d_hist, 0, (size_t) S * (W / 2) * sizeof(float2)));

    e->h_chans.resize(K);
    size_t out_off = 0, tail_off = 0;
    std::map<int, std::vector<int>> by_size;
    for (int k = 0; k < K; ++k) {
      Channel &c = e->channels[k];
      SdbChannelDev &d = e->h_chans[k];
      memset(&d, 0, sizeof(d));
      d.center = (int) c.center; d.size = (int) c.size; d.log2size = ilog2u(c.size);
      d.halfw = (int) c.halfw; d.halfsz = (int) c.halfsz;
      unsigned b0 = (c.center + W - c.halfw) % W;
      d.c1 = binmap[b0];
      d.L1 = (int) std::min<unsigned>(2 * c.halfw, W - b0);
      d.precise = c.p.precise;
      if (c.p.precise) {
        double resid = (double) c.p.f0 - 2.0 * sdbh::kPi * (double) c.center / (double) W;
        if (resid > sdbh::kPi) resid -= 2.0 * sdbh::kPi;
        float dec = (float) W / (float) c.size;
        float fnor = (float) (resid * (double) dec / sdbh::kPi);
        d.lo_omega = 3.14159265358979323846f * fnor;
      }
      std::vector<float> kh, xf;
      sdbh::channel_weights(W, c.halfw, kh);
      sdbh::xfade_fill(c.size, xf);
      float *dkh = e->dalloc<float>(kh.size()), *dxf = e->dalloc<float>(xf.size());
      if (!dkh || !dxf) return fail("out of device memory");
      CK(cudaMemcpy(dkh, kh.data(), kh.size() * sizeof(float), cudaMemcpyHostToDevice));
      CK(cudaMemcpy(dxf, xf.data(), xf.size() * sizeof(float), cudaMemcpyHostToDevice));
      d.kh = dkh; d.xfade = dxf; d.tw = e->twiddle(c.size);
      if (!d.tw) return fail("out of device memory");
      d.out_off = out_off; d.out_cap = e->max_hops * c.halfsz; out_off += d.out_cap;
      d.tail_off = tail_off; tail_off += c.halfsz;
      by_size[(int) c.size].push_back(k);
    }
    e->chan_stride = out_off; e->tail_stride = tail_off;
    e->d_chans = e->dalloc<SdbChannelDev>(K);
    e->d_chanb[0] = e->dalloc<float2>((size_t) S * out_off);
    e->d_chanb[1] = e->dalloc<float2>((size_t) S * out_off);
    e->d_tails = e->dalloc<float2>((size_t) S * tail_off);
    e->d_lo_phase = e->dalloc<float>((size_t) S * K);
    if (!e->d_chans || !e->d_chanb[0] || !e->d_chanb[1] || !e->d_tails || !e->d_lo_phase)
      return fail("out of device memory (channels)");
    CK(cudaStreamCreateWithFlags(&e->insp_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CK(cudaEventCreateWithFlags(&e->ev_chan[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&e->ev_insp[i], cudaEventDisableTiming));
    }
    CK(cudaMemcpy(e->d_chans, e->h_chans.data(), K * sizeof(SdbChannelDev), cudaMemcpyHostToDevice));
    CK(cudaMemset(e->d_tails, 0, (size_t) S * tail_off * sizeof(float2)));
    CK(cudaMemset(e->d_lo_phase, 0, (size_t) S * K * sizeof(float)));
    for (auto &kv : by_size) {
      sdb_engine::Group g; g.size = kv.first; g.len = (int) kv.second.size(); g.any_precise = 0;
      for (int id : kv.second) if (e->h_chans[id].precise) g.any_precise = 1;
      if (!sdb_chan_ifft_fits(g.size, g.any_precise))     // fail here rather than at every feed
        return fail("channel inverse transform of this size does not fit in shared memory");
      g.d_ids = e->dalloc<int>(kv.second.size());
      if (!g.d_ids) return fail("out of device memory");
      CK(cudaMemcpy(g.d_ids, kv.second.data(), kv.second.size() * sizeof(int), cudaMemcpyHostToDevice));
      e->groups.push_back(g);
    }
    // ---- inspector spectrum sources / estimators (SPEC U)
    {
      std::vector<SdbSpectCfg> sc(K);
      size_t off = 0; int max_ns = 0; bool any = false;
      for (int k = 0; k < K; ++k) {
        const Channel &c = e->channels[k];
        SdbSpectCfg &q = sc[k];
        memset(&q, 0, sizeof(q));
        if (c.spect_kind == 0 && c.est_mask == 0) continue;
        any = true;
        const unsigned ns = c.spect_size ? c.spect_size : 1024u;
        q.kind = c.spect_kind; q.ns = (int) ns; q.logns = ilog2u(ns); q.est_mask = c.est_mask;
        q.fs_ch = (float) (e->samp_rate * (double) c.size / (double) W);
        q.tw = e->twiddle(ns);
        if (!q.tw) return fail("out of device memory");
        auto it = e->bh_windows.find(ns);
        if (it == e->bh_windows.end()) {
          std::vector<float> w;
          sdbh::window_fill(w, ns, SDB_WINDOW_BLACKMANN_HARRIS);
          float *d = e->dalloc<float>(ns);
          if (!d) return fail("out of device memory");
          CK(cudaMemcpy(d, w.data(), ns * sizeof(float), cudaMemcpyHostToDevice));
          it = e->bh_windows.emplace(ns, d).first;
        }
        q.window = it->second;
        q.out_off = off; off += ns;
        max_ns = std::max(max_ns, (int) ns);
      }
      if (any) {
        e->spect_stride = off; e->spect_max_ns = max_ns; e->h_spect = sc;
        e->d_spectcfg = e->dalloc<SdbSpectCfg>(K);
        e->d_spect = e->dalloc<float>((size_t) S * off);
        e->d_spect_size = e->dalloc<uint32_t>((size_t) S * K);
        e->d_est = e->dalloc<float>((size_t) S * K * 2);
        e->d_est_valid = e->dalloc<int>((size_t) S * K * 2);
        if (!e->d_spectcfg || !e->d_spect || !e->d_spect_size || !e->d_est || !e->d_est_valid)
          return fail("out of device memory (spectrum sources)");
        CK(cudaMemcpy(e->d_spectcfg, sc.data(), K * sizeof(SdbSpectCfg), cudaMemcpyHostToDevice));
        CK(cudaMemset(e->d_spect_size, 0, (size_t) S * K * sizeof(uint32_t)));
        CK(cudaMemset(e->d_est_valid, 0, (size_t) S * K * 2 * sizeof(int)));
      }
    }
    // ---- chains
    e->h_cfg.resize(K);
    std::vector<float> taps_pool;
    size_t pool = 1, cap = 1;
    for (int k = 0; k < K; ++k) {
      if (!build_chain_cfg(e->channels[k], e->h_cfg[k], taps_pool)) return fail("invalid inspector configuration");
      SdbChainCfg &c = e->h_cfg[k];
      c.st_dl_off = 0; c.st_mh_off = 2 * (int) c.dl_size; c.st_mf_off = c.st_mh_off + (int) c.mh_size;
      c.st_pool = c.st_mf_off + 2 * c.mf_n;
      pool = std::max<size_t>(pool, (size_t) c.st_pool);
      cap = std::max<size_t>(cap, e->max_hops * e->channels[k].halfsz);
    }
    e->pool_stride = pool; e->sym_cap = cap;
    const size_t chains = (size_t) S * K;
    e->d_cfg = e->dalloc<SdbChainCfg>(K);
    e->d_state = e->dalloc<SdbChainState>(chains);
    e->insp_ctas = sdb_build_chain_map(e->h_cfg.data(), K, (int) S, e->h_chain_map);
    e->d_chain_map = e->dalloc<int>(e->h_chain_map.size());
    if (!e->d_chain_map) return fail("out of device memory (chain map)");
    CK(cudaMemcpy(e->d_chain_map, e->h_chain_map.data(), e->h_chain_map.size() * sizeof(int), cudaMemcpyHostToDevice));
    const size_t pool_floats = (size_t) e->insp_ctas * 32 * pool;   // per-CTA interleaved [slot][lane]
    e->d_pool = e->dalloc<float>(pool_floats);
    e->d_taps = e->dalloc<float>(taps_pool.size());
    for (int i = 0; i < 2; ++i) {
      e->d_softb[i] = e->dalloc<float2>(chains * cap);
      e->d_hardb[i] = e->dalloc<uint8_t>(chains * cap);
      e->d_countsb[i] = e->dalloc<uint32_t>(chains);
      if (!e->d_softb[i] || !e->d_hardb[i] || !e->d_countsb[i]) return fail("out of device memory (symbols)");
      CK(cudaMemset(e->d_countsb[i], 0, chains * sizeof(uint32_t)));
    }
    e->d_soft = e->d_softb[0]; e->d_hard = e->d_hardb[0]; e->d_counts = e->d_countsb[0];
    if (!e->d_cfg || !e->d_state || !e->d_pool || !e->d_taps || !e->d_soft || !e->d_hard || !e->d_counts)
      return fail("out of device memory (chains)");
    CK(cudaMemcpy(e->d_cfg, e->h_cfg.data(), K * sizeof(SdbChainCfg), cudaMemcpyHostToDevice));
    if (!taps_pool.empty())
      CK(cudaMemcpy(e->d_taps, taps_pool.data(), taps_pool.size() * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<SdbChainState> st(chains);
    for (size_t ci = 0; ci < chains; ++ci) {
      const SdbChainCfg &c = e->h_cfg[ci % K];
      SdbChainState &s = st[ci];
      memset(&s, 0, sizeof(s));
      s.fast_level = s.slow_level = s.peak = -160.0f;
      s.k_phi = 0.25f; s.k_bnor = c.bnor; s.eq_wr[0] = 1.0f;
    }
    CK(cudaMemcpy(e->d_state, st.data(), chains * sizeof(SdbChainState), cudaMemcpyHostToDevice));
    {
      // lines start empty: delay line and filter line 0, magnitude history at the -160 dB floor (SPEC A); the engine
      // never asks the kernel for a `fresh` start, so that a re-planned engine can take over running chains
      std::vector<float> hp(pool_floats, 0.0f);
      for (size_t q = 0; q < e->h_chain_map.size(); ++q) {
        const int g = e->h_chain_map[q];
        if (g < 0) continue;
        const SdbChainCfg &c = e->h_cfg[g / (int) S];
        if (!c.have_agc) continue;
        float *base = hp.data() + (q / 32) * 32 * pool + (q % 32);
        for (unsigned i = 0; i < c.mh_size; ++i) base[(size_t) (c.st_mh_off + (int) i) * 32] = -160.0f;
      }
      CK(cudaMemcpy(e->d_pool, hp.data(), pool_floats * sizeof(float), cudaMemcpyHostToDevice));
    }
    e->chains_fresh = false;
    CK(cudaMemset(e->d_counts, 0, chains * sizeof(uint32_t)));
  }
  if (e->prm.flags & SDB_FLAG_DC_REMOVE) {
    e->d_dc_state = e->dalloc<float2>(S); e->d_dc_cur = e->dalloc<float2>(S);
    e->d_dc_part = e->dalloc<double2>((size_t) S * ((max_feed + 255) / 256));
    e->d_xdc = e->dalloc<float2>((size_t) S * max_feed);
    if (!e->d_dc_state || !e->d_dc_cur || !e->d_dc_part || !e->d_xdc) return fail("out of device memory (DC removal)");
    CK(cudaMemset(e->d_dc_state, 0, S * sizeof(float2)));
  }
  CK(cudaStreamCreateWithFlags(&e->h2d_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&e->d2h_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    CK(cudaEventCreateWithFlags(&e->ev_psd_ready[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_psd_read[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_sym_read[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_xfree[i], cudaEventDisableTiming));
  }
  e->committed = true;
  return 0;
}

extern "C" int sdb_engine_feed_device(sdb_engine_t *e, const sdb_complex *xv, size_t stride, size_t n)
{
  if (!e || !xv) return fail("null argument");
  if (!e->committed) return fail("engine not committed");
  const unsigned S = e->prm.n_streams, W = e->W, Np = e->Np;
  const int K = (int) e->channels.size();
  if (n == 0 || n > e->prm.max_feed) return fail("feed size out of range");
  if (Np && n % Np) return fail("feed size must be a multiple of psd_size");
  if (K && n % (W / 2)) return fail("feed size must be a multiple of st_window_size / 2");
  CK(cudaSetDevice(e->prm.device));
  const void *x = reinterpret_cast<const void *>(xv);
  int fmt = e->prm.input_format | ((e->prm.flags & SDB_FLAG_IQ_REVERSE) ? SDB_FMT_SWAP : 0);
  if (e->d_xdc) {
    // SPEC R: the block is corrected with the estimate of the blocks before it; everything downstream reads the
    // corrected float32 copy (format conversion and I/Q swap happen in this pass)
    const float alpha = (float) (1.0 - exp(-(double) n / (e->samp_rate * 0.1)));
    CK(sdb_launch_dc_remove(e->stream, x, fmt, stride, n, (int) S, alpha, e->d_dc_state, e->d_dc_cur, e->d_dc_part,
                            e->d_xdc));
    e->launches += 3;
    x = e->d_xdc; fmt = SDB_FMT_F32; stride = n;
  }
  const size_t bps = sdb_fmt_bytes(fmt);
  SdbLaunchCtx ctx{ e->stream, &e->launches };
  const int shift_db = (e->prm.flags & SDB_FLAG_PSD_SHIFT_DB) ? 1 : 0;
  const int ob = (int) (e->feed_index & 1u);     // result buffers of this feed

  // transform launchers: windows [w0, w0 + cw) of the flattened [stream][window] order, scratch region `scr`
  auto psd_chunk = [&](const SdbLaunchCtx &lc, int frames, int w0, int cw, float2 *scr) -> int {
    SdbPassAArgs a{};
    a.x = x; a.fmt = fmt; a.stream_stride = stride; a.hist = nullptr; a.hist_len = 0;
    a.windows_per_stream = frames; a.first_window = 0; a.hop = (int) Np; a.base_off = 0;
    a.window = e->d_window; a.scratch = scr;
    const bool fast = e->fs_psd.N2 == 256 && e->fs_psd.N1 >= 32 && e->fs_psd.N1 <= 256;        // SPEC F.4 / F.5
    e->span_begin(FAM_COLS, lc.stream);
    if (fast && e->fs_psd.N1 == 256) CK(sdb_launch_cols256(lc, e->fs_psd, a, e->fs_psd.twN, w0, cw));
    else if (fast)                   CK(sdb_launch_cols128(lc, e->fs_psd, a, w0, cw));
    else                             CK(sdb_launch_pass_a_range(lc, e->fs_psd, a, w0, cw));
    e->span_end(lc.stream);
    SdbPassBArgs b{};
    b.scratch = scr; b.n_windows = cw; b.psd = e->d_psd + (size_t) w0 * Np;
    b.inv_n = 1.0f / (float) Np; b.shift_db = shift_db;
    e->span_begin(FAM_ROWS_PSD, lc.stream);
    if (fast) CK(sdb_launch_rows256(lc, e->fs_psd, b, 0));
    else      CK(sdb_launch_pass_b_psd(lc, e->fs_psd, b));
    e->span_end(lc.stream);
    return 0;
  };
  auto chan_chunk = [&](const SdbLaunchCtx &lc, int wps, int first, int w0, int cw, float2 *scr) -> int {
    SdbPassAArgs a{};
    a.x = x; a.fmt = fmt; a.stream_stride = stride; a.hist = e->d_hist; a.hist_len = (int) (W / 2);
    a.windows_per_stream = wps; a.first_window = first; a.hop = (int) (W / 2); a.base_off = 0;
    a.window = nullptr; a.scratch = scr;
    const bool fast = e->fs_st.N2 == 256 && e->fs_st.N1 >= 32 && e->fs_st.N1 <= 256;
    e->span_begin(FAM_COLS, lc.stream);
    if (fast && e->fs_st.N1 == 256) CK(sdb_launch_cols256(lc, e->fs_st, a, e->fs_st.twN, w0, cw));
    else if (fast)                  CK(sdb_launch_cols128(lc, e->fs_st, a, w0, cw));
    else                            CK(sdb_launch_pass_a_range(lc, e->fs_st, a, w0, cw));
    e->span_end(lc.stream);
    SdbPassBArgs b{};
    b.scratch = scr; b.n_windows = cw; b.binmap = e->d_binmap;
    b.cspec = e->d_cspec + (size_t) w0 * e->n_bins; b.n_bins = e->n_bins; b.ka_mask = e->ka_mask;
    e->span_begin(FAM_ROWS_CHAN, lc.stream);
    if (fast) CK(sdb_launch_rows256(lc, e->fs_st, b, 1));
    else      CK(sdb_launch_pass_b_chan(lc, e->fs_st, b));
    e->span_end(lc.stream);
    return 0;
  };

  const int frames = Np ? (int) (n / Np) : 0;
  const int H = K ? (int) (n / (W / 2)) : 0;
  const int first = (K && e->first_feed) ? 1 : 0;
  const int wps = K ? H - first : 0;
  // Stream groups: G whole streams per step, PSD frames on psd_stream and channeliser windows on the main stream,
  // each with its own part of the pinned scratch (G * (frames + wps) windows <= chunk_windows).
  int G = 0;
  if (e->psd_stream && Np && !e->psd_small && wps > 0) {
    G = e->chunk_windows / (frames + wps);
    // the largest group that fits the pinned scratch is the fastest (cfg2, 2048 streams: 12 streams 64.7 GS/s,
    // 9 streams -- whole waves for either kernel alone -- 63.1, 8: 60.2, 6: 54.2; the two chains overlap, so
    // wave quantisation of a single launch does not matter)
    if (const char *env = getenv("SDB_GROUP_STREAMS")) { const long v = atol(env); if (v >= 1 && v <= G * 4) G = (int) v; }
    if ((size_t) G * (frames + wps) > (size_t) e->chunk_windows) G = e->chunk_windows / (frames + wps);
  }
  if (G > (int) S) G = (int) S;

  if (Np) {
    e->last_frames = frames;
    e->d_psd = e->d_psdb[ob];
  }
  if (G >= 1) {
    // timing mode (sdb_engine_timing): every kernel on the main stream, so that the CUDA-event spans are the
    // kernels' own durations and not those of two chains sharing the SMs
    SdbLaunchCtx pctx{ e->timing ? e->stream : e->psd_stream, &e->launches };
    CK(cudaEventRecord(e->ev_feed, e->stream));              // the input is valid from here on
    CK(cudaStreamWaitEvent(e->psd_stream, e->ev_feed, 0));
    if (e->psd_read_valid[ob]) CK(cudaStreamWaitEvent(e->psd_stream, e->ev_psd_read[ob], 0));   // async read of feed i-2
    float2 *scr_psd = e->d_scratch, *scr_ch = e->d_scratch + (size_t) G * frames * Np;
    for (int s0 = 0; s0 < (int) S; s0 += G) {
      const int g = std::min(G, (int) S - s0);
      if (psd_chunk(pctx, frames, s0 * frames, g * frames, scr_psd)) return -1;
      if (chan_chunk(ctx, wps, first, s0 * wps, g * wps, scr_ch)) return -1;
    }
    if (e->chdet) CK(sdb_chdet_feed_stream(e->chdet, e->d_psd, (uint32_t) frames, (size_t) frames * Np, e->psd_stream,
                                           &e->launches));
    CK(cudaEventRecord(e->ev_psd_ready[ob], e->psd_stream));
    CK(cudaStreamWaitEvent(e->stream, e->ev_psd_ready[ob], 0));   // the main stream stays the engine's timeline
  } else {
    // ---- main PSD
    if (Np) {
      if (e->psd_read_valid[ob]) CK(cudaStreamWaitEvent(e->stream, e->ev_psd_read[ob], 0));   // async read of feed i-2
      if (e->psd_small) {
        e->span_begin(FAM_ROWS_PSD);
        CK(sdb_launch_small_psd(ctx, (int) Np, e->twiddle(Np), x, fmt, stride, frames, (int) S, e->d_window,
                                e->d_psd, shift_db));
        e->span_end();
      } else {
        const int total = frames * (int) S;
        for (int w0 = 0; w0 < total; w0 += e->chunk_windows)
          if (psd_chunk(ctx, frames, w0, std::min(e->chunk_windows, total - w0), e->d_scratch)) return -1;
      }
      if (e->chdet) CK(sdb_chdet_feed_stream(e->chdet, e->d_psd, (uint32_t) frames, (size_t) frames * Np, e->stream,
                                             &e->launches));
      CK(cudaEventRecord(e->ev_psd_ready[ob], e->stream));
    }
    // ---- channeliser forward transforms
    if (K && wps > 0) {
      const int total = wps * (int) S;
      for (int w0 = 0; w0 < total; w0 += e->chunk_windows)
        if (chan_chunk(ctx, wps, first, w0, std::min(e->chunk_windows, total - w0), e->d_scratch)) return -1;
    }
  }
  // ---- per-channel inverse transforms + inspectors
  if (K) {
    e->last_hops = wps > 0 ? wps : 0;
    if (wps > 0) {
      const int b = (int) (e->feed_index & 1u);
      e->last_buf = b;
      // buffer b was last read by the inspector launch of feed i-2
      if (e->ev_insp_valid[b]) CK(cudaStreamWaitEvent(e->stream, e->ev_insp[b], 0));
      e->span_begin(FAM_CHAN_IFFT);
      for (auto &g : e->groups)
        CK(sdb_launch_chan_ifft_group(ctx, e->d_chans, g.d_ids, g.len, g.size, K, (int) S, e->d_cspec,
                                      e->n_bins, wps, e->d_tails, e->tail_stride, e->d_lo_phase, e->d_chanb[b],
                                      e->chan_stride, g.any_precise));
      e->span_end();
      CK(cudaEventRecord(e->ev_chan[b], e->stream));
      CK(cudaStreamWaitEvent(e->insp_stream, e->ev_chan[b], 0));
      e->d_soft = e->d_softb[b]; e->d_hard = e->d_hardb[b]; e->d_counts = e->d_countsb[b];
      if (e->sym_read_valid[b]) CK(cudaStreamWaitEvent(e->insp_stream, e->ev_sym_read[b], 0));
      SdbLaunchCtx ictx{ e->timing ? e->stream : e->insp_stream, &e->launches };
      if (e->d_spectcfg)
        CK(sdb_launch_spectsrc(ictx, e->d_spectcfg, e->d_chans, K, (int) S, e->spect_max_ns, e->d_chanb[b],
                               e->chan_stride, (uint32_t) wps, e->d_spect, e->spect_stride, e->d_spect_size,
                               e->d_est, e->d_est_valid));
      e->span_begin(FAM_INSPECTOR, ictx.stream);
      CK(sdb_launch_inspectors_n(ictx, e->d_cfg, K, (int) S, e->d_chain_map, e->insp_ctas, e->d_state, e->d_pool,
                                 e->pool_stride, e->d_taps,
                                 e->d_chans, e->d_chanb[b], e->chan_stride, (uint32_t) wps, e->d_soft, e->d_hard,
                                 e->d_counts, e->sym_cap, e->chains_fresh ? 1 : 0,
                                 sdb_insp_dyn(e->h_cfg.data(), K)));
      e->chains_fresh = false;
      e->span_end(ictx.stream);
      CK(cudaEventRecord(e->ev_insp[b], ictx.stream));
      e->ev_insp_valid[b] = true;
    } else {
      e->d_counts = e->d_countsb[ob];
      e->last_buf = ob;
      if (e->sym_read_valid[ob]) CK(cudaStreamWaitEvent(e->insp_stream, e->ev_sym_read[ob], 0));
      CK(cudaMemsetAsync(e->d_counts, 0, (size_t) S * K * sizeof(uint32_t), e->insp_stream));
      CK(cudaEventRecord(e->ev_insp[ob], e->insp_stream));
      e->ev_insp_valid[ob] = true;
    }
    // keep the last half window of every stream as history for the next feed
    if (fmt == SDB_FMT_F32)
      CK(cudaMemcpy2DAsync(e->d_hist, (W / 2) * sizeof(float2), reinterpret_cast<const float2 *>(x) + (n - W / 2),
                           stride * sizeof(float2), (W / 2) * sizeof(float2), S, cudaMemcpyDeviceToDevice, e->stream));
    else
      CK(sdb_launch_hist_convert(e->stream, x, fmt, stride, n - W / 2, e->d_hist, (int) (W / 2), (int) S));
    e->first_feed = false;
  }
  ++e->feed_index;
  e->n_fed += n;
  return 0;
}

extern "C" int sdb_engine_feed_host(sdb_engine_t *e, const sdb_complex *x, size_t stride, size_t n)
{
  if (!e || !x) return fail("null argument");
  if (!e->committed) return fail("engine not committed");
  if (n == 0 || n > e->prm.max_feed) return fail("feed size out of range");
  CK(cudaSetDevice(e->prm.device));
  const unsigned S = e->prm.n_streams;
  const int hb = (int) (e->host_feeds & 1u);
  const size_t bps = sdb_fmt_bytes(e->prm.input_format);
  if (!e->d_xinb[hb]) {
    e->d_xinb[hb] = e->dalloc<float2>((size_t) S * e->prm.max_feed);
    if (!e->d_xinb[hb]) return fail("out of device memory (input staging)");
  }
  // H2D on its own stream into staging buffer hb, as soon as the kernels of feed i-2 are done with it;
  // the kernels of this feed wait for the copy.  Copies of consecutive feeds overlap compute.
  if (e->xfree_valid[hb]) CK(cudaStreamWaitEvent(e->h2d_stream, e->ev_xfree[hb], 0));
  if (stride == n)
    CK(cudaMemcpyAsync(e->d_xinb[hb], x, (size_t) S * n * bps, cudaMemcpyHostToDevice, e->h2d_stream));
  else
    CK(cudaMemcpy2DAsync(e->d_xinb[hb], n * bps, x, stride * bps, n * bps, S,
                         cudaMemcpyHostToDevice, e->h2d_stream));
  CK(cudaEventRecord(e->ev_h2d[hb], e->h2d_stream));
  CK(cudaStreamWaitEvent(e->stream, e->ev_h2d[hb], 0));
  int rc = sdb_engine_feed_device(e, reinterpret_cast<const sdb_complex *>(e->d_xinb[hb]), n, n);
  if (rc) return rc;
  CK(cudaEventRecord(e->ev_xfree[hb], e->stream));
  e->xfree_valid[hb] = true;
  ++e->host_feeds;
  return 0;
}

extern "C" int sdb_engine_sync(sdb_engine_t *e)
{
  if (!e) return fail("null engine");
  CK(cudaSetDevice(e->prm.device));
  CK(e->join());
  CK(cudaStreamSynchronize(e->stream));
  if (e->d2h_stream) CK(cudaStreamSynchronize(e->d2h_stream));
  if (e->h2d_stream) CK(cudaStreamSynchronize(e->h2d_stream));
  e->collect_spans();
  return 0;
}

// Queue a dependency: work submitted to the engine stream after this call starts only once the
// inspector kernels of all previous feeds have finished (they run on a second stream so that the
// next feed's FFT kernels overlap them).  Use before recording an event that should cover a feed.
extern "C" int sdb_engine_join(sdb_engine_t *e)
{
  if (!e) return fail("null engine");
  CK(cudaSetDevice(e->prm.device));
  CK(e->join());
  return 0;
}

extern "C" size_t sdb_engine_psd_frames(const sdb_engine_t *e) { return e ? e->last_frames : 0; }
extern "C" const float *sdb_engine_psd_device(const sdb_engine_t *e) { return e ? e->d_psd : nullptr; }

extern "C" int sdb_engine_read_psd(sdb_engine_t *e, float *dst, size_t cap)
{
  if (!e || !dst) return fail("null argument");
  const size_t n = (size_t) e->prm.n_streams * e->last_frames * e->Np;
  if (cap < n) return fail("destination too small");
  if (sdb_engine_read_psd_async(e, dst, cap)) return -1;
  CK(cudaStreamSynchronize(e->d2h_stream));
  return 0;
}

// Asynchronous variants: the copy is queued on the engine's D2H stream behind the kernels that produce
// the data; the next feed may be submitted immediately (results are double-buffered by feed parity, a
// buffer is reused two feeds later and its writer waits for this copy).  dst should be pinned memory and
// must stay valid until sdb_engine_sync().
extern "C" int sdb_engine_read_psd_async(sdb_engine_t *e, float *dst, size_t cap)
{
  if (!e || !dst) return fail("null argument");
  if (!e->committed || !e->Np || e->feed_index == 0) return fail("no PSD available");
  const size_t n = (size_t) e->prm.n_streams * e->last_frames * e->Np;
  if (cap < n) return fail("destination too small");
  const int ob = (int) ((e->feed_index - 1) & 1u);
  CK(cudaSetDevice(e->prm.device));
  CK(cudaStreamWaitEvent(e->d2h_stream, e->ev_psd_ready[ob], 0));
  CK(cudaMemcpyAsync(dst, e->d_psdb[ob], n * sizeof(float), cudaMemcpyDeviceToHost, e->d2h_stream));
  CK(cudaEventRecord(e->ev_psd_read[ob], e->d2h_stream));
  e->psd_read_valid[ob] = true;
  return 0;
}

extern "C" long sdb_engine_read_channel(sdb_engine_t *e, uint32_t stream, int handle, sdb_complex *dst, size_t cap)
{
  if (!e || !dst) return fail("null argument");
  if (handle < 0 || handle >= (int) e->channels.size()) return fail("wrong handle");
  if (stream >= e->prm.n_streams) return fail("stream out of range");
  const SdbChannelDev &d = e->h_chans[handle];
  size_t n = e->last_hops * (size_t) d.halfsz;
  if (n > cap) n = cap;
  CK(cudaSetDevice(e->prm.device));
  CK(cudaMemcpyAsync(dst, e->d_chanb[e->last_buf] + (size_t) stream * e->chan_stride + d.out_off, n * sizeof(float2),
                     cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return (long) n;
}

extern "C" long sdb_engine_read_symbols(sdb_engine_t *e, uint32_t stream, int handle, sdb_complex *soft,
                                        uint8_t *hard, size_t cap)
{
  if (!e) return fail("null argument");
  const int K = (int) e->channels.size();
  if (handle < 0 || handle >= K) return fail("wrong handle");
  if (stream >= e->prm.n_streams) return fail("stream out of range");
  const size_t chain = (size_t) stream * K + handle;
  uint32_t cnt = 0;
  CK(cudaSetDevice(e->prm.device));
  CK(e->join());
  CK(cudaMemcpyAsync(&cnt, e->d_counts + chain, sizeof(cnt), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  size_t n = cnt;
  if (n > cap) n = cap;
  if (soft) CK(cudaMemcpyAsync(soft, e->d_soft + chain * e->sym_cap, n * sizeof(float2), cudaMemcpyDeviceToHost, e->stream));
  if (hard) CK(cudaMemcpyAsync(hard, e->d_hard + chain * e->sym_cap, n, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return (long) n;
}

extern "C" int sdb_engine_read_all_symbols(sdb_engine_t *e, uint32_t *counts, sdb_complex *soft, uint8_t *hard,
                                           size_t cap)
{
  if (!e || !counts) return fail("null argument");
  const size_t chains = (size_t) e->prm.n_streams * e->channels.size();
  if (chains == 0) return 0;
  if (sdb_engine_read_all_symbols_async(e, counts, soft, hard, cap)) return -1;
  CK(cudaStreamSynchronize(e->d2h_stream));
  return 0;
}

extern "C" int sdb_engine_read_all_symbols_async(sdb_engine_t *e, uint32_t *counts, sdb_complex *soft,
                                                 uint8_t *hard, size_t cap)
{
  if (!e || !counts) return fail("null argument");
  const size_t chains = (size_t) e->prm.n_streams * e->channels.size();
  if (chains == 0) return 0;
  if (e->feed_index == 0) return fail("no symbols available");
  const int ob = (int) ((e->feed_index - 1) & 1u);
  CK(cudaSetDevice(e->prm.device));
  // everything queued so far on the inspector stream (including this feed's launch or its count reset)
  if (e->ev_insp_valid[ob]) CK(cudaStreamWaitEvent(e->d2h_stream, e->ev_insp[ob], 0));
  CK(cudaMemcpyAsync(counts, e->d_countsb[ob], chains * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->d2h_stream));
  const size_t w = std::min(cap, e->sym_cap);
  if (soft) CK(cudaMemcpy2DAsync(soft, cap * sizeof(float2), e->d_softb[ob], e->sym_cap * sizeof(float2),
                                 w * sizeof(float2), chains, cudaMemcpyDeviceToHost, e->d2h_stream));
  if (hard) CK(cudaMemcpy2DAsync(hard, cap, e->d_hardb[ob], e->sym_cap, w, chains, cudaMemcpyDeviceToHost, e->d2h_stream));
  CK(cudaEventRecord(e->ev_sym_read[ob], e->d2h_stream));
  e->sym_read_valid[ob] = true;
  return 0;
}

// destination of a device-written read: device memory as is, pinned / registered host memory through its device
// alias; anything else cannot be written by a kernel and is refused
static int device_writable(void *p, void **dev, const char *what)
{
  *dev = nullptr;
  if (!p) return 0;
  if (((uintptr_t) p & 15u) != 0) return fail(std::string("packed symbol read: ") + what + " must be 16-byte aligned");
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return fail(std::string("packed symbol read: ") + what + " is not pinned host or device memory"); }
  if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) { *dev = p; return 0; }
  if (at.type == cudaMemoryTypeHost && at.devicePointer) { *dev = at.devicePointer; return 0; }
  return fail(std::string("packed symbol read: ") + what + " must be pinned (cudaHostAlloc / cudaHostRegister) host "
              "memory or device memory: the GPU writes it directly");
}

extern "C" int sdb_engine_read_symbols_packed_async(sdb_engine_t *e, uint32_t *counts, uint64_t *offsets,
                                                    sdb_complex *soft, uint8_t *hard, size_t cap_total)
{
  if (!e || !counts || !offsets) return fail("null argument");
  const size_t chains = (size_t) e->prm.n_streams * e->channels.size();
  if (chains == 0) return 0;
  if (e->feed_index == 0) return fail("no symbols available");
  const int ob = (int) ((e->feed_index - 1) & 1u);
  CK(cudaSetDevice(e->prm.device));
  void *dsoft = nullptr, *dhard = nullptr;
  if (device_writable(soft, &dsoft, "soft") || device_writable(hard, &dhard, "hard")) return -1;
  if (!e->d_sym_off[ob]) {
    e->d_sym_off[ob] = e->dalloc<unsigned long long>(chains + 1);
    if (!e->d_sym_off[ob]) return fail("out of device memory (symbol offsets)");
  }
  if (e->ev_insp_valid[ob]) CK(cudaStreamWaitEvent(e->d2h_stream, e->ev_insp[ob], 0));
  CK(sdb_launch_sym_pack(e->d2h_stream, e->d_countsb[ob], e->d_sym_off[ob], chains, e->d_softb[ob], e->d_hardb[ob],
                         e->sym_cap, dsoft, dhard, (unsigned long long) cap_total, &e->launches));
  CK(cudaMemcpyAsync(counts, e->d_countsb[ob], chains * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->d2h_stream));
  CK(cudaMemcpyAsync(offsets, e->d_sym_off[ob], (chains + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, e->d2h_stream));
  CK(cudaEventRecord(e->ev_sym_read[ob], e->d2h_stream));
  e->sym_read_valid[ob] = true;
  return 0;
}

extern "C" int sdb_engine_read_symbols_packed(sdb_engine_t *e, uint32_t *counts, uint64_t *offsets, sdb_complex *soft,
                                              uint8_t *hard, size_t cap_total)
{
  if (sdb_engine_read_symbols_packed_async(e, counts, offsets, soft, hard, cap_total)) return -1;
  CK(cudaStreamSynchronize(e->d2h_stream));
  return 0;
}

extern "C" const uint32_t *sdb_engine_symbol_counts_device(const sdb_engine_t *e) { return e ? e->d_counts : nullptr; }
extern "C" size_t sdb_engine_symbol_capacity(const sdb_engine_t *e) { return e ? e->sym_cap : 0; }
extern "C" void *sdb_engine_stream(const sdb_engine_t *e) { return e ? (void *) e->stream : nullptr; }
extern "C" uint64_t sdb_engine_launch_count(const sdb_engine_t *e) { return e ? e->launches : 0; }
extern "C" void sdb_engine_timing(sdb_engine_t *e, int enable)
{
  if (!e) return;
  e->timing = enable != 0;
  for (int i = 0; i < FAM_COUNT; ++i) { e->fam_ms[i] = 0; e->fam_n[i] = 0; }
}
cudaError_t sdb_stage_cycles(unsigned long long out[8], int reset);
extern "C" int sdb_debug_stage_cycles(uint64_t out[8], int reset)
{
  unsigned long long tmp[8];
  CK(cudaDeviceSynchronize());
  CK(sdb_stage_cycles(tmp, reset));
  for (int i = 0; i < 8; ++i) out[i] = tmp[i];
  return 0;
}

cudaError_t sdb_stage_cta_cycles(unsigned long long out[64], int reset);
extern "C" int sdb_debug_cta_cycles(uint64_t out[64], int reset)
{
  unsigned long long tmp[64];
  CK(cudaDeviceSynchronize());
  CK(sdb_stage_cta_cycles(tmp, reset));
  for (int i = 0; i < 64; ++i) out[i] = tmp[i];
  return 0;
}

extern "C" int sdb_engine_kernel_time(sdb_engine_t *e, const char *family, double *avg_ms, uint64_t *launches)
{
  if (!e || !family) return fail("null argument");
  for (int i = 0; i < FAM_COUNT; ++i)
    if (!strcmp(family, kFamNames[i])) {
      if (avg_ms) *avg_ms = e->fam_n[i] ? e->fam_ms[i] / (double) e->fam_n[i] : 0.0;
      if (launches) *launches = e->fam_n[i];
      return 0;
    }
  return fail("unknown kernel family");
}

// ---------------------------------------------------------------------------------------------
// Tasks/ primitives on host buffers
// ---------------------------------------------------------------------------------------------
struct TaskBufs {
  float2 *src = nullptr, *dst = nullptr; float *pool = nullptr; SdbChainCfg *cfg = nullptr;
  ~TaskBufs() { cudaFree(src); cudaFree(dst); cudaFree(pool); cudaFree(cfg); }
  int put_cfg(const SdbChainCfg &c)
  {
    CK(cudaMalloc(&cfg, sizeof(c)));
    CK(cudaMemcpy(cfg, &c, sizeof(c), cudaMemcpyHostToDevice));
    return 0;
  }
};

static int task_io_begin(TaskBufs &b, const sdb_complex *src, size_t n, size_t batch)
{
  if (!src || n == 0 || batch == 0) return fail("invalid task buffer");
  if (sdb_device_count() <= 0) return fail("no CUDA device: sigdigger_b200 has no CPU fallback");
  CK(cudaMalloc(&b.src, n * batch * sizeof(float2)));
  CK(cudaMalloc(&b.dst, n * batch * sizeof(float2)));
  CK(cudaMemcpy(b.src, src, n * batch * sizeof(float2), cudaMemcpyHostToDevice));
  return 0;
}
static int task_io_end(TaskBufs &b, sdb_complex *dst, size_t n, size_t batch)
{
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(dst, b.dst, n * batch * sizeof(float2), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int sdb_task_carrier_xlate(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch,
                                      float rel_freq, float phase)
{
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  // su_ncqo_init(-relFreq); su_ncqo_set_phase(-phase)   (Tasks/CarrierXlator.cpp:36-37)
  float omega = 3.14159265358979323846f * (-rel_freq);
  float phi = -phase;
  phi = phi - 6.28318530717958647692f * floorf(phi / 6.28318530717958647692f);
  if (phi >= 6.28318530717958647692f) phi = 0.0f;
  CK(sdb_launch_task_xlate(0, b.src, b.dst, n, batch, omega, phi));
  return task_io_end(b, dst, n, batch);
}

extern "C" int sdb_task_quad_demod(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch)
{
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  CK(sdb_launch_task_quad(0, b.src, b.dst, n, batch));
  return task_io_end(b, dst, n, batch);
}

extern "C" int sdb_task_costas(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch, int kind,
                               float tau, float loop_bw)
{
  if (kind < 1 || kind > 3) return fail("invalid Costas kind");
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  SdbChainCfg c; memset(&c, 0, sizeof(c));
  // su_costas_init(&costas, kind, 0, 1/tau, 3, loopbw)   (Tasks/CostasRecoveryTask.cpp:36-41)
  c.costas_kind = kind;
  c.c_a = 3.14159265358979323846f * loop_bw;
  c.c_b = 0.5f * c.c_a * c.c_a;
  if (!sdbh::butter_lp(2, 1.0f / tau, c.af_b, c.af_a)) return fail("invalid arm bandwidth");
  c.af_n = 3;
  if (b.put_cfg(c)) return -1;
  CK(sdb_launch_task_chain(0, b.src, b.dst, n, batch, b.cfg, 0, nullptr, 0));
  return task_io_end(b, dst, n, batch);
}

extern "C" int sdb_task_pll(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch, float bw)
{
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  SdbChainCfg c; memset(&c, 0, sizeof(c));
  float fc = 3.14159265358979323846f * bw;
  float dinv = 1.0f / (1.0f + 2.0f * 0.707f * fc + fc * fc);
  c.pll_alpha = 4.0f * fc * fc * dinv;
  c.pll_beta = 4.0f * 0.707f * fc * dinv;
  if (b.put_cfg(c)) return -1;
  CK(sdb_launch_task_chain(0, b.src, b.dst, n, batch, b.cfg, 1, nullptr, 0));
  return task_io_end(b, dst, n, batch);
}

extern "C" int sdb_task_agc(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch, float tau)
{
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  SdbChainCfg c; memset(&c, 0, sizeof(c));
  // AGCTask sets only the five time constants; delay line / history keep the defaults (20)
  // (Tasks/AGCTask.cpp:43-47 and the comment in SURVEY.md 8a row a6)
  sdbh::AgcDesign d = sdbh::agc_from_tau(tau, 2.0f);
  c.knee = d.knee; c.gain_slope = d.gain_slope; c.fixed_gain = d.fixed_gain;
  c.hang_max = d.hang_max; c.dl_size = 20; c.mh_size = 20;
  c.far_ = d.far_; c.faf = d.faf; c.sar = d.sar; c.saf = d.saf;
  c.st_dl_off = 0; c.st_mh_off = 40; c.st_pool = 60;
  CK(cudaMalloc(&b.pool, ((batch + 31) / 32) * 32 * 60 * sizeof(float)));
  if (b.put_cfg(c)) return -1;
  CK(sdb_launch_task_chain(0, b.src, b.dst, n, batch, b.cfg, 2, b.pool, 60));
  return task_io_end(b, dst, n, batch);
}

// ---- bulk twins of the per-sample sigutils calls, continuing from (and returning) the caller's loop state
static int task_state_run(const sdb_complex *src, sdb_complex *dst, size_t n, int mode, void *st, size_t st_bytes)
{
  if (!src || !dst || !st) return fail("null argument");
  if (sdb_device_count() <= 0) return fail("no CUDA device: sigdigger_b200 has no CPU fallback");
  if (n == 0) return 0;
  float2 *d_x = nullptr, *d_y = nullptr; float *d_st = nullptr;
  int rc = 0;
  if (cudaMalloc(&d_x, n * sizeof(float2)) != cudaSuccess || cudaMalloc(&d_y, n * sizeof(float2)) != cudaSuccess ||
      cudaMalloc(&d_st, st_bytes) != cudaSuccess) rc = fail("out of device memory");
  if (!rc && (cudaMemcpy(d_x, src, n * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
              cudaMemcpy(d_st, st, st_bytes, cudaMemcpyHostToDevice) != cudaSuccess)) rc = fail("copy failed");
  if (!rc && sdb_launch_task_chain_state(0, d_x, d_y, n, mode, d_st) != cudaSuccess) rc = fail("launch failed");
  if (!rc && (cudaMemcpy(dst, d_y, n * sizeof(float2), cudaMemcpyDeviceToHost) != cudaSuccess ||
              cudaMemcpy(st, d_st, st_bytes, cudaMemcpyDeviceToHost) != cudaSuccess)) rc = fail(cudaGetErrorString(cudaGetLastError()));
  cudaFree(d_x); cudaFree(d_y); cudaFree(d_st);
  return rc;
}
extern "C" int sdb_task_costas_state(const sdb_complex *src, sdb_complex *dst, size_t n, const void *k, size_t k_bytes,
                                     void *s, size_t s_bytes)
{
  if (k_bytes != sdb_costas_k_bytes() || s_bytes != sdb_costas_s_bytes()) return fail("costas state size mismatch");
  std::vector<unsigned char> st(k_bytes + s_bytes);
  memcpy(st.data(), k, k_bytes); memcpy(st.data() + k_bytes, s, s_bytes);
  if (task_state_run(src, dst, n, 0, st.data(), st.size())) return -1;
  memcpy(s, st.data() + k_bytes, s_bytes);
  return 0;
}
extern "C" int sdb_task_pll_state(const sdb_complex *src, sdb_complex *dst, size_t n, float alpha, float beta,
                                  float state[2])
{
  float st[4] = { alpha, beta, state[0], state[1] };
  if (task_state_run(src, dst, n, 1, st, sizeof(st))) return -1;
  state[0] = st[2]; state[1] = st[3];
  return 0;
}

// ---- take over the running state of another engine (live re-plan: suscan keeps every inspector that stays open
// ---- running when one is opened, closed or reconfigured, Suscan/Analyzer.cpp:459-537).  Channels are matched by
// ---- their parameters (f0, bw, guard, precise), first come first served: a matched channel keeps its cross-fade
// ---- tail and LO phase; if its inspector class and the sizes of its state lines are unchanged it also keeps the
// ---- loop state of every chain (AGC, Costas / PLL, matched-filter line, Gardner, CMA...), whatever else of its
// ---- configuration changed (loop bandwidths, gains, thresholds take effect at this block boundary).
static int migrate_impl(sdb_engine_t *dst, sdb_engine_t *src, const std::vector<int> &old_of_new)
{
  CK(cudaSetDevice(dst->prm.device));
  if (sdb_engine_sync(src)) return -1;
  const unsigned S = dst->prm.n_streams, W = dst->W;
  const int Kn = (int) dst->channels.size(), Ko = (int) src->channels.size();
  if (dst->d_hist && src->d_hist)
    CK(cudaMemcpy(dst->d_hist, src->d_hist, (size_t) S * (W / 2) * sizeof(float2), cudaMemcpyDeviceToDevice));
  if (dst->d_dc_state && src->d_dc_state)
    CK(cudaMemcpy(dst->d_dc_state, src->d_dc_state, S * sizeof(float2), cudaMemcpyDeviceToDevice));
  // an engine that had no channel so far kept no input history: its first window starts with this feed
  dst->first_feed = src->d_hist ? src->first_feed : true;
  dst->n_fed = src->n_fed;
  auto slot_of = [](const sdb_engine_t *e, int chain_g) {
    for (size_t q = 0; q < e->h_chain_map.size(); ++q) if (e->h_chain_map[q] == chain_g) return (long) q;
    return -1L;
  };
  for (int kn = 0; kn < Kn; ++kn) {
    const int ko = kn < (int) old_of_new.size() ? old_of_new[kn] : -1;
    if (ko < 0 || ko >= Ko) continue;
    const Channel &cn = dst->channels[kn], &co = src->channels[ko];
    const SdbChannelDev &dn = dst->h_chans[kn], &dold = src->h_chans[ko];
    const bool same_channel = co.p.f0 == cn.p.f0 && co.p.bw == cn.p.bw && co.p.guard == cn.p.guard &&
                              co.p.precise == cn.p.precise && co.size == cn.size && co.center == cn.center;
    if (same_channel && !src->first_feed) {
      CK(cudaMemcpy2D(dst->d_tails + dn.tail_off, dst->tail_stride * sizeof(float2), src->d_tails + dold.tail_off,
                      src->tail_stride * sizeof(float2), (size_t) cn.halfsz * sizeof(float2), S, cudaMemcpyDeviceToDevice));
      CK(cudaMemcpy2D(dst->d_lo_phase + kn, (size_t) Kn * sizeof(float), src->d_lo_phase + ko, (size_t) Ko * sizeof(float),
                      sizeof(float), S, cudaMemcpyDeviceToDevice));
    }
    if (!cn.has_insp || !co.has_insp) continue;
    const SdbChainCfg &a = dst->h_cfg[kn], &b = src->h_cfg[ko];
    if (a.cls != b.cls || a.have_agc != b.have_agc || a.dl_size != b.dl_size || a.mh_size != b.mh_size ||
        a.have_mf != b.have_mf || a.mf_n != b.mf_n || a.af_n != b.af_n || a.alpf_n != b.alpf_n ||
        a.have_costas != b.have_costas || a.have_pll != b.have_pll || a.eq_type != b.eq_type ||
        a.clock_type != b.clock_type)
      continue;                                            // structural change: this inspector restarts
    CK(cudaMemcpy2D(dst->d_state + kn, (size_t) Kn * sizeof(SdbChainState), src->d_state + ko,
                    (size_t) Ko * sizeof(SdbChainState), sizeof(SdbChainState), S, cudaMemcpyDeviceToDevice));
    // clock.baud is a parameter AND the start value of the Gardner loop's own estimate: a new baud restarts it
    if (a.bnor != b.bnor) {
      std::vector<SdbChainState> st(S);
      CK(cudaMemcpy2D(st.data(), sizeof(SdbChainState), dst->d_state + kn, (size_t) Kn * sizeof(SdbChainState),
                      sizeof(SdbChainState), S, cudaMemcpyDeviceToHost));
      for (auto &q : st) q.k_bnor = a.bnor;
      CK(cudaMemcpy2D(dst->d_state + kn, (size_t) Kn * sizeof(SdbChainState), st.data(), sizeof(SdbChainState),
                      sizeof(SdbChainState), S, cudaMemcpyHostToDevice));
    }
    const size_t rows = (size_t) std::min(a.st_pool, b.st_pool);
    for (unsigned s = 0; s < S; ++s) {
      const long qn = slot_of(dst, kn * (int) S + (int) s), qo = slot_of(src, ko * (int) S + (int) s);
      if (qn < 0 || qo < 0) continue;
      float *pd = dst->d_pool + (size_t) (qn / 32) * 32 * dst->pool_stride + (qn % 32);
      const float *ps = src->d_pool + (size_t) (qo / 32) * 32 * src->pool_stride + (qo % 32);
      CK(cudaMemcpy2D(pd, 32 * sizeof(float), ps, 32 * sizeof(float), sizeof(float), rows, cudaMemcpyDeviceToDevice));
    }
  }
  return 0;
}

static int migrate_check(sdb_engine_t *dst, sdb_engine_t *src)
{
  if (!dst || !src) return fail("null engine");
  if (!dst->committed || !src->committed) return fail("both engines must be committed");
  if (dst->prm.n_streams != src->prm.n_streams || dst->W != src->W || dst->prm.device != src->prm.device)
    return fail("engines differ in streams / window / device");
  return 0;
}

// can dst continue src (same streams, window, device)?  PSD size, window function, flags and feed size may differ
extern "C" int sdb_engine_same_geometry(const sdb_engine_t *a, const sdb_engine_t *b)
{
  return a && b && a->prm.n_streams == b->prm.n_streams && a->W == b->W && a->prm.device == b->prm.device;
}

extern "C" int sdb_engine_migrate(sdb_engine_t *dst, sdb_engine_t *src)
{
  if (migrate_check(dst, src)) return -1;
  const int Kn = (int) dst->channels.size(), Ko = (int) src->channels.size();
  std::vector<int> map(Kn, -1);
  std::vector<char> used(Ko, 0);
  for (int kn = 0; kn < Kn; ++kn) {
    const Channel &cn = dst->channels[kn];
    for (int k = 0; k < Ko; ++k) {
      const Channel &co = src->channels[k];
      if (!used[k] && co.p.f0 == cn.p.f0 && co.p.bw == cn.p.bw && co.p.guard == cn.p.guard &&
          co.p.precise == cn.p.precise) { map[kn] = k; used[k] = 1; break; }
    }
  }
  return migrate_impl(dst, src, map);
}

extern "C" int sdb_engine_migrate_map(sdb_engine_t *dst, sdb_engine_t *src, const int32_t *old_of_new, size_t n)
{
  if (migrate_check(dst, src)) return -1;
  if (!old_of_new && n) return fail("null map");
  std::vector<int> map(old_of_new, old_of_new + n);
  return migrate_impl(dst, src, map);
}

// ---- TimeWindow tasks that are fully specified in-repo (SPEC Y; kernels in tasks_kernels.cu)
struct DevMem {
  void *p = nullptr;
  ~DevMem() { cudaFree(p); }
  template <typename T> T *as() { return (T *) p; }
};

static int task_src_begin(DevMem &src, const sdb_complex *host, size_t n, size_t batch)
{
  if (!host || n == 0 || batch == 0) return fail("invalid task buffer");
  if (sdb_device_count() <= 0) return fail("no CUDA device: sigdigger_b200 has no CPU fallback");
  CK(cudaMalloc(&src.p, n * batch * sizeof(float2)));
  CK(cudaMemcpy(src.p, host, n * batch * sizeof(float2), cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int sdb_task_delayed_conj(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch, size_t delay)
{
  if (delay == 0) return fail("Delay is zero samples");   // DelayedConjTask.cpp:36-37
  if (!dst) return fail("null argument");
  TaskBufs b;
  if (task_io_begin(b, src, n, batch)) return -1;
  CK(sdb_launch_task_delayed_conj(0, b.src, b.dst, n, batch, delay));
  return task_io_end(b, dst, n, batch);
}

extern "C" long sdb_task_histogram_feed(const sdb_complex *src, float *out, size_t n, size_t batch, int space)
{
  if (!out) return fail("null argument");
  if (space < SDB_SPACE_AMPLITUDE || space > SDB_SPACE_FREQUENCY) return fail("unknown decision space");
  DevMem s, o;
  if (task_src_begin(s, src, n, batch)) return -1;
  const size_t count = space == SDB_SPACE_FREQUENCY ? n - 1 : n;
  if (count == 0) return 0;
  CK(cudaMalloc(&o.p, count * batch * sizeof(float)));
  CK(sdb_launch_task_hist(0, s.as<float2>(), o.as<float>(), n, batch, space));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, o.p, count * batch * sizeof(float), cudaMemcpyDeviceToHost));
  return (long) count;
}

extern "C" long sdb_task_sample_manual(const sdb_complex *src, size_t n, size_t batch, int space, size_t symbol_sync,
                                       double symbol_count, sdb_complex *out)
{
  if (!out) return fail("null argument");
  if (space < SDB_SPACE_AMPLITUDE || space > SDB_SPACE_FREQUENCY) return fail("unknown decision space");
  if (!(symbol_count >= 1.0) || symbol_count > (double) n) return fail("symbol_count must be in [1, n]");
  DevMem s, o;
  if (task_src_begin(s, src, n, batch)) return -1;
  // WaveSampler.cpp:44-45: delta = length / symbolCount; sampOffset = symbolSync / delta
  const double delta = (double) n / symbol_count;
  const double samp_offset = (double) symbol_sync / delta;
  const float delta_inv = 1.f / (float) delta;
  const long long count = (long long) symbol_count;
  CK(cudaMalloc(&o.p, (size_t) count * batch * sizeof(float2)));
  CK(sdb_launch_task_sample_manual(0, s.as<float2>(), n, batch, space, (double) symbol_sync, delta, samp_offset,
                                   delta_inv, count, o.as<float2>()));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, o.p, (size_t) count * batch * sizeof(float2), cudaMemcpyDeviceToHost));
  return (long) count;
}

extern "C" int sdb_task_sample_zero_crossing(const sdb_complex *src, size_t n, size_t batch, int space, int amplitude,
                                             float threshold_re, float threshold_im, float zc_angle_re,
                                             float zc_angle_im, float bnor, uint8_t *sym, uint32_t *counts, size_t cap)
{
  if (!sym || !counts || cap == 0) return fail("null argument");
  if (space < SDB_SPACE_AMPLITUDE || space > SDB_SPACE_FREQUENCY) return fail("unknown decision space");
  if (!(bnor > 0.0f)) return fail("bnor must be positive");
  if (bnor > 1.0f) bnor = 1.0f;                            // WaveSampler.cpp:50-51
  DevMem s, ev, o, c;
  if (task_src_begin(s, src, n, batch)) return -1;
  const size_t pitch = (n + 15) & ~(size_t) 15;
  CK(cudaMalloc(&ev.p, pitch * batch));
  CK(cudaMalloc(&o.p, cap * batch));
  CK(cudaMalloc(&c.p, batch * sizeof(unsigned)));
  CK(cudaMemset(o.p, 0, cap * batch));
  // WaveSampler.cpp:236-241
  const float thres = amplitude ? threshold_re * threshold_re + threshold_im * threshold_im
                                : threshold_re * zc_angle_re - threshold_im * zc_angle_im;
  CK(sdb_launch_task_zero_crossing(0, s.as<float2>(), n, batch, space, amplitude ? 1 : 0, thres,
                                   make_float2(zc_angle_re, zc_angle_im), bnor, ev.as<unsigned char>(), pitch,
                                   o.as<unsigned char>(), c.as<unsigned>(), cap));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(sym, o.p, cap * batch, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(counts, c.p, batch * sizeof(unsigned), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int sdb_task_carrier_detect(const sdb_complex *src, size_t n, size_t batch, double avg_rel_bw,
                                       double dc_notch_rel_bw, float *peak)
{
  if (!peak) return fail("null argument");
  if (n > ((size_t) 1 << 20)) return fail("carrier detector: at most 2^20 samples");
  if (!(avg_rel_bw >= 0.0 && avg_rel_bw <= 1.0)) return fail("avg_rel_bw must be in [0, 1]");
  if (!(dc_notch_rel_bw >= 0.0)) dc_notch_rel_bw = 0.0;   // qBound(0., x, 1.), CarrierDetector.cpp:35
  if (dc_notch_rel_bw > 1.0) dc_notch_rel_bw = 1.0;
  DevMem s, w, buf, pk;
  if (task_src_begin(s, src, n, batch)) return -1;
  size_t alloc = 64;                                        // SPEC Y.5: transform size >= 64
  while (alloc < n) alloc <<= 1;
  std::vector<float> win;
  sdbh::window_fill(win, (unsigned) n, SDB_WINDOW_BLACKMANN_HARRIS);
  CK(cudaMalloc(&w.p, n * sizeof(float)));
  CK(cudaMemcpy(w.p, win.data(), n * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&buf.p, alloc * batch * sizeof(float2)));
  CK(cudaMalloc(&pk.p, batch * sizeof(float)));
  CK(sdb_launch_task_carrier_prep(0, s.as<float2>(), w.as<float>(), n, alloc, batch, buf.as<float2>()));
  CK(cudaDeviceSynchronize());
  // the transform is the engine's own PSD (rectangular window: the taps are already applied)
  sdb_engine_params prm; memset(&prm, 0, sizeof(prm));
  prm.n_streams = (uint32_t) batch; prm.psd_size = (uint32_t) alloc; prm.psd_window = SDB_WINDOW_NONE;
  prm.max_feed = (uint32_t) alloc;
  sdb_engine_t *e = sdb_engine_new(&prm, 1.0);
  if (!e) return -1;
  int rc = sdb_engine_commit(e);
  if (!rc) rc = sdb_engine_feed_device(e, (const sdb_complex *) buf.p, alloc, alloc);
  if (!rc) rc = sdb_engine_sync(e);
  if (!rc) {
    const int bins = (int) ((double) alloc * avg_rel_bw) + 1;
    const int skip = (int) (.5 * dc_notch_rel_bw * (double) alloc);
    cudaError_t ce = sdb_launch_task_carrier_find(0, sdb_engine_psd_device(e), alloc, batch, bins, (bins - 1) / 2, skip,
                                                  pk.as<float>());
    if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(peak, pk.p, batch * sizeof(float), cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) { g_err = std::string("carrier detector: ") + cudaGetErrorString(ce); rc = -1; }
  }
  sdb_engine_destroy(e);
  return rc;
}

extern "C" int sdb_task_decide(const sdb_complex *soft, uint8_t *sym, size_t n, int mode, unsigned bps, float min,
                               float max)
{
  if (!sym) return fail("null argument");
  if (mode < 0 || mode > 1 || bps < 1 || bps > 8 || !(max > min)) return fail("invalid decider");
  DevMem s, o;
  if (task_src_begin(s, soft, n, 1)) return -1;
  CK(cudaMalloc(&o.p, n));
  CK(sdb_launch_task_decide(0, s.as<float2>(), o.as<unsigned char>(), n, mode, min, max - min, 1 << bps));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(sym, o.p, n, cudaMemcpyDeviceToHost));
  return 0;
}

// Offline inspector over `batch` captured channel-rate buffers (what the GUI's TimeWindow / SamplerDialog
// do block-wise on the CPU, Components/TimeWindow.cpp:1571-2183): one GPU chain per buffer.
extern "C" long sdb_task_inspector(const sdb_inspector_config *cfg, const sdb_complex *src, size_t n,
                                   size_t batch, sdb_complex *soft, uint8_t *hard, uint32_t *counts, size_t cap)
{
  if (!cfg || !src || !counts || n == 0 || batch == 0) return fail("invalid argument");
  if (sdb_device_count() <= 0) return fail("no CUDA device: sigdigger_b200 has no CPU fallback");
  Channel ch; memset(&ch.p, 0, sizeof(ch.p));
  ch.center = 0; ch.size = 2; ch.width = 2; ch.halfw = 1; ch.halfsz = 1; ch.has_insp = true; ch.cfg = *cfg;
  SdbChainCfg c; std::vector<float> taps;
  if (!build_chain_cfg(ch, c, taps)) return fail("invalid inspector configuration");
  c.st_dl_off = 0; c.st_mh_off = 2 * (int) c.dl_size; c.st_mf_off = c.st_mh_off + (int) c.mh_size;
  c.st_pool = c.st_mf_off + 2 * c.mf_n;
  const size_t pool = (size_t) std::max(1, c.st_pool);
  SdbChannelDev cd; memset(&cd, 0, sizeof(cd)); cd.halfsz = 1; cd.out_off = 0;
  std::vector<SdbChainState> st(batch);
  const size_t pool_floats = ((batch + 31) / 32) * 32 * pool;
  for (size_t i = 0; i < batch; ++i) {
    memset(&st[i], 0, sizeof(SdbChainState));
    st[i].fast_level = st[i].slow_level = st[i].peak = -160.0f;
    st[i].k_phi = 0.25f; st[i].k_bnor = c.bnor; st[i].eq_wr[0] = 1.0f;
  }
  struct Bufs { void *p[9] = {0}; ~Bufs() { for (auto q : p) cudaFree(q); } } b;
  float2 *d_src, *d_soft; uint8_t *d_hard; uint32_t *d_cnt; SdbChainCfg *d_cfg; SdbChainState *d_st;
  float *d_pool, *d_taps; SdbChannelDev *d_cd;
  CK(cudaMalloc(&b.p[0], n * batch * sizeof(float2))); d_src = (float2 *) b.p[0];
  CK(cudaMalloc(&b.p[1], cap * batch * sizeof(float2))); d_soft = (float2 *) b.p[1];
  CK(cudaMalloc(&b.p[2], cap * batch)); d_hard = (uint8_t *) b.p[2];
  CK(cudaMalloc(&b.p[3], batch * sizeof(uint32_t))); d_cnt = (uint32_t *) b.p[3];
  CK(cudaMalloc(&b.p[4], sizeof(SdbChainCfg))); d_cfg = (SdbChainCfg *) b.p[4];
  CK(cudaMalloc(&b.p[5], batch * sizeof(SdbChainState))); d_st = (SdbChainState *) b.p[5];
  CK(cudaMalloc(&b.p[6], pool_floats * sizeof(float))); d_pool = (float *) b.p[6];
  CK(cudaMalloc(&b.p[7], std::max<size_t>(1, taps.size()) * sizeof(float))); d_taps = (float *) b.p[7];
  CK(cudaMalloc(&b.p[8], sizeof(SdbChannelDev))); d_cd = (SdbChannelDev *) b.p[8];
  CK(cudaMemcpy(d_src, src, n * batch * sizeof(float2), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_cfg, &c, sizeof(c), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_st, st.data(), batch * sizeof(SdbChainState), cudaMemcpyHostToDevice));
  CK(cudaMemset(d_pool, 0, pool_floats * sizeof(float)));
  if (!taps.empty()) CK(cudaMemcpy(d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_cd, &cd, sizeof(cd), cudaMemcpyHostToDevice));
  SdbLaunchCtx ctx{ 0, nullptr };
  // every chain is "stream s, channel 0"; chan_stream_stride = n
  CK(sdb_launch_inspectors_n(ctx, d_cfg, 1, (int) batch, nullptr, 0, d_st, d_pool, pool, d_taps, d_cd, d_src, n,
                             (uint32_t) n, d_soft, d_hard, d_cnt, cap, 1, sdb_insp_dyn(&c, 1)));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(counts, d_cnt, batch * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (soft) CK(cudaMemcpy(soft, d_soft, cap * batch * sizeof(float2), cudaMemcpyDeviceToHost));
  if (hard) CK(cudaMemcpy(hard, d_hard, cap * batch, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int sdb_task_lpf(const sdb_complex *src, sdb_complex *dst, size_t n, size_t batch, float bw)
{
  // LPFTask: specttuner with the default 4096-sample window, one channel at f0 = 0 with
  // guard = 2 pi / bw (no decimation), input flushed with zeros until n outputs exist
  // (Tasks/LPFTask.cpp:52-69,104-107).
  if (!src || !dst || n == 0 || batch == 0) return fail("invalid task buffer");
  const unsigned W = 4096;   // sigutils_specttuner_params_INITIALIZER default window (SURVEY.md A.2)
  sdb_engine_params p; memset(&p, 0, sizeof(p));
  size_t padded = ((n + W / 2 + W / 2 - 1) / (W / 2)) * (W / 2);   // + half-window latency, rounded up
  p.n_streams = (uint32_t) batch; p.psd_size = 0; p.st_window_size = W; p.max_feed = (uint32_t) padded; p.device = 0;
  int dev = 0; cudaGetDevice(&dev); p.device = dev;
  sdb_engine_t *e = sdb_engine_new(&p, 1.0);
  if (!e) return -1;
  sdb_channel_params cp; cp.f0 = 0.0f; cp.bw = 3.14159265358979323846f * bw; cp.guard = 6.28318530717958647692f / cp.bw;
  cp.precise = 0;
  int rc = -1;
  std::vector<float2> in(batch * padded, make_float2(0.f, 0.f)), out(padded);
  for (size_t b = 0; b < batch; ++b) memcpy(&in[b * padded], src + b * n, n * sizeof(float2));
  do {
    int h = sdb_engine_open_channel(e, &cp, nullptr);
    if (h < 0) break;
    if (sdb_engine_commit(e)) break;
    if (sdb_engine_feed_host(e, reinterpret_cast<const sdb_complex *>(in.data()), padded, padded)) break;
    bool ok = true;
    for (size_t b = 0; b < batch && ok; ++b) {
      long got = sdb_engine_read_channel(e, (uint32_t) b, h, reinterpret_cast<sdb_complex *>(out.data()), padded);
      if (got < (long) n) { g_err = "lpf produced too few samples"; ok = false; break; }
      memcpy(dst + b * n, out.data(), n * sizeof(float2));
    }
    if (ok) rc = 0;
  } while (0);
  sdb_engine_destroy(e);
  return rc;
}

// ---------------------------------------------------------------------------------------------
// SpectrumView (Panoramic/Scanner.cpp:36-293): panoramic stitcher
// ---------------------------------------------------------------------------------------------
cudaError_t sdb_launch_sview_project(cudaStream_t s, double freq_min, double freq_range, double fft_bandwidth,
                                     float rel_bw, unsigned spectrum_size, const float *psd, size_t psd_size,
                                     const double *centers_dev, int n_hops, int adjust_sides, int *j0, int *nb,
                                     float *va, float *vc, int max_bins);
cudaError_t sdb_launch_sview_accumulate(cudaStream_t s, unsigned spectrum_size, const int *j0, const int *nb,
                                        const float *va, const float *vc, int n_hops, int max_bins, float *psd,
                                        float *accum, float *count, float *count_snapshot);

struct sdb_sview {
  int device = 0;
  double freq_min = 0, freq_max = 0, freq_range = 0, fft_bandwidth = 0;
  float rel_bw = 0.5f;                     // include/Scanner.h:70
  unsigned spectrum_size = 65536;          // SIGDIGGER_SCANNER_SPECTRUM_SIZE
  int max_bins = 0;
  float *d_psd = nullptr, *d_accum = nullptr, *d_count = nullptr, *d_count_snap = nullptr;
  size_t hop_cap = 0;
  double *d_centers = nullptr; int *d_j0 = nullptr, *d_nb = nullptr; float *d_va = nullptr, *d_vc = nullptr;
};

extern "C" sdb_sview_t *sdb_sview_new(int device)
{
  if (sdb_device_count() <= 0) { g_err = "no CUDA device: sigdigger_b200 has no CPU fallback"; return nullptr; }
  CKP(cudaSetDevice(device));
  sdb_sview *v = new sdb_sview();
  v->device = device;
  const size_t n = 65536 * sizeof(float);
  if (cudaMalloc(&v->d_psd, n) != cudaSuccess || cudaMalloc(&v->d_accum, n) != cudaSuccess ||
      cudaMalloc(&v->d_count, n) != cudaSuccess || cudaMalloc(&v->d_count_snap, n) != cudaSuccess) { g_err = "out of device memory"; delete v; return nullptr; }
  cudaMemset(v->d_psd, 0, n); cudaMemset(v->d_accum, 0, n); cudaMemset(v->d_count, 0, n);
  return v;
}

extern "C" void sdb_sview_destroy(sdb_sview_t *v)
{
  if (!v) return;
  cudaSetDevice(v->device);
  cudaFree(v->d_psd); cudaFree(v->d_accum); cudaFree(v->d_count); cudaFree(v->d_count_snap); cudaFree(v->d_centers);
  cudaFree(v->d_j0); cudaFree(v->d_nb); cudaFree(v->d_va); cudaFree(v->d_vc);
  delete v;
}

extern "C" int sdb_sview_reset(sdb_sview_t *v)
{
  if (!v) return fail("null view");
  CK(cudaSetDevice(v->device));
  const size_t n = 65536 * sizeof(float);          // SpectrumView::reset, Scanner.cpp:287-293
  CK(cudaMemset(v->d_psd, 0, n)); CK(cudaMemset(v->d_accum, 0, n)); CK(cudaMemset(v->d_count, 0, n));
  return 0;
}

int sdb_sview_reset_async(sdb_sview_t *v, cudaStream_t st)     // the same, ordered on the caller's stream
{
  if (!v) return fail("null view");
  const size_t n = 65536 * sizeof(float);
  CK(cudaMemsetAsync(v->d_psd, 0, n, st)); CK(cudaMemsetAsync(v->d_accum, 0, n, st));
  CK(cudaMemsetAsync(v->d_count, 0, n, st));
  return 0;
}

extern "C" int sdb_sview_set_range(sdb_sview_t *v, double fmin, double fmax, double fft_bandwidth, float rel_bw)
{
  if (!v) return fail("null view");
  if (!(fmax > fmin) || !(fft_bandwidth > 0)) return fail("invalid frequency range");
  v->freq_min = fmin; v->freq_max = fmax; v->freq_range = fmax - fmin;   // setRange, Scanner.cpp:41-54
  unsigned n = (unsigned) (v->freq_range / 1000.0), sz = 1;               // SIGDIGGER_SCANNER_FREQ_RESOLUTION
  while (sz < n) sz <<= 1;
  if (sz > 65536) sz = 65536;
  v->spectrum_size = sz;
  v->fft_bandwidth = fft_bandwidth; v->rel_bw = rel_bw;
  // a hop contributes at most sz * (fft_bandwidth - 2 skip) / freq_range + 1 bins, and every projection uses THIS
  // fft_bandwidth (the kernels take the geometry from the view, not from the call): the `nb > max_bins` clamp in the
  // projection kernels is a guard that cannot bind
  double mb = (double) sz * fft_bandwidth / v->freq_range + 4.0;
  v->max_bins = mb > (double) sz ? (int) sz : (int) mb;
  if (v->max_bins < 2) v->max_bins = 2;
  v->hop_cap = 0;   // contribution buffers depend on max_bins: reallocate lazily
  return sdb_sview_reset(v);
}

extern "C" uint32_t sdb_sview_size(const sdb_sview_t *v) { return v ? v->spectrum_size : 0; }
extern "C" uint32_t sdb_sview_max_bins(const sdb_sview_t *v) { return v ? (uint32_t) v->max_bins : 0; }

extern "C" int sdb_sview_project(sdb_sview_t *v, const float *psd_dev, size_t psd_size, const double *centers,
                                 size_t n_hops, int adjust_sides)
{
  if (!v || !psd_dev || !centers) return fail("null argument");
  if (v->max_bins <= 0) return fail("set_range first");
  CK(cudaSetDevice(v->device));
  if (n_hops > v->hop_cap) {
    cudaFree(v->d_centers); cudaFree(v->d_j0); cudaFree(v->d_nb); cudaFree(v->d_va); cudaFree(v->d_vc);
    v->d_centers = nullptr; v->d_j0 = v->d_nb = nullptr; v->d_va = v->d_vc = nullptr;
    CK(cudaMalloc(&v->d_centers, n_hops * sizeof(double)));
    CK(cudaMalloc(&v->d_j0, n_hops * sizeof(int)));
    CK(cudaMalloc(&v->d_nb, n_hops * sizeof(int)));
    CK(cudaMalloc(&v->d_va, n_hops * (size_t) v->max_bins * sizeof(float)));
    CK(cudaMalloc(&v->d_vc, n_hops * (size_t) v->max_bins * sizeof(float)));
    v->hop_cap = n_hops;
  }
  CK(cudaMemcpy(v->d_centers, centers, n_hops * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemset(v->d_va, 0, n_hops * (size_t) v->max_bins * sizeof(float)));
  CK(cudaMemset(v->d_vc, 0, n_hops * (size_t) v->max_bins * sizeof(float)));
  CK(sdb_launch_sview_project(0, v->freq_min, v->freq_range, v->fft_bandwidth, v->rel_bw, v->spectrum_size, psd_dev,
                              psd_size, v->d_centers, (int) n_hops, adjust_sides, v->d_j0, v->d_nb, v->d_va, v->d_vc,
                              v->max_bins));
  return 0;
}

// ---- stream-ordered variants for the panoramic sweep (panoramic.cu): caller-owned device buffers, no host copies,
// ---- no default-stream work.  `centers_dev` holds the hop centres on the device.
cudaError_t sdb_launch_sview_project_tiled(cudaStream_t s, double freq_min, double freq_range, double fft_bandwidth,
                                           float rel_bw, unsigned spectrum_size, const float *psd, size_t psd_size,
                                           size_t hop_stride, int psd_is_linear, const double *centers_dev, int n_hops,
                                           int adjust_sides, int *j0, int *nb, float *va, float *vc, int max_bins);
// psd_dev: hop h's frame at psd_dev + h * hop_stride; psd_is_linear: the engine's linear natural-order PSD (the
// PSDMessage conversion happens inside the projection) instead of shifted dB.  Returns 1 when the geometry needs the
// general kernel (histogram mode or a very wide hop): the caller then converts and calls with psd_is_linear = 0.
int sdb_sview_project_async(sdb_sview_t *v, cudaStream_t st, const float *psd_dev, size_t psd_size, size_t hop_stride,
                            int psd_is_linear, const double *centers_dev, size_t n_hops, int adjust_sides, int32_t *j0,
                            int32_t *nb, float *va, float *vc)
{
  if (!v || !psd_dev || !centers_dev || !j0 || !nb || !va || !vc) return fail("null argument");
  if (v->max_bins <= 0) return fail("set_range first");
  const bool linear_mode = v->fft_bandwidth / v->freq_range * v->spectrum_size >= 2.001;  // every hop, with margin
                                                                                              // for the kernel's own test
  if (linear_mode && v->max_bins <= 384) {
    CK(sdb_launch_sview_project_tiled(st, v->freq_min, v->freq_range, v->fft_bandwidth, v->rel_bw, v->spectrum_size,
                                      psd_dev, psd_size, hop_stride, psd_is_linear, centers_dev, (int) n_hops,
                                      adjust_sides, j0, nb, va, vc, v->max_bins));
    return 0;
  }
  if (psd_is_linear || hop_stride != psd_size) return 1;
  CK(sdb_launch_sview_project(st, v->freq_min, v->freq_range, v->fft_bandwidth, v->rel_bw, v->spectrum_size, psd_dev,
                              psd_size, centers_dev, (int) n_hops, adjust_sides, j0, nb, va, vc, v->max_bins));
  return 0;
}

int sdb_sview_accumulate_async(sdb_sview_t *v, cudaStream_t st, const int32_t *j0, const int32_t *nb, const float *va,
                               const float *vc, size_t n_hops)
{
  if (!v) return fail("null view");
  CK(sdb_launch_sview_accumulate(st, v->spectrum_size, j0, nb, va, vc, (int) n_hops, v->max_bins, v->d_psd, v->d_accum,
                                 v->d_count, v->d_count_snap));
  return 0;
}

cudaError_t sdb_chdet_pack_device(sdb_chdet_t *d, double samp_rate, const double *centers_dev, sdb_detected_channel *out_dev,
                                  size_t cap, int *counts_dev, cudaStream_t stream);
// channel lists of the last feed, converted to Hz on the device (sdb_engine_read_all_channels without the host)
int sdb_engine_pack_channels_device(sdb_engine_t *e, const double *centers_dev, sdb_detected_channel *out_dev, size_t cap,
                                    int *counts_dev, cudaStream_t st)
{
  if (!e || !e->committed || !e->chdet) return fail("channel detector not enabled");
  CK(sdb_chdet_pack_device(e->chdet, e->samp_rate, centers_dev, out_dev, cap, counts_dev, st));
  return 0;
}

cudaError_t sdb_launch_psd_shift_db(cudaStream_t s, const float *lin, float *db, size_t n_frames, unsigned n);
int sdb_psd_shift_db_async(cudaStream_t st, const float *lin_dev, float *db_dev, size_t n_frames, uint32_t psd_size)
{
  if (!lin_dev || !db_dev || lin_dev == db_dev) return fail("invalid argument");
  CK(sdb_launch_psd_shift_db(st, lin_dev, db_dev, n_frames, psd_size));
  return 0;
}


extern "C" int sdb_psd_shift_db_device(const float *lin_dev, float *db_dev, size_t n_frames, uint32_t psd_size)
{
  if (!lin_dev || !db_dev) return fail("null argument");
  if (lin_dev == db_dev) return fail("in-place conversion is not supported (the halves swap)");
  if (psd_size < 2 || (psd_size & (psd_size - 1))) return fail("psd_size must be a power of two");
  CK(sdb_launch_psd_shift_db(0, lin_dev, db_dev, n_frames, psd_size));
  return 0;
}

// ---- SpectrumView::feed(SpectrumView const &) (Panoramic/Scanner.cpp:276-286; used by the zoom path of
// ---- Scanner::setViewRange, :471-479): project the other view's accumulators / counts, then the same accumulate
// ---- + interpolate pass a hop gets.
cudaError_t sdb_launch_sview_project_view(cudaStream_t s, double freq_min, double freq_range, unsigned spectrum_size,
                                          const float *src_acc, const float *src_cnt, unsigned src_size, double fmin,
                                          double fmax, int *j0, int *nb, float *va, float *vc);

extern "C" int sdb_sview_feed_view(sdb_sview_t *v, const sdb_sview_t *detail)
{
  if (!v || !detail) return fail("null view");
  if (v == detail) return fail("a view cannot be fed into itself");
  if (v->max_bins <= 0 || detail->max_bins <= 0) return fail("set_range first");
  if (v->device != detail->device) return fail("both views must live on the same device");
  CK(cudaSetDevice(v->device));
  int *j0 = nullptr, *nb = nullptr; float *va = nullptr, *vc = nullptr;
  const size_t row = 65536 * sizeof(float);
  cudaError_t e = cudaMalloc(&j0, sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&nb, sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&va, row);
  if (e == cudaSuccess) e = cudaMalloc(&vc, row);
  if (e == cudaSuccess) e = cudaMemset(j0, 0, sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(nb, 0, sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(va, 0, row);
  if (e == cudaSuccess) e = cudaMemset(vc, 0, row);
  if (e == cudaSuccess)
    e = sdb_launch_sview_project_view(0, v->freq_min, v->freq_range, v->spectrum_size, detail->d_accum, detail->d_count,
                                      detail->spectrum_size, detail->freq_min, detail->freq_max, j0, nb, va, vc);
  if (e == cudaSuccess)
    e = sdb_launch_sview_accumulate(0, v->spectrum_size, j0, nb, va, vc, 1, 65536, v->d_psd, v->d_accum, v->d_count,
                                    v->d_count_snap);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaFree(j0); cudaFree(nb); cudaFree(va); cudaFree(vc);
  if (e != cudaSuccess) return fail(std::string("sdb_sview_feed_view: ") + cudaGetErrorString(e));
  return 0;
}

// ---- SNR estimator on the inspectors' decision-space histograms (Misc/SNREstimator.cpp; SPEC Y.7)
cudaError_t sdb_launch_snr_feed(cudaStream_t s, const unsigned *history, unsigned length, unsigned n, void *states,
                                float *gaussian, float *hi, float *htilde, float *term);
struct SnrHostState { float sigma, alpha, delta; unsigned intervals; };
struct sdb_snr_estimator {
  int device = 0; unsigned n = 0, length = 0;
  std::vector<SnrHostState> st; std::vector<unsigned> bps;
  bool dirty = true;                       // host copy of the states newer than the device copy
  unsigned *d_hist = nullptr; void *d_states = nullptr; float *d_work = nullptr;   // gaussian | hi | htilde | term
};

extern "C" sdb_snr_estimator_t *sdb_snr_estimator_new(uint32_t n_estimators, uint32_t length, int device)
{
  if (sdb_device_count() <= 0) { g_err = "no CUDA device: sigdigger_b200 has no CPU fallback"; return nullptr; }
  if (n_estimators == 0 || length == 0) { g_err = "snr estimator: empty geometry"; return nullptr; }
  CKP(cudaSetDevice(device));
  sdb_snr_estimator *e = new sdb_snr_estimator();
  e->device = device; e->n = n_estimators; e->length = length;
  e->st.assign(n_estimators, SnrHostState{ 1.f / 8.f, 1.f, 0.f, 0u });   // SNR_ESTIMATOR_DEFAULT_SIGMA / _ALPHA
  e->bps.assign(n_estimators, 0u);
  const size_t tot = (size_t) n_estimators * length;
  if (cudaMalloc(&e->d_hist, tot * sizeof(unsigned)) != cudaSuccess ||
      cudaMalloc(&e->d_states, n_estimators * sizeof(SnrHostState)) != cudaSuccess ||
      cudaMalloc(&e->d_work, 4 * tot * sizeof(float)) != cudaSuccess) {
    cudaFree(e->d_hist); cudaFree(e->d_states); cudaFree(e->d_work);
    g_err = "out of device memory"; delete e; return nullptr;
  }
  cudaMemset(e->d_work, 0, 4 * tot * sizeof(float));
  return e;
}

extern "C" void sdb_snr_estimator_destroy(sdb_snr_estimator_t *e)
{
  if (!e) return;
  cudaSetDevice(e->device);
  cudaFree(e->d_hist); cudaFree(e->d_states); cudaFree(e->d_work);
  delete e;
}

static int snr_pull(sdb_snr_estimator *e)
{
  if (e->dirty) return 0;
  CK(cudaSetDevice(e->device));
  CK(cudaMemcpy(e->st.data(), e->d_states, e->n * sizeof(SnrHostState), cudaMemcpyDeviceToHost));
  return 0;
}

// setBps (SNREstimator.cpp:122-131): a change of bps restarts sigma
extern "C" int sdb_snr_estimator_set_bps(sdb_snr_estimator_t *e, uint32_t index, uint32_t bps)
{
  if (!e || index >= e->n) return fail("wrong estimator index");
  if (bps > 8) return fail("bps out of range");
  if (snr_pull(e)) return -1;
  if (e->bps[index] != bps) {                  // as the reference: setBps(0) on a fresh estimator leaves it idle
    e->bps[index] = bps; e->st[index].sigma = 1.f / 8.f; e->st[index].intervals = 1u << bps;
  }
  e->dirty = true;
  return 0;
}

extern "C" int sdb_snr_estimator_set_alpha(sdb_snr_estimator_t *e, uint32_t index, float alpha)
{
  if (!e || index >= e->n) return fail("wrong estimator index");
  if (snr_pull(e)) return -1;
  e->st[index].alpha = alpha; e->dirty = true;
  return 0;
}

extern "C" int sdb_snr_estimator_set_sigma(sdb_snr_estimator_t *e, uint32_t index, float sigma)
{
  if (!e || index >= e->n) return fail("wrong estimator index");
  if (snr_pull(e)) return -1;
  e->st[index].sigma = sigma; e->dirty = true;
  return 0;
}

// feed (SNREstimator.cpp:133-158) for every estimator: histories [n][length] counts, host memory
extern "C" int sdb_snr_estimator_feed(sdb_snr_estimator_t *e, const uint32_t *histories)
{
  if (!e || !histories) return fail("null argument");
  CK(cudaSetDevice(e->device));
  const size_t tot = (size_t) e->n * e->length;
  if (e->dirty) {
    CK(cudaMemcpy(e->d_states, e->st.data(), e->n * sizeof(SnrHostState), cudaMemcpyHostToDevice));
    e->dirty = false;
  }
  CK(cudaMemcpy(e->d_hist, histories, tot * sizeof(unsigned), cudaMemcpyHostToDevice));
  CK(sdb_launch_snr_feed(0, e->d_hist, e->length, e->n, e->d_states, e->d_work, e->d_work + tot, e->d_work + 2 * tot,
                         e->d_work + 3 * tot));
  CK(cudaDeviceSynchronize());
  return 0;
}

// getSigma / getSNR (include/SNREstimator.h:74-84) and getModel (:61-65); any pointer may be NULL
extern "C" int sdb_snr_estimator_read(sdb_snr_estimator_t *e, float *sigma, float *snr, float *model)
{
  if (!e) return fail("null argument");
  if (snr_pull(e)) return -1;
  for (unsigned i = 0; i < e->n; ++i) {
    if (sigma) sigma[i] = e->st[i].sigma;
    if (snr) snr[i] = 1.f / (e->st[i].intervals * e->st[i].sigma);
  }
  if (model) {
    const size_t tot = (size_t) e->n * e->length;
    CK(cudaSetDevice(e->device));
    CK(cudaMemcpy(model, e->d_work + tot, tot * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return 0;
}

// ---- spectrum averager (Misc/Averager.cpp:25-60)
cudaError_t sdb_launch_psd_average(cudaStream_t s, const float *psd, size_t stream_stride, unsigned frames, unsigned n,
                                   size_t n_streams, float alpha, int primed, float *last);
struct sdb_averager {
  int device = 0; unsigned n = 0; size_t n_streams = 0; float alpha = 1.0f; bool primed = false;
  float *d_last = nullptr;
};

extern "C" sdb_averager_t *sdb_averager_new(uint32_t psd_size, uint32_t n_streams, float alpha, int device)
{
  if (sdb_device_count() <= 0) { g_err = "no CUDA device: sigdigger_b200 has no CPU fallback"; return nullptr; }
  if (psd_size == 0 || n_streams == 0) { g_err = "averager: empty geometry"; return nullptr; }
  CKP(cudaSetDevice(device));
  sdb_averager *a = new sdb_averager();
  a->device = device; a->n = psd_size; a->n_streams = n_streams; a->alpha = alpha;
  if (cudaMalloc(&a->d_last, (size_t) psd_size * n_streams * sizeof(float)) != cudaSuccess) {
    g_err = "out of device memory"; delete a; return nullptr;
  }
  cudaMemset(a->d_last, 0, (size_t) psd_size * n_streams * sizeof(float));
  return a;
}

extern "C" void sdb_averager_destroy(sdb_averager_t *a)
{
  if (!a) return;
  cudaSetDevice(a->device);
  cudaFree(a->d_last);
  delete a;
}

extern "C" int sdb_averager_set_alpha(sdb_averager_t *a, float alpha)
{
  if (!a) return fail("null averager");
  a->alpha = alpha;
  return 0;
}

extern "C" int sdb_averager_reset(sdb_averager_t *a)
{
  if (!a) return fail("null averager");
  a->primed = false;
  return 0;
}

extern "C" int sdb_averager_feed_device(sdb_averager_t *a, const float *psd_dev, size_t frames, size_t stream_stride)
{
  if (!a || !psd_dev) return fail("null argument");
  if (frames == 0) return 0;
  if (stream_stride < frames * a->n && a->n_streams > 1) return fail("stream stride smaller than the frames");
  CK(cudaSetDevice(a->device));
  CK(sdb_launch_psd_average(0, psd_dev, stream_stride, (unsigned) frames, a->n, a->n_streams, a->alpha,
                            a->primed ? 1 : 0, a->d_last));
  a->primed = true;
  return 0;
}

extern "C" const float *sdb_averager_device(const sdb_averager_t *a) { return a ? a->d_last : nullptr; }

extern "C" int sdb_averager_read(sdb_averager_t *a, float *dst, size_t cap)
{
  if (!a || !dst) return fail("null argument");
  const size_t tot = (size_t) a->n * a->n_streams;
  if (cap < tot) return fail("destination too small");
  CK(cudaSetDevice(a->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(dst, a->d_last, tot * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int sdb_sview_contrib(sdb_sview_t *v, int32_t **j0, int32_t **nb, float **va, float **vc)
{
  if (!v) return fail("null view");
  if (j0) *j0 = v->d_j0;
  if (nb) *nb = v->d_nb;
  if (va) *va = v->d_va;
  if (vc) *vc = v->d_vc;
  return 0;
}

// copy the last projection's contribution lists into caller-owned DEVICE buffers (the send buffers of the
// NCCL gather): j0/nb [n_hops] int32, va/vc [n_hops][max_bins] float32
extern "C" int sdb_sview_contrib_copy(sdb_sview_t *v, int32_t *j0, int32_t *nb, float *va, float *vc, size_t n_hops)
{
  if (!v || !j0 || !nb || !va || !vc) return fail("null argument");
  if (n_hops > v->hop_cap) return fail("more hops than the last projection held");
  CK(cudaSetDevice(v->device));
  const size_t row = (size_t) v->max_bins * sizeof(float);
  CK(cudaMemcpy(j0, v->d_j0, n_hops * sizeof(int), cudaMemcpyDeviceToDevice));
  CK(cudaMemcpy(nb, v->d_nb, n_hops * sizeof(int), cudaMemcpyDeviceToDevice));
  CK(cudaMemcpy(va, v->d_va, n_hops * row, cudaMemcpyDeviceToDevice));
  CK(cudaMemcpy(vc, v->d_vc, n_hops * row, cudaMemcpyDeviceToDevice));
  return 0;
}

extern "C" int sdb_sview_accumulate(sdb_sview_t *v, const int32_t *j0, const int32_t *nb, const float *va,
                                    const float *vc, size_t n_hops)
{
  if (!v) return fail("null view");
  CK(cudaSetDevice(v->device));
  CK(sdb_launch_sview_accumulate(0, v->spectrum_size, j0, nb, va, vc, (int) n_hops, v->max_bins, v->d_psd, v->d_accum,
                                 v->d_count, v->d_count_snap));
  return 0;
}

extern "C" int sdb_sview_read(sdb_sview_t *v, float *psd, float *accum, float *count, size_t cap)
{
  if (!v) return fail("null view");
  if (cap < v->spectrum_size) return fail("destination too small");
  CK(cudaSetDevice(v->device));
  CK(cudaDeviceSynchronize());
  const size_t n = v->spectrum_size * sizeof(float);
  if (psd) CK(cudaMemcpy(psd, v->d_psd, n, cudaMemcpyDeviceToHost));
  if (accum) CK(cudaMemcpy(accum, v->d_accum, n, cudaMemcpyDeviceToHost));
  if (count) CK(cudaMemcpy(count, v->d_count, n, cudaMemcpyDeviceToHost));
  return 0;
}
