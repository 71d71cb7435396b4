// sdb_internal.h -- structures shared by the host runtime (engine.cu) and the kernels.
// Product code: nothing here includes or links oracle/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "sdb_iq.h"
#ifdef __cplusplus
#include <atomic>
// cudaFuncSetAttribute applies to the CURRENT device: a process that drives several GPUs (one GUI process, two
// analyzers) must set it once per device, not once per process.  Returns true the first time on each device.
static inline bool sdb_first_on_device(std::atomic<unsigned long long> &mask)
{
  int dev = 0;
  cudaGetDevice(&dev);
  const unsigned long long bit = 1ull << (dev & 63);
  return (mask.fetch_or(bit) & bit) == 0;
}
#endif

#define SDB_MAX_FIR      1024
#define SDB_MAX_IIR      5        // coefficients (order <= 4)
#define SDB_MAX_AGC_HIST 4096
#define SDB_EQ_LEN       10

// ---------------------------------------------------------------------------------------------
// FFT plan pieces (fft_kernels.cu)
// ---------------------------------------------------------------------------------------------
struct SdbFourStep {
  int N, N1, N2;            // N = N1 * N2; pass A does N1-point column FFTs, pass B N2-point row FFTs
  const float2 *twN1;       // W_N1^i, i < N1 (forward sign)
  const float2 *twN2;
  const float2 *twN;        // W_N^i, i < N
  const float2 *twPQ;       // N = 65536 / 32768: SPEC F.4 / F.5 inter-pass twiddle [k1][n2] = W_N1^(p>>8) x W_N^(p&255), p = n2 k1
};

struct SdbPassAArgs {
  const void   *x;          // new samples, stream 0, in format `fmt` (sdb_iq.h)
  int           fmt;
  size_t        stream_stride;      // in samples
  const float2 *hist;       // [S][hist_len] samples preceding x (may be null when hist_len == 0)
  int           hist_len;
  int           windows_per_stream; // windows handled per stream in this launch
  int           first_window;       // index of the first window (per stream) in this launch
  int           hop;                // samples between consecutive windows
  int           base_off;           // offset of window 0 in the virtual buffer hist ++ x
  const float  *window;             // N taps or null
  float2       *scratch;            // [launch windows][N1][N2] as [k1][n2]
};

struct SdbPassBArgs {
  const float2 *scratch;
  int           n_windows;          // windows in this launch (flattened stream-major)
  // PSD epilogue
  float        *psd;                // [n_windows][N]
  float         inv_n;
  int           shift_db;
  // channeliser epilogue
  const int    *binmap;             // N entries, compact index or -1
  float2       *cspec;              // [n_windows][n_bins]
  int           n_bins;
  unsigned      ka_mask;            // 65536 path: bit (k >> 8) & 15 set for every needed bin k (0 = all)
};

// ---------------------------------------------------------------------------------------------
// channel plan (channeliser inverse side)
// ---------------------------------------------------------------------------------------------
struct SdbChannelDev {
  int    center, size, log2size, halfw, halfsz;
  // the channel's bins are the circular range [center-halfw, center+halfw) of the N-bin spectrum;
  // in the compacted spectrum they form one run (c1, L1 entries) plus, when the range wraps past
  // bin N-1, a second run starting at compact index 0.
  int    c1, L1;
  int    precise;
  float  lo_omega;          // rad / channel sample
  const float  *kh;         // 2*halfw weights k*h, ordered from bin center-halfw upwards
  const float  *xfade;      // size cross-fade weights sin^2(pi i / size)
  const float2 *tw;         // W_size^i (forward sign; conjugated for the inverse)
  size_t out_off;           // offset (complex samples) of this channel inside one stream's channel block
  size_t out_cap;           // capacity per feed
  size_t tail_off;          // offset of this channel's halfsz-sample tail inside one stream's tail block
};

// ---------------------------------------------------------------------------------------------
// inspector chains (chain_kernels.cu). Layout mirrors SPEC.md sections A, C, G, X.
// ---------------------------------------------------------------------------------------------
struct SdbChainCfg {
  int   cls;                // SDB_INSP_*
  int   have_agc, have_costas, have_pll, have_lo, have_mf;
  int   clock_type, clock_running;
  float gain2;
  // agc
  float knee, gain_slope, fixed_gain;
  unsigned hang_max, dl_size, mh_size;
  float far_, faf, sar, saf;
  // costas / pll / lo
  int   costas_kind;
  float c_a, c_b;
  int   af_n;               // arm filter coefficient count (1 = pass-through)
  float af_b[SDB_MAX_IIR], af_a[SDB_MAX_IIR];
  float pll_alpha, pll_beta;
  float lo_omega;
  // fsk / ask
  int   fsk_quad_demod;
  float fsk_rot_re, fsk_rot_im;
  int   ask_channel;
  // matched filter
  int   mf_n;
  int   mf_off;             // offset into the taps pool
  // clock
  float clk_gain, clk_alpha, clk_beta, bnor;
  float smp_period, smp_phase0;
  // decider
  int   dec_mode, dec_intervals;
  float dec_min, dec_h;
  // audio
  int   audio_demod, audio_squelch;
  float audio_volume, dc_alpha, sq_alpha, sq_thr;
  int   alpf_n;
  float alpf_b[SDB_MAX_IIR], alpf_a[SDB_MAX_IIR];
  double rs_step;
  // CMA equaliser (SPEC E)
  int   eq_type, eq_locked;
  float eq_mu;
  // per-chain state pool sizes (in floats) so the kernel can index the pools
  int   st_dl_off, st_mh_off, st_mf_off;  // offsets inside one chain's float pool
  int   st_pool;                           // floats per chain
};

struct SdbChainState {
  // agc
  float fast_level, slow_level, peak;
  unsigned hang_n, dl_ptr, mh_ptr;
  // costas
  float c_phi, c_omega, c_lock, c_yre, c_yim;
  float afx_re[SDB_MAX_IIR], afx_im[SDB_MAX_IIR], afy_re[SDB_MAX_IIR], afy_im[SDB_MAX_IIR];
  unsigned afxp, afyp;
  // pll / lo
  float p_phi, p_omega, lo_phi;
  // fsk / fm
  float prev_re, prev_im;
  // mf
  unsigned mf_ptr;
  // clock
  float k_phi, k_bnor, k_x0r, k_x0i, k_x1r, k_x1i, k_x2r, k_x2i, k_pr, k_pi;
  int   k_half;
  float s_phase, s_pr, s_pi;
  // audio
  float dc, sq_level, rs_prev;
  float al_x[SDB_MAX_IIR], al_y[SDB_MAX_IIR];
  unsigned al_xp, al_yp;
  double rs_phase;
  int   fm_primed;
  float eq_wr[SDB_EQ_LEN], eq_wi[SDB_EQ_LEN], eq_xr[SDB_EQ_LEN], eq_xi[SDB_EQ_LEN];
};

// ---------------------------------------------------------------------------------------------
// inspector spectrum sources + baud estimators (SPEC U; kernel in fft_kernels.cu)
// ---------------------------------------------------------------------------------------------
#define SDB_U5_KMIN 8
struct SdbSpectCfg {
  int   kind;               // SDB_SPECTSRC_* (0 = none)
  int   ns, logns;          // frame size
  unsigned est_mask;        // bit i = estimator i enabled
  float fs_ch;              // channel sample rate (Hz)
  const float2 *tw;         // W_ns^i
  const float  *window;     // Blackman-Harris(ns)
  size_t out_off;           // offset (floats) of this channel's spectrum inside one stream's block
};

// plan-dependent shared-memory lines of k_inspectors (chain_kernels.cu): sized from the channel plan
#define SDB_INSP_CHUNK 16          // samples per pipeline chunk (CH in chain_kernels.cu)
#define SDB_INSP_MF_RING_MAX 209   // longest matched filter served from the shared-memory ring (256 slots)
struct SdbInspDyn {
  int rb_slots;             // carrier ring slots (power of two >= longest ring-served filter - 1 + 2 chunks)
  int mf_rows;              // tap rows [t][lane] of the longest ring-served matched filter
  int agc_rows;             // floats per chain for the AGC delay line + magnitude history
  int use_eq;               // some chain runs the CMA equaliser
  unsigned long long role_lut, part_lut;   // nibble w = role / part of warp w (0 = the kernel's default placement)
};
static inline SdbInspDyn sdb_insp_dyn(const SdbChainCfg *cfgs, int n)
{
  SdbInspDyn d = { 4 * SDB_INSP_CHUNK, 1, 8, 0, 0ull, 0ull };   // the ring holds the chunks of the carrier, demod and filter steps
  for (int k = 0; k < n; ++k) {
    const SdbChainCfg &c = cfgs[k];
    if (c.have_mf && c.mf_n <= SDB_INSP_MF_RING_MAX) {        // longer filters stay in the global pool
      int need = c.mf_n - 1 + 3 * SDB_INSP_CHUNK, slots = 4 * SDB_INSP_CHUNK;
      while (slots < need) slots <<= 1;
      if (slots > d.rb_slots) d.rb_slots = slots;
      if (c.mf_n > d.mf_rows) d.mf_rows = c.mf_n;
    }
    if (c.have_agc) {
      const int need = (int) (2 * c.dl_size + c.mh_size);
      if (need <= 160 && need > d.agc_rows) d.agc_rows = need;
    }
    if (c.eq_type == 1) d.use_eq = 1;
  }
  return d;
}

#ifdef __cplusplus
#include <vector>
#include <algorithm>
// CTA slot -> chain (channel-major index k * S + s) or -1.  A CTA holds chains of ONE inspector class so that its
// role warps do not diverge (a single source with a psk / fsk / ask mix would otherwise execute all three carrier
// stages in every warp); the classes with the longest recurrences come first so that their CTAs start first.
static inline int sdb_build_chain_map(const SdbChainCfg *cfgs, int K, int S, std::vector<int> &map)
{
  auto cost = [&](const SdbChainCfg &c) {          // rough per-sample cost order of the carrier stage
    if (c.cls == 2) return c.have_pll ? 0 : 3;     // ask (PLL: atan2 + sincos in the loop)
    if (c.cls == 0) return c.have_costas ? 1 : 3;  // psk
    if (c.cls == 3) return 2;                      // audio
    if (c.cls == 1) return 3;                      // fsk
    return 4;                                      // raw
  };
  std::vector<int> order(K);
  for (int k = 0; k < K; ++k) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
    const int ca = cost(cfgs[a]) * 8 + cfgs[a].cls, cb = cost(cfgs[b]) * 8 + cfgs[b].cls;
    return ca < cb;
  });
  map.clear();
  int prev_key = -1;
  for (int idx = 0; idx < K; ++idx) {
    const int k = order[idx];
    const int key = cost(cfgs[k]) * 8 + cfgs[k].cls;
    if (key != prev_key) while (map.size() % 32) map.push_back(-1);
    prev_key = key;
    for (int s = 0; s < S; ++s) map.push_back(k * S + s);
  }
  while (map.size() % 32) map.push_back(-1);
  return (int) (map.size() / 32);
}
#endif

// host-callable launchers ----------------------------------------------------------------------
struct SdbLaunchCtx {
  cudaStream_t stream;
  uint64_t    *launch_counter;
};

cudaError_t sdb_launch_pass_a_range(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassAArgs &a,
                                    int win_base, int n_win);
// 65536 = 256 x 256 specialisation (fft256_kernels.cu)
cudaError_t sdb_launch_cols128(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassAArgs &a, int win_base, int n_win);
cudaError_t sdb_launch_cols256(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassAArgs &a,
                               const float2 *twfine, int win_base, int n_win);
cudaError_t sdb_launch_rows256(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a, int mode);
cudaError_t sdb_launch_pass_b_psd(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a);
cudaError_t sdb_launch_pass_b_chan(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a);
cudaError_t sdb_launch_hist_convert(cudaStream_t s, const void *x, int fmt, size_t stream_stride, size_t offset,
                                    float2 *hist, int hist_len, int n_streams);
cudaError_t sdb_launch_small_psd(const SdbLaunchCtx &c, int N, const float2 *tw, const void *x, int fmt,
                                 size_t stream_stride, int frames_per_stream, int n_streams,
                                 const float *window, float *psd, int shift_db);
cudaError_t sdb_launch_chan_ifft_group(const SdbLaunchCtx &c, const SdbChannelDev *chans_dev,
                                       const int *group_dev, int group_len, int size, int n_channels,
                                       int n_streams, const float2 *cspec, int n_bins, int wps,
                                       float2 *tails, size_t tail_stream_stride, float *lo_phase,
                                       float2 *chan_out, size_t chan_stream_stride, int any_precise = 1);
bool sdb_chan_ifft_fits(int size, int any_precise);
cudaError_t sdb_launch_sym_pack(cudaStream_t stream, const uint32_t *counts, unsigned long long *offsets, size_t chains,
                                const float2 *soft, const unsigned char *hard, size_t cap, void *out_soft,
                                void *out_hard, unsigned long long cap_total, uint64_t *launch_counter);
size_t sdb_inspector_smem_bytes(const SdbInspDyn &dyn);
// chain_map / n_ctas from sdb_build_chain_map (null: identity, (chains + 31) / 32 CTAs); the pool holds
// n_ctas * 32 * pool_stride floats
cudaError_t sdb_launch_inspectors_n(const SdbLaunchCtx &c, const SdbChainCfg *cfg_dev, int n_channels,
                                    int n_streams, const int *chain_map, int n_ctas, SdbChainState *state,
                                    float *pool, size_t pool_stride,
                                    const float *taps_pool, const SdbChannelDev *chans_dev,
                                    const float2 *chan_in, size_t chan_stream_stride, uint32_t n_hops,
                                    float2 *soft, uint8_t *hard, uint32_t *sym_counts, size_t sym_cap,
                                    int fresh, const SdbInspDyn &dyn);
cudaError_t sdb_launch_spectsrc(const SdbLaunchCtx &c, const SdbSpectCfg *cfg_dev, const SdbChannelDev *chans_dev,
                                int n_channels, int n_streams, int max_ns, const float2 *chan_in,
                                size_t chan_stream_stride, uint32_t n_hops, float *spect, size_t spect_stream_stride,
                                uint32_t *spect_size, float *est, int *est_valid);
cudaError_t sdb_launch_task_xlate(cudaStream_t s, const float2 *src, float2 *dst, size_t n, size_t batch,
                                  float omega, float phi0);
cudaError_t sdb_launch_task_chain_state(cudaStream_t s, const float2 *src, float2 *dst, size_t n, int mode, float *st);
size_t sdb_costas_k_bytes(void);
size_t sdb_costas_s_bytes(void);
cudaError_t sdb_launch_task_quad(cudaStream_t s, const float2 *src, float2 *dst, size_t n, size_t batch);
cudaError_t sdb_launch_task_chain(cudaStream_t s, const float2 *src, float2 *dst, size_t n, size_t batch,
                                  const SdbChainCfg *cfg_dev, int mode, float *pool, size_t pool_stride);
// tasks_kernels.cu (SPEC Y)
cudaError_t sdb_launch_task_delayed_conj(cudaStream_t s, const float2 *src, float2 *dst, size_t n, size_t batch,
                                         size_t delay);
cudaError_t sdb_launch_task_hist(cudaStream_t s, const float2 *src, float *out, size_t n, size_t batch, int space);
cudaError_t sdb_launch_task_sample_manual(cudaStream_t s, const float2 *src, size_t n, size_t batch, int space,
                                          double sync, double delta, double samp_offset, float delta_inv,
                                          long long count, float2 *out);
cudaError_t sdb_launch_task_zero_crossing(cudaStream_t s, const float2 *src, size_t n, size_t batch, int space,
                                          int amplitude, float thres, float2 zca, float bnor, unsigned char *ev,
                                          size_t ev_pitch, unsigned char *sym, unsigned *counts, size_t cap);
cudaError_t sdb_launch_task_carrier_prep(cudaStream_t s, const float2 *src, const float *w, size_t n, size_t alloc,
                                         size_t batch, float2 *dst);
cudaError_t sdb_launch_task_carrier_find(cudaStream_t s, const float *psd, size_t alloc, size_t batch, int bins,
                                         int delta, int skip, float *peak);
cudaError_t sdb_launch_dc_remove(cudaStream_t st, const void *x, int fmt, size_t stream_stride, size_t n, int n_streams,
                                 float alpha, float2 *state, float2 *cur, double2 *part, float2 *out);
cudaError_t sdb_launch_task_decide(cudaStream_t s, const float2 *x, unsigned char *sym, size_t n, int mode, float dmin,
                                   float dh, int intervals);
