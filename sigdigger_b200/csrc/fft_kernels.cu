// fft_kernels.cu -- cuFFT-free FFT machinery of the analyzer hot path, hand-written for sm_100a.
//
//   * block_fft_inplace: Stockham radix-4 (+ one radix-2) transform of M points held in shared
//     memory, twiddles from a correctly rounded table (W_M^i computed in double on the host).
//   * four-step N = N1 x N2 transform in two kernels:
//       pass A (k_pass_a): coalesced float2 tile loads of CW adjacent columns, optional window
//                          multiply (main PSD), N1-point column FFTs, twiddle W_N^(n2 k1), transposed
//                          coalesced store to an L2-resident scratch;
//       pass B (k_pass_b): N2-point row FFTs + fused epilogue: |X|^2/N (+ optional fft-shift and dB)
//                          for the main PSD (SURVEY.md 8a rows a2, a17), or a compacting scatter of
//                          only the bins some channel needs (su_specttuner forward side, row a4).
//   * k_small_psd: one CTA per frame for N <= 4096.
//   * k_chan_ifft: su_specttuner inverse side: gather + k*h shaping + small IFFT + sin^2
//     cross-fade with the previous half window, optional per-sample LO ("precise").
//
// Reference behaviour being replaced: su_specttuner feed (Tasks/LPFTask.cpp:52-69,83-87) and the PSD
// message payload (Suscan/Messages/PSDMessage.cpp:26-39).  Compiled with -fmad=false; the only fused operations
// are the explicit __fmaf_rn of SPEC F.1 (twiddle products, PSD power), so results are bit-identical to
// oracle/fft_spec.c.
#include "sdb_internal.h"
#include "../../include/sigdigger_b200.h"
#include "sdb_math.h"
#include "sdb_cpx.h"
#include <math_constants.h>
#include <stdlib.h>

// SPEC F.1 twiddle product: one rounded product + one fused multiply-add per component
static __device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
  return make_float2(__fmaf_rn(a.x, b.x, -(a.y * b.y)), __fmaf_rn(a.x, b.y, a.y * b.x));
}
static __device__ __forceinline__ float2 cmulc(float2 a, float2 b)  // a * conj(b)
{
  return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
static __device__ __forceinline__ float2 ldtw(const float2 *__restrict__ tw, int i)
{
  return __ldg(tw + i);
}

// ---------------------------------------------------------------------------------------------
// In-place shared-memory FFT of M = 2^logM points.  `nthr` threads (lane = 0..nthr-1) cooperate,
// nthr * BPT >= M / 4.  Every thread of the CTA must call this with the same M (CTA-wide barriers).
// DIR = -1 forward, +1 inverse (unnormalised).
// ---------------------------------------------------------------------------------------------
template <int DIR, int BPT>
static __device__ __forceinline__ void block_fft_inplace(float2 *s, const int M, const int logM,
                                                         const int lane, const int nthr,
                                                         const float2 *__restrict__ tw)
{
  const int q = M >> 2;
  int logNs = 0;
  for (; logNs + 2 <= logM; logNs += 2) {
    const int Ns = 1 << logNs;
    float2 v[BPT][4];
#pragma unroll
    for (int b = 0; b < BPT; ++b) {
      const int j = lane + b * nthr;
      if (j < q) {
#pragma unroll
        for (int t = 0; t < 4; ++t) v[b][t] = s[j + t * q];
      }
    }
    __syncthreads();
#pragma unroll
    for (int b = 0; b < BPT; ++b) {
      const int j = lane + b * nthr;
      if (j < q) {
        const int k = j & (Ns - 1);
        // packed FP32x2 arithmetic (sdb_cpx.h): the same IEEE operations per component as the scalar statement of
        // SPEC F.1 / F.2 (a complex add is one FADD2, the twiddle product one FMUL2 + one FFMA2), so the results
        // are bit-identical and the butterfly issues ~14 instead of ~34 arithmetic instructions
        if (logNs > 0) {
          const int step = M >> (logNs + 2);
          float2 w1 = ldtw(tw, k * step), w2 = ldtw(tw, 2 * k * step), w3 = ldtw(tw, 3 * k * step);
          if (DIR > 0) { w1.y = -w1.y; w2.y = -w2.y; w3.y = -w3.y; }
          v[b][1] = cmulf(v[b][1], w1);
          v[b][2] = cmulf(v[b][2], w2);
          v[b][3] = cmulf(v[b][3], w3);
        }
        const float2 a = cadd(v[b][0], v[b][2]);
        const float2 bb = csub(v[b][0], v[b][2]);
        const float2 c = cadd(v[b][1], v[b][3]);
        const float2 dd = csub(v[b][1], v[b][3]);
        // forward: d = -i * dd ; inverse: d = +i * dd
        const float2 d = DIR < 0 ? make_float2(dd.y, -dd.x) : make_float2(-dd.y, dd.x);
        const int j0 = ((j - k) << 2) + k;
        s[j0]          = cadd(a, c);
        s[j0 + Ns]     = cadd(bb, d);
        s[j0 + 2 * Ns] = csub(a, c);
        s[j0 + 3 * Ns] = csub(bb, d);
      }
    }
    __syncthreads();
  }
  if (logNs < logM) {  // one radix-2 stage with Ns = M/2: in place, butterfly j touches s[j], s[j+h]
    const int h = M >> 1;
#pragma unroll
    for (int b = 0; b < 2 * BPT; ++b) {
      const int j = lane + b * nthr;
      if (j < h) {
        float2 w = ldtw(tw, j);
        if (DIR > 0) w.y = -w.y;
        const float2 a = s[j], t = cmulf(s[j + h], w);
        s[j]     = cadd(a, t);
        s[j + h] = csub(a, t);
      }
    }
    __syncthreads();
  }
}

static inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// ---------------------------------------------------------------------------------------------
// pass A: column FFTs
// ---------------------------------------------------------------------------------------------
struct PassAK {
  SdbFourStep fs;
  SdbPassAArgs a;
  int CW, logN1, win_base;
};

__global__ void __launch_bounds__(1024) k_pass_a(const PassAK p)
{
  extern __shared__ float2 sm[];
  const int N1 = p.fs.N1, N2 = p.fs.N2, LD = N1 + 1, CW = p.CW;
  const int w = p.win_base + blockIdx.y;
  const int stream = w / p.a.windows_per_stream;
  const int j = p.a.first_window + (w - stream * p.a.windows_per_stream);
  const int col0 = blockIdx.x * CW;
  const long v0 = (long) p.a.base_off + (long) j * p.a.hop;
  const int fmt = p.a.fmt;
  const char *__restrict__ xs = reinterpret_cast<const char *>(p.a.x) + (size_t) stream * p.a.stream_stride * sdb_fmt_bytes(fmt);
  const float2 *__restrict__ hs = p.a.hist ? p.a.hist + (size_t) stream * p.a.hist_len : nullptr;
  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int total = N1 * CW;

  for (int idx = tid; idx < total; idx += nthreads) {
    const int r = idx / CW, c = idx - r * CW;
    const long vi = v0 + (long) r * N2 + col0 + c;
    float2 val = vi < p.a.hist_len ? __ldg(hs + vi) : sdb_ld_iq(xs, vi - p.a.hist_len, fmt);
    if (p.a.window) {
      const float wv = __ldg(p.a.window + r * N2 + col0 + c);
      val.x *= wv; val.y *= wv;
    }
    sm[c * LD + r] = val;
  }
  __syncthreads();
  {
    const int per = nthreads / CW;
    const int t = tid / per, lane = tid - t * per;
    block_fft_inplace<-1, 1>(sm + t * LD, N1, p.logN1, lane, per, p.fs.twN1);
  }
  float2 *__restrict__ out = p.a.scratch + (size_t) blockIdx.y * p.fs.N;
  for (int idx = tid; idx < total; idx += nthreads) {
    const int k1 = idx / CW, c = idx - k1 * CW;
    const float2 v = sm[c * LD + k1];
    const float2 tw = ldtw(p.fs.twN, (col0 + c) * k1);
    out[(size_t) k1 * N2 + col0 + c] = cmul(v, tw);
  }
}

cudaError_t sdb_launch_pass_a_range(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassAArgs &a,
                                    int win_base, int n_win)
{
  PassAK p;
  p.fs = fs; p.a = a; p.win_base = win_base;
  p.logN1 = ilog2(fs.N1);
  int cw = 4096 / fs.N1; if (cw > 16) cw = 16; if (cw > fs.N2) cw = fs.N2; if (cw < 1) cw = 1;
  p.CW = cw;
  const int threads = cw * (fs.N1 / 4);
  const size_t smem = (size_t) cw * (fs.N1 + 1) * sizeof(float2);
  static std::atomic<unsigned long long> attr_done{ 0 };   // one bit per device: function attributes are per context
  if (sdb_first_on_device(attr_done)) {
    cudaFuncSetAttribute(k_pass_a, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  }
  dim3 grid(fs.N2 / cw, n_win);
  k_pass_a<<<grid, threads, smem, c.stream>>>(p);
  if (c.launch_counter) ++*c.launch_counter;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// pass B: row FFTs + epilogue
// ---------------------------------------------------------------------------------------------
struct PassBK {
  SdbFourStep fs;
  SdbPassBArgs a;
  int RW, logN2;
};

template <int MODE>  // 0 = PSD, 1 = channeliser scatter
__global__ void __launch_bounds__(1024) k_pass_b(const PassBK p)
{
  extern __shared__ float2 sm[];
  const int N1 = p.fs.N1, N2 = p.fs.N2, N = p.fs.N, LD = N2 + 1, RW = p.RW;
  const int win = blockIdx.y;
  const int k1_0 = blockIdx.x * RW;
  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int total = RW * N2;
  const float2 *__restrict__ in = p.a.scratch + (size_t) win * N + (size_t) k1_0 * N2;

  for (int idx = tid; idx < total; idx += nthreads) {
    const int r = idx / N2, n2 = idx - r * N2;
    sm[r * LD + n2] = in[idx];
  }
  __syncthreads();
  {
    const int per = nthreads / RW;
    const int t = tid / per, lane = tid - t * per;
    block_fft_inplace<-1, 1>(sm + t * LD, N2, p.logN2, lane, per, p.fs.twN2);
  }
  if (MODE == 0) {
    float *__restrict__ psd = p.a.psd + (size_t) win * N;
    const int half = N >> 1;
    for (int idx = tid; idx < total; idx += nthreads) {
      const int k2 = idx / RW, r = idx - k2 * RW;
      const float2 X = sm[r * LD + k2];
      const int k = k1_0 + r + N1 * k2;
      float pw = __fmaf_rn(X.x, X.x, X.y * X.y) * p.a.inv_n;
      if (p.a.shift_db) {
        // Suscan/Messages/PSDMessage.cpp:32-38: swap halves, SU_POWER_DB
        pw = 10.0f * d_log10f(pw + 1e-8f);
        psd[(k + half) & (N - 1)] = pw;
      } else {
        psd[k] = pw;
      }
    }
  } else {
    float2 *__restrict__ cs = p.a.cspec + (size_t) win * p.a.n_bins;
    for (int idx = tid; idx < total; idx += nthreads) {
      const int k2 = idx / RW, r = idx - k2 * RW;
      const int k = k1_0 + r + N1 * k2;
      const int m = __ldg(p.a.binmap + k);
      if (m >= 0) cs[m] = sm[r * LD + k2];
    }
  }
}

static cudaError_t launch_pass_b(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a,
                                 int mode)
{
  PassBK p;
  p.fs = fs; p.a = a;
  p.logN2 = ilog2(fs.N2);
  int rw = 4096 / fs.N2; if (rw > 16) rw = 16; if (rw > fs.N1) rw = fs.N1; if (rw < 1) rw = 1;
  p.RW = rw;
  const int threads = rw * (fs.N2 / 4);
  const size_t smem = (size_t) rw * (fs.N2 + 1) * sizeof(float2);
  static std::atomic<unsigned long long> attr_done{ 0 };   // one bit per device: function attributes are per context
  if (sdb_first_on_device(attr_done)) {
    cudaFuncSetAttribute(k_pass_b<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(k_pass_b<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  }
  dim3 grid(fs.N1 / rw, a.n_windows);
  if (mode == 0) k_pass_b<0><<<grid, threads, smem, c.stream>>>(p);
  else           k_pass_b<1><<<grid, threads, smem, c.stream>>>(p);
  if (c.launch_counter) ++*c.launch_counter;
  return cudaGetLastError();
}

cudaError_t sdb_launch_pass_b_psd(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a)
{
  return launch_pass_b(c, fs, a, 0);
}
cudaError_t sdb_launch_pass_b_chan(const SdbLaunchCtx &c, const SdbFourStep &fs, const SdbPassBArgs &a)
{
  return launch_pass_b(c, fs, a, 1);
}

// ---------------------------------------------------------------------------------------------
// small PSD: one CTA per frame, N <= 4096
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_small_psd(int N, int logN, const float2 *__restrict__ tw,
                                                     const void *__restrict__ x, int fmt, size_t stream_stride,
                                                     int frames_per_stream, const float *__restrict__ window,
                                                     float *__restrict__ psd, int shift_db)
{
  extern __shared__ float2 sm[];
  const int f = blockIdx.x;
  const int stream = f / frames_per_stream, fr = f - stream * frames_per_stream;
  const char *__restrict__ in = reinterpret_cast<const char *>(x)
                                + ((size_t) stream * stream_stride + (size_t) fr * N) * sdb_fmt_bytes(fmt);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float2 v = sdb_ld_iq(in, i, fmt);
    if (window) { const float w = __ldg(window + i); v.x *= w; v.y *= w; }
    sm[i] = v;
  }
  __syncthreads();
  block_fft_inplace<-1, 1>(sm, N, logN, threadIdx.x, blockDim.x, tw);
  const float inv_n = 1.0f / (float) N;
  float *__restrict__ out = psd + (size_t) f * N;
  const int half = N >> 1;
  for (int k = threadIdx.x; k < N; k += blockDim.x) {
    const float2 X = sm[k];
    float pw = __fmaf_rn(X.x, X.x, X.y * X.y) * inv_n;
    if (shift_db) { pw = 10.0f * d_log10f(pw + 1e-8f); out[(k + half) & (N - 1)] = pw; }
    else out[k] = pw;
  }
}

cudaError_t sdb_launch_small_psd(const SdbLaunchCtx &c, int N, const float2 *tw, const void *x, int fmt,
                                 size_t stream_stride, int frames_per_stream, int n_streams,
                                 const float *window, float *psd, int shift_db)
{
  int threads = N / 4; if (threads < 32) threads = 32;
  k_small_psd<<<frames_per_stream * n_streams, threads, (size_t) N * sizeof(float2), c.stream>>>(
      N, ilog2(N), tw, x, fmt, stream_stride, frames_per_stream, window, psd, shift_db);
  if (c.launch_counter) ++*c.launch_counter;
  return cudaGetLastError();
}

// last `hist_len` samples of every stream (starting at sample `offset`) -> complex float32 history
__global__ void k_hist_convert(const void *__restrict__ x, int fmt, size_t stream_stride, size_t offset,
                               float2 *__restrict__ hist, int hist_len)
{
  const int s = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hist_len) return;
  const char *xs = reinterpret_cast<const char *>(x) + ((size_t) s * stream_stride + offset) * sdb_fmt_bytes(fmt);
  hist[(size_t) s * hist_len + i] = sdb_ld_iq(xs, i, fmt);
}

cudaError_t sdb_launch_hist_convert(cudaStream_t s, const void *x, int fmt, size_t stream_stride, size_t offset,
                                    float2 *hist, int hist_len, int n_streams)
{
  dim3 grid((hist_len + 255) / 256, n_streams);
  k_hist_convert<<<grid, 256, 0, s>>>(x, fmt, stream_stride, offset, hist, hist_len);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Inspector spectrum sources and baud estimators (SPEC U): one CTA per (channel, stream) works on the last
// ns channel-rate samples of the feed.  Replaces what suscan's spectsrc / estimator workers would send as
// kind=SPECTRUM / kind=ESTIMATOR inspector messages (consumers: Default/GenericInspector/GenericInspector.cpp:232-264);
// the fast autocorrelation follows Default/GenericInspector/FACTab.cpp:209-221.
// ---------------------------------------------------------------------------------------------
static __device__ __forceinline__ float2 csq(float2 a)
{
  const float m = a.x * a.y;
  return make_float2(a.x * a.x - a.y * a.y, m + m);
}
static __device__ __forceinline__ float2 spect_pre(int kind, float2 x, float2 p)
{
  switch (kind) {
    case SDB_SPECTSRC_CYCLO: return make_float2(x.x * p.x + x.y * p.y, x.y * p.x - x.x * p.y);
    case SDB_SPECTSRC_FMSPECT: {
      const float dr = x.x * p.x + x.y * p.y, di = x.y * p.x - x.x * p.y;
      return make_float2(d_atan2f(di, dr) * 0.318309886f, 0.0f);
    }
    case SDB_SPECTSRC_TIMEDIFF: return make_float2(x.x - p.x, x.y - p.y);
    case SDB_SPECTSRC_ABSTIMEDIFF: return make_float2(d_cabsf(x.x - p.x, x.y - p.y), 0.0f);
    case SDB_SPECTSRC_EXP_2: return csq(x);
    case SDB_SPECTSRC_EXP_4: return csq(csq(x));
    case SDB_SPECTSRC_EXP_8: return csq(csq(csq(x)));
    default: return x;       // PSD, FAC
  }
}

// (value, index) arg-max over the CTA, lowest index on ties; every thread gets the result
static __device__ void block_argmax(float &v, int &i, float *sv, int *si)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_down_sync(0xffffffffu, v, o);
    const int oi = __shfl_down_sync(0xffffffffu, i, o);
    if (oi >= 0 && (i < 0 || ov > v || (ov == v && oi < i))) { v = ov; i = oi; }
  }
  const int warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { sv[warp] = v; si[warp] = i; }
  __syncthreads();
  v = sv[0]; i = si[0];
  for (int w = 1; w < nw; ++w)
    if (si[w] >= 0 && (i < 0 || sv[w] > v || (sv[w] == v && si[w] < i))) { v = sv[w]; i = si[w]; }
  __syncthreads();
}

__global__ void __launch_bounds__(1024) k_spectsrc(const SdbSpectCfg *__restrict__ cfgs,
                                                    const SdbChannelDev *__restrict__ chans, int n_channels,
                                                    const float2 *__restrict__ chan_in, size_t chan_stream_stride,
                                                    uint32_t n_hops, float *__restrict__ spect,
                                                    size_t spect_stream_stride, uint32_t *__restrict__ spect_size,
                                                    float *__restrict__ est, int *__restrict__ est_valid)
{
  extern __shared__ float2 sm[];
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  const int k = blockIdx.x, st = blockIdx.y;
  const SdbSpectCfg c = cfgs[k];
  if (c.kind == 0 && c.est_mask == 0) return;
  const int ns = c.ns, half = ns >> 1, chain = st * n_channels + k;
  const uint32_t n_ch = n_hops * (uint32_t) chans[k].halfsz;
  if (n_ch < (uint32_t) ns + 1u) {             // SPEC U.1: nothing is emitted for this feed
    if (threadIdx.x == 0) {
      spect_size[chain] = 0;
      est_valid[2 * chain] = 0; est_valid[2 * chain + 1] = 0;
    }
    return;
  }
  const float2 *__restrict__ x = chan_in + (size_t) st * chan_stream_stride + chans[k].out_off + (n_ch - ns);
  const float inv_n = 1.0f / (float) ns;
  if (c.kind) {
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
      float2 v = spect_pre(c.kind, x[i], x[i - 1]);
      if (c.kind != SDB_SPECTSRC_FAC) { const float w = __ldg(c.window + i); v.x *= w; v.y *= w; }
      sm[i] = v;
    }
    __syncthreads();
    block_fft_inplace<-1, 1>(sm, ns, c.logns, threadIdx.x, blockDim.x, c.tw);
    float *__restrict__ out = spect + (size_t) st * spect_stream_stride + c.out_off;
    if (c.kind != SDB_SPECTSRC_FAC) {
      for (int i = threadIdx.x; i < ns; i += blockDim.x)
        out[i] = __fmaf_rn(sm[i].x, sm[i].x, sm[i].y * sm[i].y) * inv_n;
      if (threadIdx.x == 0) spect_size[chain] = (uint32_t) ns;
    } else {
      for (int i = threadIdx.x; i < ns; i += blockDim.x)
        sm[i] = make_float2(__fmaf_rn(sm[i].x, sm[i].x, sm[i].y * sm[i].y), 0.0f);
      __syncthreads();
      block_fft_inplace<+1, 1>(sm, ns, c.logns, threadIdx.x, blockDim.x, c.tw);
      for (int i = threadIdx.x; i < half; i += blockDim.x) out[i] = d_cabsf(sm[i].x, sm[i].y) * inv_n;
      if (threadIdx.x == 0) spect_size[chain] = (uint32_t) half;
    }
    __syncthreads();
  }
  if (c.est_mask & 2u) {      // baud-nonlinear: line of |x[n] - x[n-1]| at the symbol rate
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
      float2 v = spect_pre(SDB_SPECTSRC_ABSTIMEDIFF, x[i], x[i - 1]);
      const float w = __ldg(c.window + i);
      v.x *= w; v.y *= w;
      sm[i] = v;
    }
    __syncthreads();
    block_fft_inplace<-1, 1>(sm, ns, c.logns, threadIdx.x, blockDim.x, c.tw);
    float bv = 0.0f; int bi = -1;
    for (int i = SDB_U5_KMIN + threadIdx.x; i < half; i += blockDim.x) {
      const float v = __fmaf_rn(sm[i].x, sm[i].x, sm[i].y * sm[i].y) * inv_n;
      if (bi < 0 || v > bv) { bv = v; bi = i; }
    }
    block_argmax(bv, bi, s_v, s_i);
    if (threadIdx.x == 0) {
      const bool ok = bi >= 0 && bv > 0.0f;
      est_valid[2 * chain + 1] = ok ? 1 : 0;
      est[2 * chain + 1] = ok ? (float) bi * c.fs_ch / (float) ns : 0.0f;
    }
    __syncthreads();
  } else if (threadIdx.x == 0) est_valid[2 * chain + 1] = 0;
  if (c.est_mask & 1u) {      // baud-fac: autocorrelation of the mean-removed |x[n] - x[n-1]|
    for (int i = threadIdx.x; i < ns; i += blockDim.x) sm[i] = spect_pre(SDB_SPECTSRC_ABSTIMEDIFF, x[i], x[i - 1]);
    __syncthreads();
    block_fft_inplace<-1, 1>(sm, ns, c.logns, threadIdx.x, blockDim.x, c.tw);
    for (int i = threadIdx.x; i < ns; i += blockDim.x)
      sm[i] = make_float2(i == 0 ? 0.0f : __fmaf_rn(sm[i].x, sm[i].x, sm[i].y * sm[i].y), 0.0f);
    __syncthreads();
    block_fft_inplace<+1, 1>(sm, ns, c.logns, threadIdx.x, blockDim.x, c.tw);
    // first lag >= 1 with a negative value: arg-max of (-index) among the negative ones
    float fv = 0.0f; int fi = -1;
    for (int i = 1 + threadIdx.x; i < half; i += blockDim.x)
      if (sm[i].x < 0.0f) { fv = (float) -i; fi = i; break; }
    block_argmax(fv, fi, s_v, s_i);
    const int from = fi;
    float bv = 0.0f; int bi = -1;
    if (from >= 1) {
      for (int i = from + threadIdx.x; i < half; i += blockDim.x) {
        const float v = sm[i].x;
        if (bi < 0 || v > bv) { bv = v; bi = i; }
      }
    }
    block_argmax(bv, bi, s_v, s_i);
    // first local maximum reaching half of the largest one (every multiple of the period peaks alike)
    float pv = 0.0f; int pi = -1;
    if (from >= 1 && bi >= 0 && bv > 0.0f) {
      const float thr = 0.5f * bv;
      for (int i = from + threadIdx.x; i + 1 < half; i += blockDim.x)
        if (sm[i].x >= thr && sm[i].x >= sm[i - 1].x && sm[i].x >= sm[i + 1].x) { pv = (float) -i; pi = i; break; }
    }
    block_argmax(pv, pi, s_v, s_i);
    if (threadIdx.x == 0) {
      const bool ok = pi >= 1;
      est_valid[2 * chain] = ok ? 1 : 0;
      est[2 * chain] = ok ? c.fs_ch / (float) pi : 0.0f;
    }
  } else if (threadIdx.x == 0) est_valid[2 * chain] = 0;
}

cudaError_t sdb_launch_spectsrc(const SdbLaunchCtx &c, const SdbSpectCfg *cfg_dev, const SdbChannelDev *chans_dev,
                                int n_channels, int n_streams, int max_ns, const float2 *chan_in,
                                size_t chan_stream_stride, uint32_t n_hops, float *spect, size_t spect_stream_stride,
                                uint32_t *spect_size, float *est, int *est_valid)
{
  int threads = max_ns / 4; if (threads < 32) threads = 32;
  dim3 grid(n_channels, n_streams);
  k_spectsrc<<<grid, threads, (size_t) max_ns * sizeof(float2), c.stream>>>(
      cfg_dev, chans_dev, n_channels, chan_in, chan_stream_stride, n_hops, spect, spect_stream_stride, spect_size,
      est, est_valid);
  if (c.launch_counter) ++*c.launch_counter;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// channeliser inverse side.  One CTA per (channel, stream).  Only the cross-fade couples consecutive hops (it needs
// the second half of the previous hop's IFFT), so the CTA transforms P hops at a time -- P x size/4 threads, every
// barrier of the shared-memory transform paid once per P hops, P gathers in flight -- and cross-fades them from the
// buffers of their left neighbours; the last hop's second half is carried in shared memory (and between feeds in
// `tails`).  Round 1 ran one hop at a time with size/4 threads: 22 us per 2048-point hop against < 1 us of work.
// BPT > 1 (8192 and 16384 points, one hop per pass) carries that half window in `tails` itself: a 16384-point
// channel's transform buffer, two shared half windows and the LO phases would need 288 KB, over the 227 KB a CTA
// can have.  Each thread reads and rewrites only its own tail entries, so the global carry needs no barrier.
// The LO phase array is only present when the group has a precise channel (launcher's `any_precise`).
// ---------------------------------------------------------------------------------------------
template <int BPT>
__global__ void __launch_bounds__(1024) k_chan_ifft(const SdbChannelDev *__restrict__ chans,
                                                     const int *__restrict__ group, int n_channels,
                                                     const float2 *__restrict__ cspec, int n_bins,
                                                     int wps, int P, float2 *__restrict__ tails,
                                                     size_t tail_stream_stride, float *__restrict__ lo_phase,
                                                     float2 *__restrict__ chan_out, size_t chan_stream_stride)
{
  constexpr bool kSmemTail = BPT == 1;
  extern __shared__ float2 sm[];
  const int ci = group[blockIdx.x];
  const SdbChannelDev ch = chans[ci];
  const int s = blockIdx.y;
  const int size = ch.size, hs = ch.halfsz, hw = ch.halfw;
  float2 *bufs = sm;                                   // [P][size]
  float2 *prevb[2] = { sm + (size_t) P * size, sm + (size_t) P * size + hs };   // BPT = 1 only
  float *phase = reinterpret_cast<float *>(sm + (size_t) P * size + (kSmemTail ? 2 * hs : 0));   // [P][hs]
  const int tid = threadIdx.x;
  const int per = BPT == 1 ? (size >= 4 ? size >> 2 : 1) : (int) blockDim.x;   // threads per hop
  const int g = tid / per, l = tid - g * per;
  float2 *__restrict__ tail = tails + (size_t) s * tail_stream_stride + ch.tail_off;
  float2 *__restrict__ out = chan_out + (size_t) s * chan_stream_stride + ch.out_off;

  if (kSmemTail)
    for (int i = tid; i < hs; i += blockDim.x) prevb[0][i] = tail[i];
  float lo_phi = ch.precise ? lo_phase[(size_t) s * n_channels + ci] : 0.0f;
  int pb = 0;
  __syncthreads();

  for (int j0 = 0; j0 < wps; j0 += P) {
    const int Pg = wps - j0 < P ? wps - j0 : P;        // hops in this group
    const bool active = g < Pg;
    float2 *buf = bufs + (size_t) (active ? g : 0) * size;
    if (active) {
      const float2 *__restrict__ cs = cspec + ((size_t) s * wps + j0 + g) * n_bins;
      // zero the guard region between the two sidebands, then gather + shape the channel's bins
      for (int i = hw + l; i < size - hw; i += per) buf[i] = make_float2(0.0f, 0.0f);
      for (int i = l; i < 2 * hw; i += per) {
        const int cidx = i < ch.L1 ? ch.c1 + i : i - ch.L1;
        float2 X = __ldg(cs + cidx);
        const float w = __ldg(ch.kh + i);
        const int r = i - hw;
        X.x *= w; X.y *= w;
        buf[r >= 0 ? r : size + r] = X;
      }
    }
    if (ch.precise && tid == 0) {
      // sequential phase accumulation, exactly as the per-sample NCQO would do it
      float phi = lo_phi;
      for (int i = 0; i < Pg * hs; ++i) {
        phase[i] = phi;
        phi += ch.lo_omega;
        if (phi >= 6.28318530717958647692f) phi -= 6.28318530717958647692f;
        else if (phi < 0.0f) phi += 6.28318530717958647692f;
      }
      lo_phi = phi;
    }
    __syncthreads();
    block_fft_inplace<+1, BPT>(buf, size, ch.log2size, active ? l : size, per, ch.tw);
    if (active) {
      const float2 *pvb = g > 0 ? buf - size + hs : (kSmemTail ? prevb[pb] : tail);
      for (int i = l; i < hs; i += per) {
        const float al = __ldg(ch.xfade + i), be = __ldg(ch.xfade + i + hs);
        const float2 cu = buf[i], pv = pvb[i];
        float2 o = make_float2(al * cu.x + be * pv.x, al * cu.y + be * pv.y);
        if (ch.precise) {
          float sn, cs_;
          d_sincosf(phase[g * hs + i], &sn, &cs_);            // SPEC M.1, as the per-sample NCQO read does
          o = cmulc(o, make_float2(cs_, sn));
        }
        out[(size_t) (j0 + g) * hs + i] = o;
        if (g == Pg - 1) {
          if (kSmemTail) prevb[pb ^ 1][i] = buf[i + hs];
          else tail[i] = buf[i + hs];
        }
      }
    }
    pb ^= 1;
    __syncthreads();
  }
  if (kSmemTail)
    for (int i = tid; i < hs; i += blockDim.x) tail[i] = prevb[pb][i];
  if (ch.precise && tid == 0) lo_phase[(size_t) s * n_channels + ci] = lo_phi;
}

// ---------------------------------------------------------------------------------------------
// channeliser inverse side, sizes 512 ... 4096: the same Stockham radix-4 dataflow (SPEC F.2: levels Ns = 1, 4, 16 ...
// then one radix-2 level when log2(size) is odd, butterflies and twiddle products statement for statement those of
// block_fft_inplace, hence bit-identical), but TWO levels per trip through shared memory: a thread owns 16 points,
// runs the four level-Ns butterflies that feed the four level-4Ns butterflies in registers and writes their 16
// results.  size/16 threads per hop (1024 points: two warps), synchronised with a named barrier of their own, so a
// 256-thread CTA transforms 256/(size/16) hops side by side and only the cross-fade -- which needs the left
// neighbour's second half -- pays a CTA-wide barrier.  Against the one-level kernel above (1024-point channels):
// 3 trips instead of 5, 6 two-warp barriers instead of 10 eight-warp ones, a quarter of the index arithmetic.
// The buffers carry one float2 of padding per 16 (PADI): every access pattern of the three kinds of trip is then
// conflict-free per half-warp.
// ---------------------------------------------------------------------------------------------
#define PADI(i) ((i) + ((i) >> 4))

template <int DIR>
static __device__ __forceinline__ void r4_core(float2 &x0, float2 &x1, float2 &x2, float2 &x3)
{
  const float2 a = cadd(x0, x2), bb = csub(x0, x2), c = cadd(x1, x3), dd = csub(x1, x3);
  const float2 d = DIR < 0 ? make_float2(dd.y, -dd.x) : make_float2(-dd.y, dd.x);
  x0 = cadd(a, c); x1 = cadd(bb, d); x2 = csub(a, c); x3 = csub(bb, d);
}
template <int DIR>
static __device__ __forceinline__ float2 twd(const float2 *__restrict__ tw, int i)
{
  float2 w = __ldg(tw + i);
  if (DIR > 0) w.y = -w.y;
  return w;
}
static __device__ __forceinline__ void group_sync(int bar_id, int per)
{
  if (per <= 32) __syncwarp();
  else asm volatile("barrier.sync %0, %1;" :: "r"(bar_id), "r"(per) : "memory");
}

// s: padded buffer of M points; jb = 0 .. M/16-1 (the `per` = M/16 threads of one group); M >= 16
template <int DIR>
static __device__ __forceinline__ void group_fft16(float2 *s, const int M, const int logM, const int jb,
                                                   const int per, const int bar_id,
                                                   const float2 *__restrict__ tw)
{
  const int q = M >> 2, e = M >> 4;
  float2 v[4][4];                                      // v[u][t] = s[jb + u e + t q]
  int logNs = 0;
  for (; logNs + 4 <= logM; logNs += 4) {
    const int Ns = 1 << logNs, k = jb & (Ns - 1);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int t = 0; t < 4; ++t) v[u][t] = s[PADI(jb + u * e + t * q)];
    group_sync(bar_id, per);
    // level Ns: butterflies j = jb + u e, all with the same k (e is a multiple of Ns)
    if (logNs > 0) {
      const int step = M >> (logNs + 2);
      const float2 w1 = twd<DIR>(tw, k * step), w2 = twd<DIR>(tw, 2 * k * step), w3 = twd<DIR>(tw, 3 * k * step);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        v[u][1] = cmulf(v[u][1], w1); v[u][2] = cmulf(v[u][2], w2); v[u][3] = cmulf(v[u][3], w3);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) r4_core<DIR>(v[u][0], v[u][1], v[u][2], v[u][3]);
    // level 4 Ns: butterfly j' = 4 (jb - k) + k + t Ns takes output t of the four butterflies above (its inputs
    // j' + u q); k' = k + t Ns
    {
      const int step = M >> (logNs + 4);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int kp = (k + t * Ns) * step;
        const float2 w1 = twd<DIR>(tw, kp), w2 = twd<DIR>(tw, 2 * kp), w3 = twd<DIR>(tw, 3 * kp);
        v[1][t] = cmulf(v[1][t], w1); v[2][t] = cmulf(v[2][t], w2); v[3][t] = cmulf(v[3][t], w3);
        r4_core<DIR>(v[0][t], v[1][t], v[2][t], v[3][t]);
      }
    }
    const int base = ((jb - k) << 4) + k;
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int t = 0; t < 4; ++t) s[PADI(base + (t + 4 * u) * Ns)] = v[u][t];
    group_sync(bar_id, per);
  }
  if (logNs + 2 <= logM) {                             // one level left over: four independent butterflies
    const int Ns = 1 << logNs, step = M >> (logNs + 2);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int t = 0; t < 4; ++t) v[u][t] = s[PADI(jb + u * e + t * q)];
    group_sync(bar_id, per);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = jb + u * e, k = j & (Ns - 1);
      if (logNs > 0) {
        const float2 w1 = twd<DIR>(tw, k * step), w2 = twd<DIR>(tw, 2 * k * step), w3 = twd<DIR>(tw, 3 * k * step);
        v[u][1] = cmulf(v[u][1], w1); v[u][2] = cmulf(v[u][2], w2); v[u][3] = cmulf(v[u][3], w3);
      }
      r4_core<DIR>(v[u][0], v[u][1], v[u][2], v[u][3]);
      const int j0 = ((j - k) << 2) + k;
#pragma unroll
      for (int t = 0; t < 4; ++t) s[PADI(j0 + t * Ns)] = v[u][t];
    }
    group_sync(bar_id, per);
    logNs += 2;
  }
  if (logNs < logM) {                                  // radix-2 level, in place
    const int h = M >> 1;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int j = jb + b * e;
      const float2 w = twd<DIR>(tw, j);
      const float2 a = s[PADI(j)], t = cmulf(s[PADI(j + h)], w);
      s[PADI(j)]     = cadd(a, t);
      s[PADI(j + h)] = csub(a, t);
    }
    group_sync(bar_id, per);
  }
}

#define IFFT16_THREADS 256
// MINB = resident CTAs per SM the register allocation aims at: 3 -> 80 registers, 4 -> 64 (72 bytes of spills)
template <int MINB>
__global__ void __launch_bounds__(IFFT16_THREADS, MINB)
k_chan_ifft16(const SdbChannelDev *__restrict__ chans, const int *__restrict__ group, int n_channels,
              const float2 *__restrict__ cspec, int n_bins, int wps, int any_precise,
              float2 *__restrict__ tails, size_t tail_stream_stride, float *__restrict__ lo_phase,
              float2 *__restrict__ chan_out, size_t chan_stream_stride)
{
  extern __shared__ float2 sm[];
  const int ci = group[blockIdx.x];
  const SdbChannelDev ch = chans[ci];
  const int s = blockIdx.y;
  const int size = ch.size, hs = ch.halfsz, hw = ch.halfw;
  const int per = size >> 4, P = IFFT16_THREADS / per;  // threads per hop, hops per round
  const int padsz = size + (size >> 4);
  float2 *bufs = sm;                                    // [P][padsz]
  float2 *prevb[2] = { sm + (size_t) P * padsz, sm + (size_t) P * padsz + hs };
  float *phase = reinterpret_cast<float *>(sm + (size_t) P * padsz + 2 * hs);   // [P][hs], precise channels only
  const int tid = threadIdx.x;
  const int g = tid / per, l = tid - g * per;
  float2 *__restrict__ tail = tails + (size_t) s * tail_stream_stride + ch.tail_off;
  float2 *__restrict__ out = chan_out + (size_t) s * chan_stream_stride + ch.out_off;

  for (int i = tid; i < hs; i += IFFT16_THREADS) prevb[0][i] = tail[i];
  float lo_phi = (any_precise && ch.precise) ? lo_phase[(size_t) s * n_channels + ci] : 0.0f;
  int pb = 0;
  __syncthreads();

  for (int j0 = 0; j0 < wps; j0 += P) {
    const int Pg = wps - j0 < P ? wps - j0 : P;         // hops in this round
    const bool active = g < Pg;
    float2 *buf = bufs + (size_t) g * padsz;
    if (active) {
      const float2 *__restrict__ cs = cspec + ((size_t) s * wps + j0 + g) * n_bins;
      for (int i = hw + l; i < size - hw; i += per) buf[PADI(i)] = make_float2(0.0f, 0.0f);
#pragma unroll 4
      for (int i = l; i < 2 * hw; i += per) {
        const int cidx = i < ch.L1 ? ch.c1 + i : i - ch.L1;
        float2 X = __ldg(cs + cidx);
        const float w = __ldg(ch.kh + i);
        const int r = i - hw;
        X.x *= w; X.y *= w;
        const int o = r >= 0 ? r : size + r;
        buf[PADI(o)] = X;
      }
    }
    if (any_precise && ch.precise && tid == IFFT16_THREADS - 1) {
      // sequential phase accumulation, exactly as the per-sample NCQO would do it
      float phi = lo_phi;
      for (int i = 0; i < Pg * hs; ++i) {
        phase[i] = phi;
        phi += ch.lo_omega;
        if (phi >= 6.28318530717958647692f) phi -= 6.28318530717958647692f;
        else if (phi < 0.0f) phi += 6.28318530717958647692f;
      }
      lo_phi = phi;
    }
    if (active) {
      group_sync(1 + g, per);
      group_fft16<+1>(buf, size, ch.log2size, l, per, 1 + g, ch.tw);
    }
    __syncthreads();
    if (active) {
      const float2 *pvb = g > 0 ? buf - padsz : nullptr;
      for (int i = l; i < hs; i += per) {
        const float al = __ldg(ch.xfade + i), be = __ldg(ch.xfade + i + hs);
        const float2 cu = buf[PADI(i)], pv = g > 0 ? pvb[PADI(i + hs)] : prevb[pb][i];
        float2 o = make_float2(al * cu.x + be * pv.x, al * cu.y + be * pv.y);
        if (any_precise && ch.precise) {
          float sn, cs_;
          d_sincosf(phase[g * hs + i], &sn, &cs_);            // SPEC M.1, as the per-sample NCQO read does
          o = cmulc(o, make_float2(cs_, sn));
        }
        out[(size_t) (j0 + g) * hs + i] = o;
        if (g == Pg - 1) prevb[pb ^ 1][i] = buf[PADI(i + hs)];
      }
    }
    pb ^= 1;
    __syncthreads();
  }
  for (int i = tid; i < hs; i += IFFT16_THREADS) tail[i] = prevb[pb][i];
  if (any_precise && ch.precise && tid == IFFT16_THREADS - 1) lo_phase[(size_t) s * n_channels + ci] = lo_phi;
}

// host side: channels grouped by size so that every CTA of a launch has the right block size.  The launch shape of a
// group depends only on its size, its hops per feed and whether it holds a precise channel.
struct ChanIfftPlan { bool use16; int bpt, threads, P; size_t smem, smem_max; };

static ChanIfftPlan chan_ifft_plan(int size, int wps, int any_precise)
{
  static const int use16 = getenv("SDB_IFFT16") ? atoi(getenv("SDB_IFFT16")) : 1;
  ChanIfftPlan q{};
  const size_t phase_bytes = any_precise ? (size_t) (size / 2) * sizeof(float) : 0;   // per hop of a pass
  if (use16 && size >= 512 && size <= 4096) {
    const int per = size / 16;
    q.use16 = true; q.bpt = 1; q.threads = IFFT16_THREADS; q.P = IFFT16_THREADS / per;
    q.smem = (size_t) q.P * (size + size / 16) * sizeof(float2) + (size_t) size * sizeof(float2) + q.P * phase_bytes;
    q.smem_max = 100 * 1024;
    return q;
  }
  int bpt = 1, threads = size / 4;
  while (threads > 1024) { threads >>= 1; bpt <<= 1; }
  // hops per pass.  Measured on cfg3 (1024-point channels, 8 hops): P = 4 (1024-thread CTAs, 2 per SM) 1.21 ms
  // against 0.85 ms for P = 1 (256-thread CTAs, 8 per SM): the barriers of a big CTA cost more than the hops it
  // overlaps, so one hop per pass stays the default (SDB_IFFT_HOPS overrides for experiments).
  int P = 1;
  static const int env_hops = getenv("SDB_IFFT_HOPS") ? atoi(getenv("SDB_IFFT_HOPS")) : 1;
  if (bpt == 1 && env_hops > 1) {
    const int per = size >= 4 ? size / 4 : 1;
    P = 1024 / per;
    if (P > env_hops) P = env_hops;
    if (P > wps) P = wps;
    if ((size_t) P * size > 8192) P = (int) (8192 / size);
    if (P < 1) P = 1;
    threads = ((P * per + 31) / 32) * 32;
  } else if (bpt == 1) {
    threads = size / 4;
  }
  if (threads < 32) threads = 32;
  q.use16 = false; q.bpt = bpt; q.threads = threads; q.P = P;
  // P transform buffers, the two carried half windows when they live in shared memory (BPT = 1), the LO phases
  q.smem = (size_t) P * size * sizeof(float2) + (bpt == 1 ? (size_t) size * sizeof(float2) : 0) + P * phase_bytes;
  q.smem_max = 200 * 1024;
  return q;
}

// whether a group of `size`-point channels can be launched, for any number of hops per feed
bool sdb_chan_ifft_fits(int size, int any_precise)
{
  const ChanIfftPlan q = chan_ifft_plan(size, 1 << 30, any_precise);
  return q.smem <= q.smem_max && (q.use16 || q.bpt <= 4);
}

cudaError_t sdb_launch_chan_ifft_group(const SdbLaunchCtx &c, const SdbChannelDev *chans_dev,
                                       const int *group_dev, int group_len, int size, int n_channels,
                                       int n_streams, const float2 *cspec, int n_bins, int wps,
                                       float2 *tails, size_t tail_stream_stride, float *lo_phase,
                                       float2 *chan_out, size_t chan_stream_stride, int any_precise)
{
  static std::atomic<unsigned long long> attr_done{ 0 };   // one bit per device: function attributes are per context
  const ChanIfftPlan q = chan_ifft_plan(size, wps, any_precise);
  if (q.smem > q.smem_max) return cudaErrorInvalidValue;
  const size_t smem = q.smem;
  if (q.use16) {
    static std::atomic<unsigned long long> attr16_done{ 0 };
    static const int occ = getenv("SDB_IFFT16_OCC") ? atoi(getenv("SDB_IFFT16_OCC")) : 3;
    if (sdb_first_on_device(attr16_done)) {
      cudaFuncSetAttribute(k_chan_ifft16<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
      cudaFuncSetAttribute(k_chan_ifft16<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    }
    dim3 grid(group_len, n_streams);
    if (occ == 4)
      k_chan_ifft16<4><<<grid, IFFT16_THREADS, smem, c.stream>>>(chans_dev, group_dev, n_channels, cspec, n_bins, wps,
                                                                 any_precise, tails, tail_stream_stride, lo_phase,
                                                                 chan_out, chan_stream_stride);
    else
      k_chan_ifft16<3><<<grid, IFFT16_THREADS, smem, c.stream>>>(chans_dev, group_dev, n_channels, cspec, n_bins, wps,
                                                                 any_precise, tails, tail_stream_stride, lo_phase,
                                                                 chan_out, chan_stream_stride);
    if (c.launch_counter) ++*c.launch_counter;
    return cudaGetLastError();
  }
  if (sdb_first_on_device(attr_done)) {
    cudaFuncSetAttribute(k_chan_ifft<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(k_chan_ifft<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(k_chan_ifft<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  }
  const int bpt = q.bpt, threads = q.threads, P = q.P;
  dim3 grid(group_len, n_streams);
  if (bpt == 1)
    k_chan_ifft<1><<<grid, threads, smem, c.stream>>>(chans_dev, group_dev, n_channels, cspec, n_bins, wps, P,
                                                      tails, tail_stream_stride, lo_phase, chan_out,
                                                      chan_stream_stride);
  else if (bpt == 2)
    k_chan_ifft<2><<<grid, threads, smem, c.stream>>>(chans_dev, group_dev, n_channels, cspec, n_bins, wps, P,
                                                      tails, tail_stream_stride, lo_phase, chan_out,
                                                      chan_stream_stride);
  else if (bpt == 4)
    k_chan_ifft<4><<<grid, threads, smem, c.stream>>>(chans_dev, group_dev, n_channels, cspec, n_bins, wps, P,
                                                      tails, tail_stream_stride, lo_phase, chan_out,
                                                      chan_stream_stride);
  else
    return cudaErrorInvalidValue;
  if (c.launch_counter) ++*c.launch_counter;
  return cudaGetLastError();
}
