// Track features of analyze_track (tasks/analysis.py:344-365) on the device, sm_100a: librosa's beat_track tempo,
// mean RMS energy, estimate_tuning + chroma_stft mean, and the key / scale block.  oracle/track_features.py is the
// numpy restatement every value here is checked against.
//
// Tracks of any length are packed into one buffer by offsets.  All of them share one framing: n_fft 2048, hop 512,
// center=True with zero padding, T = 1 + L / 512 frames.  Kernels, in launch order:
//   tf_stft_kernel      CTA = 16 frames of one track, warp = one frame: sum of squares (rms), periodic Hann + register
//                       rFFT-2048 (fft_reg.cuh) -> power S (f32, frame-major), 128 Slaney mel dB values, the frame's
//                       dB max, and the piptrack candidates (pitch, mag) in fixed per-frame slots (ballot compaction)
//   tf_track_kernel     CTA = one track: max dB (top_db), mean energy, median of the candidate mags by radix select on
//                       their bit patterns (every mag is > 0), tuning histogram and its first argmax
//   tf_onset_kernel     warp = one frame: clipped dB differences, median of 128 by rank counting in shared memory
//   tf_tempogram_kernel CTA = 64 frames of one track: linear-ramp padded, Hann-windowed frames of 250, direct fp32
//                       autocorrelation, per-frame max normalisation, float64 partial sums per lag
//   tf_chroma_fb_kernel the track's chroma filterbank from its tuning, in float64, stored as float32
//   tf_chroma_kernel    CTA = 64 frames: fb @ S per frame, max normalisation, float64 partial sums per chroma
//   tf_finalize_kernel  CTA = one track: partials reduced in chunk order, tempo argmax in double, chroma mean, key
// No float atomics: every reduction runs in a fixed order, so a run is bit-reproducible.
#include "common.cuh"
#include "fft_reg.cuh"

#include <cfloat>
#include <cmath>
#include <memory>

namespace {

using namespace am;

constexpr int kNfft = 2048, kHop = 512, kBins = 1025, kMels = 128;
constexpr int kStftFrames = 16, kWarps = 8, kThreads = 256, kTr = 33;
constexpr int kChunk = 64;                   // frames per tempogram / chroma CTA
constexpr int kWin = 250;                    // floor(8.0 * 16000 / 512) tempogram lags
constexpr int kMinLag = 6;                   // 1875 / k < 320 BPM
constexpr int kPipLo = 20, kPipHi = 511;     // 150 <= f * 16000 / 2048 < 4000
constexpr int kSlots = 256;                  // candidate slots per frame (at most 246 local maxima in [20, 511])
constexpr int kHist = 100;

struct FeatTables {
  const float* window;    // [2048]
  const float2* fft_tw;   // [32*32]
  const float2* post_tw;  // [1024]
  const int* band;        // [3][128] start, len, offset
  const float* weights;   // [nnz]
};

struct TrackInfo {
  int T;          // frames
  int f0;         // first global frame
  int c0, nc;     // first 64-frame chunk, chunk count
  long long s0;   // first sample
  int L;          // samples
};

// -------------------------------------------------------------------------------------------- STFT pass
__global__ void __launch_bounds__(kThreads, 2)
tf_stft_kernel(const float* __restrict__ pcm, const TrackInfo* __restrict__ tracks, const int2* __restrict__ chunks,
               int nnz, FeatTables tb, float* __restrict__ S, float* __restrict__ D, float* __restrict__ dmax,
               float* __restrict__ rms, float2* __restrict__ cand, int* __restrict__ ncand) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int n_stage = (kStftFrames - 1) * kHop + kNfft;
  float* s_x = reinterpret_cast<float*>(smem_raw);       // [n_stage]
  float* s_win = s_x + n_stage;                           // [2048]
  float2* s_tw = reinterpret_cast<float2*>(s_win + kNfft);  // [1024]
  float* s_tr = reinterpret_cast<float*>(s_tw + 32 * 32);   // [8][32*33]
  float* s_wt = s_tr + kWarps * 32 * kTr;                 // [nnz]
  int* s_band = reinterpret_cast<int*>(s_wt + nnz);       // [3][128]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int2 ch = chunks[blockIdx.x];
  const TrackInfo tk = tracks[ch.x];
  const int t0 = ch.y, nf = min(kStftFrames, tk.T - t0);
  const int count = (nf - 1) * kHop + kNfft;
  const long long p0 = (long long)t0 * kHop - kNfft / 2;
  for (int i = tid; i < count; i += kThreads) {   // zero padding (pad_mode='constant') resolved here
    const long long src = p0 + i;
    s_x[i] = (src >= 0 && src < tk.L) ? __ldg(pcm + tk.s0 + src) : 0.f;
  }
  for (int i = tid; i < kNfft; i += kThreads) s_win[i] = tb.window[i];
  for (int i = tid; i < 32 * 32; i += kThreads) s_tw[i] = tb.fft_tw[i];
  for (int i = tid; i < nnz; i += kThreads) s_wt[i] = tb.weights[i];
  for (int i = tid; i < 3 * kMels; i += kThreads) s_band[i] = tb.band[i];
  __syncthreads();

  float* tr = s_tr + warp * 32 * kTr;
  for (int f = warp; f < nf; f += kWarps) {
    const long long g = (long long)tk.f0 + t0 + f;
    const float* xf0 = s_x + f * kHop;
    // ---- rms: mean of x^2 over the unwindowed frame
    float ss = 0.f;
    for (int j = 0; j < kNfft / 32; ++j) {
      const float v = xf0[lane + 32 * j];
      ss = fmaf(v, v, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) rms[g] = sqrtf(ss / (float)kNfft);

    // ---- rFFT-2048 (the layout of fft_reg.cuh)
    float re[32], im[32];
    const float2* xf = reinterpret_cast<const float2*>(xf0);
    const float2* wf = reinterpret_cast<const float2*>(s_win);
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
      const float2 x = xf[32 * n1 + lane];
      const float2 w = wf[32 * n1 + lane];
      re[n1] = x.x * w.x;
      im[n1] = x.y * w.y;
    }
    fft32(re, im);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int k1 = rev5(i);
      const float2 w = s_tw[k1 * 32 + lane];
      const float r = re[i], q = im[i];
      re[i] = fmaf(r, w.x, -q * w.y);
      im[i] = fmaf(r, w.y, q * w.x);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) tr[rev5(i) * kTr + lane] = re[i];
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) re[n2] = tr[lane * kTr + n2];
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 32; ++i) tr[rev5(i) * kTr + lane] = im[i];
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) im[n2] = tr[lane * kTr + n2];
    __syncwarp();
    fft32(re, im);
    const int partner = (32 - lane) & 31;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int k2 = rev5(i);
      float pr = __shfl_sync(0xffffffffu, re[31 - i], partner);
      float pi = __shfl_sync(0xffffffffu, im[31 - i], partner);
      if (lane == 0) {
        pr = re[rev5((32 - k2) & 31)];
        pi = im[rev5((32 - k2) & 31)];
      }
      const int k = lane + 32 * k2;
      const float2 w = __ldg(&tb.post_tw[k]);
      const float er = re[i] + pr, ei = im[i] - pi;
      const float orr = re[i] - pr, oi = im[i] + pi;
      const float xr = 0.5f * (er + fmaf(w.x, oi, w.y * orr));
      const float xi = 0.5f * (ei - fmaf(w.x, orr, -w.y * oi));
      tr[k] = fmaf(xr, xr, xi * xi);
    }
    if (lane == 0) {
      const float ny = re[0] - im[0];
      tr[1024] = ny * ny;
    }
    __syncwarp();

    // ---- S (frame-major) and the frame's max over all bins
    float* Sg = S + g * kBins;
    float mx = 0.f;
    for (int k = lane; k < kBins; k += 32) {
      const float v = tr[k];
      Sg[k] = v;
      mx = fmaxf(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));

    // ---- onset mel dB (power_to_db before the top_db clip) and its max
    float dm = -FLT_MAX;
#pragma unroll
    for (int j = 0; j < kMels / 32; ++j) {
      const int m = lane + 32 * j;
      const int st = s_band[m], len = s_band[kMels + m];
      const float* wt = s_wt + s_band[2 * kMels + m];
      float acc = 0.f;
      for (int q = 0; q < len; ++q) acc = fmaf(wt[q], tr[st + q], acc);
      const float db = 10.0f * log10f(fmaxf(acc, 1e-10f));
      D[g * kMels + m] = db;
      dm = fmaxf(dm, db);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dm = fmaxf(dm, __shfl_xor_sync(0xffffffffu, dm, o));
    if (lane == 0) dmax[g] = dm;

    // ---- piptrack candidates: local maxima of S * (S > 0.1 max) in [150, 4000) Hz, shift from the unmasked S.
    // Explicit _rn intrinsics keep numpy's float32 rounding (no FMA contraction).
    const float ref = __fmul_rn(0.1f, mx);
    int base = 0;
    for (int f0 = kPipLo; f0 <= kPipHi; f0 += 32) {
      const int fb = f0 + lane;
      bool is_c = false;
      float pitch = 0.f, mag = 0.f;
      if (fb <= kPipHi) {
        const float s0 = tr[fb - 1], s1 = tr[fb], s2 = tr[fb + 1];
        const float m0 = s0 > ref ? s0 : 0.f, m1 = s1 > ref ? s1 : 0.f, m2 = s2 > ref ? s2 : 0.f;
        is_c = (m1 > m0) && (m1 >= m2);
        if (is_c) {
          const float a = __fsub_rn(__fadd_rn(s2, s0), __fmul_rn(2.0f, s1));
          const float b = __fmul_rn(__fsub_rn(s2, s0), 0.5f);
          const float shift = fabsf(b) >= fabsf(a) ? 0.f : __fdiv_rn(-b, a);
          pitch = (float)(((double)fb + (double)shift) * (16000.0 / 2048.0));
          mag = __fadd_rn(s1, __fmul_rn(__fmul_rn(0.5f, b), shift));
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, is_c);
      if (is_c) cand[g * kSlots + base + __popc(bal & ((1u << lane) - 1u))] = make_float2(pitch, mag);
      base += __popc(bal);
    }
    if (lane == 0) ncand[g] = base;
    __syncwarp();
  }
}

// -------------------------------------------------------------------------------------------- per-track reductions
// np.linspace(-0.5, 0.5, 101)[i] = i * 0.01 + -0.5, rounded twice as numpy does (no FMA contraction)
__device__ __forceinline__ double edge_of(int i) { return i == kHist ? 0.5 : __dadd_rn(__dmul_rn((double)i, 0.01), -0.5); }

// numpy.histogram's bin of a value in [-0.5, 0.5] over linspace(-0.5, 0.5, 101) (last bin closed)
__device__ __forceinline__ int hist_bin(float r) {
  const double v = (double)r;
  int i = (int)floor((v - -0.5) * (kHist / 1.0));
  i = min(max(i, 0), kHist - 1);
  if (v < edge_of(i)) --i;
  else if (i != kHist - 1 && v >= edge_of(i + 1)) ++i;
  return min(max(i, 0), kHist - 1);
}

// k-th smallest (0-based) candidate mag of a track; mags are positive floats, so uint order is float order
__device__ unsigned radix_select(const float2* cand, const int* ncand, int f0, int T, int k, unsigned* s_hist,
                                 unsigned* s_sel) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  unsigned prefix = 0, mask = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    for (int f = warp; f < T; f += nw) {
      const int n = ncand[f0 + f];
      for (int j = lane; j < n; j += 32) {
        const unsigned u = __float_as_uint(cand[(long long)(f0 + f) * kSlots + j].y);
        if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
      }
    }
    __syncthreads();
    if (tid == 0) {
      unsigned acc = 0;
      int b = 0;
      for (; b < 255; ++b) {
        if (acc + s_hist[b] > (unsigned)k) break;
        acc += s_hist[b];
      }
      s_sel[0] = (unsigned)b;
      s_sel[1] = acc;
    }
    __syncthreads();
    prefix |= s_sel[0] << shift;
    mask |= 255u << shift;
    k -= (int)s_sel[1];
    __syncthreads();
  }
  return prefix;
}

__global__ void __launch_bounds__(1024)
tf_track_kernel(const TrackInfo* __restrict__ tracks, const float* __restrict__ dmax, const float* __restrict__ rms,
                const float2* __restrict__ cand, const int* __restrict__ ncand, float* __restrict__ t_dbmax,
                float* __restrict__ t_energy, double* __restrict__ t_tuning, int* __restrict__ t_counts,
                int* __restrict__ t_kept) {
  __shared__ unsigned s_hist[256];
  __shared__ unsigned s_sel[2];
  __shared__ double s_red[32];
  __shared__ float s_fmax[32];
  __shared__ int s_n[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const TrackInfo tk = tracks[blockIdx.x];
  const int T = tk.T;
  if (T == 0) {
    if (tid < kHist) t_counts[blockIdx.x * kHist + tid] = 0;
    if (tid == 0) {
      t_dbmax[blockIdx.x] = 0.f;
      t_energy[blockIdx.x] = 0.f;
      t_tuning[blockIdx.x] = 0.0;
      t_kept[blockIdx.x] = 0;
    }
    return;
  }
  // max dB, sum of rms (float64, fixed order), candidate count
  float m = -FLT_MAX;
  double e = 0.0;
  int n = 0;
  for (int f = tid; f < T; f += blockDim.x) {
    m = fmaxf(m, dmax[tk.f0 + f]);
    e += (double)rms[tk.f0 + f];
    n += ncand[tk.f0 + f];
  }
  e = warp_sum(e);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    n += __shfl_xor_sync(0xffffffffu, n, o);
  }
  if (lane == 0) {
    s_red[warp] = e;
    s_fmax[warp] = m;
    s_n[warp] = n;
  }
  __syncthreads();
  if (tid == 0) {
    double es = 0.0;
    float ms = -FLT_MAX;
    int ns = 0;
    for (int w = 0; w < nw; ++w) {
      es += s_red[w];
      ms = fmaxf(ms, s_fmax[w]);
      ns += s_n[w];
    }
    t_dbmax[blockIdx.x] = ms;
    t_energy[blockIdx.x] = (float)(es / T);
    s_n[0] = ns;
  }
  __syncthreads();
  const int nc = s_n[0];
  __syncthreads();
  // estimate_tuning: threshold = float32 median of the mags (0 when there are none)
  float thr = 0.f;
  if (nc > 0) {
    const unsigned lo = radix_select(cand, ncand, tk.f0, T, (nc - 1) / 2, s_hist, s_sel);
    const unsigned hi = (nc & 1) ? lo : radix_select(cand, ncand, tk.f0, T, nc / 2, s_hist, s_sel);
    thr = (nc & 1) ? __uint_as_float(lo) : __fmul_rn(__fadd_rn(__uint_as_float(lo), __uint_as_float(hi)), 0.5f);
  }
  for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  for (int f = warp; f < T; f += nw) {
    const int cnt = ncand[tk.f0 + f];
    for (int j = lane; j < cnt; j += 32) {
      const float2 c = cand[(long long)(tk.f0 + f) * kSlots + j];
      if (c.y >= thr && c.x > 0.f) {
        // 12 * log2(p / (440 / 16)) mod 1, folded to [-0.5, 0.5), in float32
        const float o = __fmul_rn(12.0f, log2f(__fdiv_rn(c.x, 27.5f)));
        float r = fmodf(o, 1.0f);
        if (r < 0.f) r += 1.0f;
        if (r >= 0.5f) r -= 1.0f;
        atomicAdd(&s_hist[hist_bin(r)], 1u);
        atomicAdd(&s_hist[255], 1u);
      }
    }
  }
  __syncthreads();
  if (tid < kHist) t_counts[blockIdx.x * kHist + tid] = (int)s_hist[tid];
  if (tid == 0) {
    int best = 0;
    for (int i = 1; i < kHist; ++i)
      if (s_hist[i] > s_hist[best]) best = i;
    const int kept = (int)s_hist[255];
    t_kept[blockIdx.x] = kept;
    t_tuning[blockIdx.x] = kept ? edge_of(best) : 0.0;
  }
}

// -------------------------------------------------------------------------------------------- onset envelope
__global__ void __launch_bounds__(kThreads)
tf_onset_kernel(const TrackInfo* __restrict__ tracks, const int2* __restrict__ chunks, const float* __restrict__ D,
                const float* __restrict__ t_dbmax, float* __restrict__ env) {
  __shared__ float s_v[kWarps][kMels];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int2 ch = chunks[blockIdx.x];
  const TrackInfo tk = tracks[ch.x];
  const float lo = __fsub_rn(t_dbmax[ch.x], 80.0f);
  const int nf = min(kStftFrames, tk.T - ch.y);
  for (int f = warp; f < nf; f += kWarps) {
    const int i = ch.y + f;
    const long long g = (long long)tk.f0 + i;
    if (i < 3) {
      if (lane == 0) env[g] = 0.f;
      continue;
    }
    const float* d1 = D + (g - 2) * kMels;   // D[:, i-2]
    const float* d0 = D + (g - 3) * kMels;   // D[:, i-3]
#pragma unroll
    for (int j = 0; j < kMels / 32; ++j) {
      const int m = lane + 32 * j;
      s_v[warp][m] = fmaxf(0.f, __fsub_rn(fmaxf(d1[m], lo), fmaxf(d0[m], lo)));
    }
    __syncwarp();
    // median of 128: the values of ranks 63 and 64 (rank = #smaller + #equal with a lower index)
    float v63 = 0.f, v64 = 0.f;
#pragma unroll
    for (int j = 0; j < kMels / 32; ++j) {
      const int m = lane + 32 * j;
      const float v = s_v[warp][m];
      int r = 0;
      for (int q = 0; q < kMels; ++q) {
        const float u = s_v[warp][q];
        r += (u < v) || (u == v && q < m);
      }
      if (r == 63) v63 = v;
      if (r == 64) v64 = v;
    }
    const unsigned b63 = __ballot_sync(0xffffffffu, v63 != 0.f), b64 = __ballot_sync(0xffffffffu, v64 != 0.f);
    // the holder of each rank is unique; a zero value needs no shuffle
    const float a = b63 ? __shfl_sync(0xffffffffu, v63, __ffs(b63) - 1) : 0.f;
    const float b = b64 ? __shfl_sync(0xffffffffu, v64, __ffs(b64) - 1) : 0.f;
    if (lane == 0) env[g] = __fmul_rn(__fadd_rn(a, b), 0.5f);
    __syncwarp();
  }
}

// -------------------------------------------------------------------------------------------- tempogram
__global__ void __launch_bounds__(kThreads)
tf_tempogram_kernel(const TrackInfo* __restrict__ tracks, const int2* __restrict__ chunks,
                    const float* __restrict__ env, const float* __restrict__ hann250, double* __restrict__ part) {
  __shared__ float s_p[kChunk + kWin];   // padded envelope [t0, t0 + nf + 249]
  __shared__ float s_w[kWin];
  __shared__ float s_x[kWin + 2];
  __shared__ float s_m[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int2 ch = chunks[blockIdx.x];
  const TrackInfo tk = tracks[ch.x];
  const int T = tk.T, t0 = ch.y, nf = min(kChunk, T - t0);
  const float* e = env + tk.f0;
  // np.pad(env, 125, mode='linear_ramp', end_values=0): the left ramp is zero (env[0] == 0); the right one descends
  // from 124/125 of env[T-1] to 0, each value float32(q * (env[T-1] / 125)) in double
  const double step = (double)e[T - 1] / 125.0;
  for (int j = tid; j < nf + kWin - 1; j += kThreads) {
    const int pj = t0 + j;   // index into the padded envelope
    float v;
    if (pj < kWin / 2) v = 0.f;
    else if (pj < kWin / 2 + T) v = e[pj - kWin / 2];
    else v = (float)((double)(124 - (pj - kWin / 2 - T)) * step);
    s_p[j] = v;
  }
  for (int j = tid; j < kWin; j += kThreads) s_w[j] = hann250[j];
  double acc = 0.0;
  for (int f = 0; f < nf; ++f) {
    __syncthreads();
    if (tid < kWin) s_x[tid] = s_p[f + tid] * s_w[tid];
    __syncthreads();
    float r = 0.f;
    if (tid < kWin)
      for (int i = 0; i + tid < kWin; ++i) r = fmaf(s_x[i], s_x[i + tid], r);
    float m = fabsf(r);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_m[warp] = m;
    __syncthreads();
    float mx = s_m[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) mx = fmaxf(mx, s_m[w]);
    acc += mx > 0.f ? (double)r / (double)mx : (double)r;
  }
  if (tid < kWin) part[(long long)blockIdx.x * kWin + tid] = acc;
}

// -------------------------------------------------------------------------------------------- chroma
// librosa.filters.chroma(sr=16000, n_fft=2048, tuning, n_chroma=12, ctroct=5, octwidth=2, norm=2, base_c=True)
__global__ void __launch_bounds__(kThreads)
tf_chroma_fb_kernel(const double* __restrict__ t_tuning, float* __restrict__ fb) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (f >= kBins) return;
  const double a440 = 440.0 * exp2(t_tuning[t] / 12.0);
  auto frq = [&](int k) { return 12.0 * log2(((double)k * (16000.0 / 2048.0)) / (a440 / 16.0)); };
  const double q1 = frq(1);
  const double fq = f == 0 ? q1 - 1.5 * 12.0 : frq(f);
  const double fq_next = frq(f + 1);
  const double width = fmax(fq_next - fq, 1.0);
  double w[12], ss = 0.0;
#pragma unroll
  for (int c = 0; c < 12; ++c) {
    double d = fq - (double)c;
    d = d + 6.0 + 120.0;
    d = fmod(d, 12.0);   // np.remainder: d > 0 here
    d -= 6.0;
    const double z = 2.0 * d / width;
    w[c] = exp(-0.5 * (z * z));
    ss += w[c] * w[c];
  }
  double len = sqrt(ss);
  if (len < DBL_MIN) len = 1.0;
  const double oct = (fq / 12.0 - 5.0) / 2.0;
  const double g = exp(-0.5 * (oct * oct));
#pragma unroll
  for (int c = 0; c < 12; ++c) fb[((long long)t * 12 + c) * kBins + f] = (float)(w[(c + 3) % 12] / len * g);
}

__global__ void __launch_bounds__(kThreads)
tf_chroma_kernel(const TrackInfo* __restrict__ tracks, const int2* __restrict__ chunks, const float* __restrict__ S,
                 const float* __restrict__ fb, double* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_fb = reinterpret_cast<float*>(smem_raw);   // [12][1025]
  __shared__ double s_acc[kWarps][12];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int2 ch = chunks[blockIdx.x];
  const TrackInfo tk = tracks[ch.x];
  const int nf = min(kChunk, tk.T - ch.y);
  const float* fbt = fb + (long long)ch.x * 12 * kBins;
  for (int i = tid; i < 12 * kBins; i += kThreads) s_fb[i] = fbt[i];
  __syncthreads();
  double acc[12];
#pragma unroll
  for (int c = 0; c < 12; ++c) acc[c] = 0.0;
  for (int f = warp; f < nf; f += kWarps) {
    const float* Sg = S + ((long long)tk.f0 + ch.y + f) * kBins;
    float v[12];
#pragma unroll
    for (int c = 0; c < 12; ++c) v[c] = 0.f;
    for (int k = lane; k < kBins; k += 32) {
      const float s = Sg[k];
#pragma unroll
      for (int c = 0; c < 12; ++c) v[c] = fmaf(s_fb[c * kBins + k], s, v[c]);
    }
    float mx = 0.f;
#pragma unroll
    for (int c = 0; c < 12; ++c) {
      v[c] = warp_sum(v[c]);
      mx = fmaxf(mx, fabsf(v[c]));
    }
    const float den = mx < FLT_MIN ? 1.f : mx;
#pragma unroll
    for (int c = 0; c < 12; ++c) acc[c] += (double)__fdiv_rn(v[c], den);
  }
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 12; ++c) s_acc[warp][c] = acc[c];
  __syncthreads();
  if (tid < 12) {
    double s = 0.0;
    for (int w = 0; w < kWarps; ++w) s += s_acc[w][tid];
    part[(long long)blockIdx.x * 12 + tid] = s;
  }
}

// -------------------------------------------------------------------------------------------- finalize
__global__ void __launch_bounds__(kThreads)
tf_finalize_kernel(const TrackInfo* __restrict__ tracks, const float* __restrict__ env,
                   const double* __restrict__ tg_part, const double* __restrict__ ch_part,
                   const float* __restrict__ t_energy, const double* __restrict__ t_tuning,
                   const int* __restrict__ t_counts, const int* __restrict__ t_kept, am_track_feat* __restrict__ out,
                   float* __restrict__ tg_out) {
  __shared__ double s_score[kThreads];
  __shared__ int s_k[kThreads];
  __shared__ int s_any;
  __shared__ float s_cm[12];
  const int tid = threadIdx.x, t = blockIdx.x;
  const TrackInfo tk = tracks[t];
  am_track_feat* o = out + t;
  if (tid == 0) s_any = 0;
  __syncthreads();
  for (int i = tid; i < tk.T; i += kThreads)
    if (env[tk.f0 + i] != 0.f) s_any = 1;
  __syncthreads();
  const bool any = s_any != 0;
  // tempogram mean per lag: chunk partials in chunk order
  double tg = 0.0;
  if (tid < kWin && tk.T > 0) {
    for (int c = 0; c < tk.nc; ++c) tg += tg_part[(long long)(tk.c0 + c) * kWin + tid];
    tg /= (double)tk.T;
  }
  if (tg_out && tid < kWin) tg_out[(long long)t * kWin + tid] = (float)tg;
  double sc = -INFINITY;
  if (tid >= kMinLag && tid < kWin) {
    const double bpm = 60.0 * 16000.0 / (512.0 * (double)tid);
    const double lp = log2(bpm) - log2(120.0);
    sc = log1p(1e6 * tg) + -0.5 * (lp * lp);
  }
  s_score[tid] = sc;
  s_k[tid] = tid;
  __syncthreads();
  for (int h = kThreads / 2; h > 0; h >>= 1) {   // argmax, first index on ties
    if (tid < h) {
      const double a = s_score[tid], b = s_score[tid + h];
      if (b > a || (b == a && s_k[tid + h] < s_k[tid])) {
        s_score[tid] = b;
        s_k[tid] = s_k[tid + h];
      }
    }
    __syncthreads();
  }
  if (tid < 12) {
    double s = 0.0;
    for (int c = 0; c < tk.nc; ++c) s += ch_part[(long long)(tk.c0 + c) * 12 + tid];
    s_cm[tid] = tk.T > 0 ? (float)(s / (double)tk.T) : 0.f;
  }
  if (tid < kHist) o->tuning_counts[tid] = t_counts[t * kHist + tid];
  __syncthreads();
  if (tid == 0) {
    const int k = s_k[0];
    o->period = any ? k : 0;
    o->tempo = any ? 60.0 * 16000.0 / (512.0 * (double)k) : 0.0;
    o->energy = t_energy[t];
    o->tuning = t_tuning[t];
    o->n_frames = tk.T;
    o->n_pitches = t_kept[t];
    // key: corrcoef(chroma_mean, roll(major, j)) for the 12 rotations, in double
    const int major[12] = {1, 0, 1, 0, 1, 1, 0, 1, 0, 1, 0, 1};
    double xm = 0.0;
    for (int c = 0; c < 12; ++c) {
      o->chroma_mean[c] = s_cm[c];
      xm += (double)s_cm[c];
    }
    xm /= 12.0;
    double sxx = 0.0;
    for (int c = 0; c < 12; ++c) sxx += ((double)s_cm[c] - xm) * ((double)s_cm[c] - xm);
    double corr[12];
    for (int j = 0; j < 12; ++j) {
      const double pm = 7.0 / 12.0;   // every rotation of the profile has seven ones
      double sxy = 0.0, spp = 0.0;
      for (int c = 0; c < 12; ++c) {
        const double p = (double)major[(c - j + 12) % 12] - pm;
        sxy += ((double)s_cm[c] - xm) * p;
        spp += p * p;
      }
      corr[j] = fmin(1.0, fmax(-1.0, sxy / (sqrt(sxx) * sqrt(spp))));   // NaN when chroma_mean is constant
    }
    // minor_profile == roll(major_profile, 3): minor[i] = corr[(i + 3) % 12]; np.argmax returns the first NaN
    auto first_argmax = [](const double* v, int rot) {
      int best = 0;
      for (int i = 0; i < 12; ++i) {
        const double x = v[(i + rot) % 12], b = v[(best + rot) % 12];
        if (isnan(b)) break;
        if (isnan(x) || x > b) best = i;
      }
      return best;
    };
    const int kmaj = first_argmax(corr, 0), kmin = first_argmax(corr, 3);
    const bool major_wins = corr[kmaj] > corr[(kmin + 3) % 12];   // the same twelve numbers: never true
    o->is_major = major_wins ? 1 : 0;
    o->key = major_wins ? kmaj : kmin;
  }
}

}  // namespace

// -------------------------------------------------------------------------------------------- handle
struct am_features {
  am::Stream stream;
  int nnz = 0;
  am::DevBuf<char> tables;
  FeatTables tb{};
  const float* hann250 = nullptr;
  // workspace, grown on demand
  am::DevBuf<float> pcm, S, D, dmax, rms, env, fb, t_dbmax, t_energy, tg_out;
  am::DevBuf<float2> cand;
  am::DevBuf<int> ncand, t_counts, t_kept;
  am::DevBuf<double> t_tuning, tg_part, ch_part;
  am::DevBuf<TrackInfo> tracks;
  am::DevBuf<int2> ch16, ch64;
  am::DevBuf<am_track_feat> out;
};

namespace {

size_t stft_smem(int nnz) {
  return ((size_t)(kStftFrames - 1) * kHop + kNfft + kNfft + 2 * 32 * 32 + (size_t)kWarps * 32 * kTr + nnz) * 4 +
         3 * kMels * 4;
}

int run(am_features* h, const float* pcm_dev, const int64_t* offsets, int n, am_track_feat* out, float* tempogram,
        cudaStream_t st) {
  std::vector<TrackInfo> tk((size_t)n);
  std::vector<int2> c16, c64;
  int F = 0;
  for (int t = 0; t < n; ++t) {
    const int64_t L = offsets[t + 1] - offsets[t];
    AM_CHECK(L >= 0 && L < ((int64_t)1 << 31), "am_features_run: track %d has %lld samples", t, (long long)L);
    TrackInfo& k = tk[(size_t)t];
    k.L = (int)L;
    k.s0 = offsets[t] - offsets[0];
    k.T = L > 0 ? 1 + (int)(L / kHop) : 0;
    k.f0 = F;
    k.c0 = (int)c64.size();
    for (int t0 = 0; t0 < k.T; t0 += kStftFrames) c16.push_back(make_int2(t, t0));
    for (int t0 = 0; t0 < k.T; t0 += kChunk) c64.push_back(make_int2(t, t0));
    k.nc = (int)c64.size() - k.c0;
    F += k.T;
  }
  const size_t nF = std::max(F, 1), n16 = std::max<size_t>(c16.size(), 1), n64 = std::max<size_t>(c64.size(), 1);
  AM_TRY(h->S.ensure(nF * kBins));
  AM_TRY(h->D.ensure(nF * kMels));
  AM_TRY(h->dmax.ensure(nF));
  AM_TRY(h->rms.ensure(nF));
  AM_TRY(h->env.ensure(nF));
  AM_TRY(h->cand.ensure(nF * kSlots));
  AM_TRY(h->ncand.ensure(nF));
  AM_TRY(h->fb.ensure((size_t)n * 12 * kBins));
  AM_TRY(h->t_dbmax.ensure(n));
  AM_TRY(h->t_energy.ensure(n));
  AM_TRY(h->t_tuning.ensure(n));
  AM_TRY(h->t_counts.ensure((size_t)n * kHist));
  AM_TRY(h->t_kept.ensure(n));
  AM_TRY(h->tg_part.ensure(n64 * kWin));
  AM_TRY(h->ch_part.ensure(n64 * 12));
  AM_TRY(h->tracks.ensure(n));
  AM_TRY(h->ch16.ensure(n16));
  AM_TRY(h->ch64.ensure(n64));
  AM_TRY(h->out.ensure(n));
  if (tempogram) AM_TRY(h->tg_out.ensure((size_t)n * kWin));
  AM_CUDA(cudaMemcpyAsync(h->tracks.p, tk.data(), tk.size() * sizeof(TrackInfo), cudaMemcpyHostToDevice, st));
  if (!c16.empty()) {
    AM_CUDA(cudaMemcpyAsync(h->ch16.p, c16.data(), c16.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
    AM_CUDA(cudaMemcpyAsync(h->ch64.p, c64.data(), c64.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
    AM_LAUNCH(tf_stft_kernel, (int)c16.size(), kThreads, stft_smem(h->nnz), st, pcm_dev, h->tracks.p, h->ch16.p,
              h->nnz, h->tb, h->S.p, h->D.p, h->dmax.p, h->rms.p, h->cand.p, h->ncand.p);
  }
  AM_LAUNCH(tf_track_kernel, n, 1024, 0, st, h->tracks.p, h->dmax.p, h->rms.p, h->cand.p, h->ncand.p, h->t_dbmax.p,
            h->t_energy.p, h->t_tuning.p, h->t_counts.p, h->t_kept.p);
  if (!c16.empty()) {
    AM_LAUNCH(tf_onset_kernel, (int)c16.size(), kThreads, 0, st, h->tracks.p, h->ch16.p, h->D.p, h->t_dbmax.p,
              h->env.p);
    AM_LAUNCH(tf_tempogram_kernel, (int)c64.size(), kThreads, 0, st, h->tracks.p, h->ch64.p, h->env.p, h->hann250,
              h->tg_part.p);
  }
  AM_LAUNCH(tf_chroma_fb_kernel, dim3(ceil_div(kBins, kThreads), n), kThreads, 0, st, h->t_tuning.p, h->fb.p);
  if (!c16.empty())
    AM_LAUNCH(tf_chroma_kernel, (int)c64.size(), kThreads, 12 * kBins * 4, st, h->tracks.p, h->ch64.p, h->S.p,
              h->fb.p, h->ch_part.p);
  AM_LAUNCH(tf_finalize_kernel, n, kThreads, 0, st, h->tracks.p, h->env.p, h->tg_part.p, h->ch_part.p,
            h->t_energy.p, h->t_tuning.p, h->t_counts.p, h->t_kept.p, h->out.p, tempogram ? h->tg_out.p : nullptr);
  AM_CUDA(cudaMemcpyAsync(out, h->out.p, (size_t)n * sizeof(am_track_feat), cudaMemcpyDeviceToHost, st));
  if (tempogram)
    AM_CUDA(cudaMemcpyAsync(tempogram, h->tg_out.p, (size_t)n * kWin * 4, cudaMemcpyDeviceToHost, st));
  AM_CUDA(cudaStreamSynchronize(st));
  return AM_OK;
}

}  // namespace

extern "C" int am_features_create(am_features** out) {
  AM_CHECK(out != nullptr, "am_features_create: out is NULL");
  *out = nullptr;
  AM_TRY(ensure_init());
  // onset mel filters: the mel plan's filterbank at (16000, 2048, 128, 0, 8000), in CSR form
  am_mel_cfg cfg{16000, kNfft, kHop, kMels, 0.f, 8000.f, 0};
  std::vector<float> dense((size_t)kMels * kBins);
  AM_TRY(am_mel_filterbank(&cfg, dense.data()));
  std::vector<int> band(3 * kMels);
  std::vector<float> wts;
  for (int m = 0; m < kMels; ++m) {
    int lo = -1, hi = -1;
    for (int k = 0; k < kBins; ++k)
      if (dense[(size_t)m * kBins + k] != 0.0f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    band[m] = lo < 0 ? 0 : lo;
    band[kMels + m] = lo < 0 ? 0 : hi - lo + 1;
    band[2 * kMels + m] = (int)wts.size();
    for (int k = 0; k < band[kMels + m]; ++k) wts.push_back(dense[(size_t)m * kBins + band[m] + k]);
  }
  std::vector<float> win(kNfft), h250(kWin);
  for (int i = 0; i < kNfft; ++i) win[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * i / kNfft));
  for (int i = 0; i < kWin; ++i) h250[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * i / kWin));
  std::vector<float2> ftw, ptw;
  fill_fft_twiddles(ftw, ptw);
  const size_t o_win = 0, o_ftw = round_up(o_win + win.size() * 4, 256), o_ptw = round_up(o_ftw + ftw.size() * 8, 256),
               o_band = round_up(o_ptw + ptw.size() * 8, 256), o_w = round_up(o_band + band.size() * 4, 256),
               o_h = round_up(o_w + wts.size() * 4, 256), total = round_up(o_h + h250.size() * 4, 256);
  std::unique_ptr<am_features> h(new am_features());
  AM_TRY(h->stream.create());
  AM_TRY(h->tables.alloc(total));
  std::vector<char> host(total, 0);
  std::memcpy(host.data() + o_win, win.data(), win.size() * 4);
  std::memcpy(host.data() + o_ftw, ftw.data(), ftw.size() * 8);
  std::memcpy(host.data() + o_ptw, ptw.data(), ptw.size() * 8);
  std::memcpy(host.data() + o_band, band.data(), band.size() * 4);
  std::memcpy(host.data() + o_w, wts.data(), wts.size() * 4);
  std::memcpy(host.data() + o_h, h250.data(), h250.size() * 4);
  AM_CUDA(cudaMemcpy(h->tables.p, host.data(), total, cudaMemcpyHostToDevice));
  char* b = h->tables.p;
  h->tb.window = reinterpret_cast<const float*>(b + o_win);
  h->tb.fft_tw = reinterpret_cast<const float2*>(b + o_ftw);
  h->tb.post_tw = reinterpret_cast<const float2*>(b + o_ptw);
  h->tb.band = reinterpret_cast<const int*>(b + o_band);
  h->tb.weights = reinterpret_cast<const float*>(b + o_w);
  h->hann250 = reinterpret_cast<const float*>(b + o_h);
  h->nnz = (int)wts.size();
  AM_CUDA(cudaFuncSetAttribute(tf_stft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stft_smem(h->nnz)));
  AM_CUDA(cudaFuncSetAttribute(tf_chroma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 12 * kBins * 4));
  *out = h.release();
  return AM_OK;
}

extern "C" void am_features_free(am_features* h) {
  if (h) {
    cudaDeviceSynchronize();
    delete h;
  }
}

extern "C" int am_features_release_workspace(am_features* h) {
  AM_CHECK(h != nullptr, "am_features_release_workspace: NULL handle");
  // am_features_run_dev may have queued work on a caller's stream: wait for the whole device
  AM_CUDA(cudaDeviceSynchronize());
  for (auto* b : {&h->pcm, &h->S, &h->D, &h->dmax, &h->rms, &h->env, &h->fb, &h->t_dbmax, &h->t_energy, &h->tg_out})
    b->release();
  h->cand.release();
  h->ncand.release();
  h->t_counts.release();
  h->t_kept.release();
  h->t_tuning.release();
  h->tg_part.release();
  h->ch_part.release();
  h->tracks.release();
  h->ch16.release();
  h->ch64.release();
  h->out.release();
  return AM_OK;
}

extern "C" int am_features_run_dev(am_features* h, const float* pcm_dev, const int64_t* offsets, int n_tracks,
                                   am_track_feat* out, float* tempogram, void* stream) {
  AM_CHECK(h && offsets && out && n_tracks >= 0, "am_features_run_dev: NULL argument");
  if (n_tracks == 0) return AM_OK;
  AM_CHECK(pcm_dev || offsets[n_tracks] == offsets[0], "am_features_run_dev: NULL pcm");
  return run(h, pcm_dev + offsets[0], offsets, n_tracks, out, tempogram, (cudaStream_t)stream);
}

extern "C" int am_features_run(am_features* h, const float* pcm, const int64_t* offsets, int n_tracks,
                               am_track_feat* out, float* tempogram) {
  AM_CHECK(h && offsets && out && n_tracks >= 0, "am_features_run: NULL argument");
  if (n_tracks == 0) return AM_OK;
  const int64_t total = offsets[n_tracks] - offsets[0];
  AM_CHECK(total >= 0 && (pcm || total == 0), "am_features_run: bad pcm buffer");
  cudaStream_t st = h->stream.s;
  AM_TRY(h->pcm.ensure((size_t)std::max<int64_t>(total, 1)));
  if (total) AM_CUDA(cudaMemcpyAsync(h->pcm.p, pcm + offsets[0], (size_t)total * 4, cudaMemcpyHostToDevice, st));
  return run(h, h->pcm.p, offsets, n_tracks, out, tempogram, st);
}
