// K1: fused  frame -> Hann window -> rFFT-2048 -> |.|^2 -> sparse mel -> 10*log10  (sm_100a)
//
// Replaces librosa.feature.melspectrogram + power_to_db as called from
// tasks/clap_analyzer.py:438-454.  One HBM pass: PCM in (int16 or f32), log-mel out.
//
// Work decomposition
//   grid = (ceil(T / 16), B); a CTA (8 warps) owns 16 consecutive frames of one 10 s window.
//   The (16-1)*hop + 2048 samples those frames cover are staged ONCE in shared memory
//   (frames overlap 4.27x at hop 480), reflect padding resolved at staging time.
//   One warp computes one frame at a time, entirely in registers + one 32x33 smem transpose:
//     2048 real samples -> 1024-point complex FFT as 32 x 32 (each lane does two radix-2
//     32-point FFTs in registers, twiddles from a conflict-free smem table) -> real-FFT
//     split (partner bins via warp shuffle) -> |X|^2 -> triangular mel filters in CSR form
//     (each lane owns bands lane, lane+32, ...) -> dB.
//   The 16 x n_mels tile is staged in smem and written with 64-byte row segments.
//
// Algorithmic traffic per 10 s window: 480000*2 B (PCM16) or *4 B (f32) in, 128*1001*4 B out.
#include "common.cuh"
#include "fft_reg.cuh"

#include <cmath>

namespace am {

constexpr int kNfft = 2048;
constexpr int kNc = 1024;       // complex FFT length
constexpr int kFramesPerCta = 16;
constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kTrStride = 33;   // padded row stride of the per-warp transpose buffer

struct MelTables {
  float* window;      // [2048]
  float2* fft_tw;     // [32*32]  fft_tw[k1*32 + n2] = W_1024^(n2*k1)
  float2* post_tw;    // [1024]   W_2048^k
  int* band_start;    // [n_mels] first FFT bin with non-zero weight
  int* band_len;      // [n_mels]
  int* band_off;      // [n_mels] offset into weights
  float* weights;     // [nnz]
};

}  // namespace am

struct am_mel_plan {
  am_mel_cfg cfg;
  int center = 1;    // 1: librosa center=True (reflect pad n_fft/2); 0: frame t starts at t * hop
  int log_mode = 0;  // 0: 10 log10(max(1e-10, .)) (power_to_db); 1: log10(1 + 10000 .) (tasks/analysis.py:374)
  am::MelTables t;
  int max_bin;   // highest FFT bin with non-zero mel weight
  int nnz;
  am::DevBuf<char> storage;
};

namespace am {

// ---------------------------------------------------------------- host: tables
static double hz_to_mel(double f) {
  const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = 1000.0 / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz(double m) {
  const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = 1000.0 / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

// Slaney-scale, slaney-normalised triangular filterbank with librosa.filters.mel's dtype
// discipline (float64 ramps, float32 storage, float32 *= float64 normalisation).
int build_filterbank(const am_mel_cfg& c, std::vector<float>& w /* [n_mels * bins] */) {
  AM_CHECK(c.n_mels > 0 && c.n_fft > 0 && c.sr > 0, "mel cfg: non-positive size");
  const int bins = c.n_fft / 2 + 1;
  const double fmax = c.fmax > 0 ? (double)c.fmax : c.sr / 2.0;
  AM_CHECK(fmax > c.fmin && fmax <= c.sr / 2.0 + 1e-6, "mel cfg: need fmin < fmax <= sr/2");
  const int n = c.n_mels + 2;
  std::vector<double> mel_f(n);
  const double m0 = hz_to_mel(c.fmin), m1 = hz_to_mel(fmax);
  for (int i = 0; i < n; ++i) {
    // np.linspace: start + i*step, last point exactly stop
    double m = (i == n - 1) ? m1 : m0 + (m1 - m0) / (double)(n - 1) * i;
    mel_f[i] = mel_to_hz(m);
  }
  const double val = 1.0 / (c.n_fft * (1.0 / c.sr));  // np.fft.rfftfreq
  w.assign((size_t)c.n_mels * bins, 0.0f);
  for (int i = 0; i < c.n_mels; ++i) {
    const double fd0 = mel_f[i + 1] - mel_f[i], fd1 = mel_f[i + 2] - mel_f[i + 1];
    const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
    for (int k = 0; k < bins; ++k) {
      const double f = k * val;
      const double lower = -(mel_f[i] - f) / fd0;
      const double upper = (mel_f[i + 2] - f) / fd1;
      const float tri = (float)std::fmax(0.0, std::fmin(lower, upper));
      w[(size_t)i * bins + k] = (float)((double)tri * enorm);
    }
  }
  return AM_OK;
}

// ---------------------------------------------------------------- device: kernel
// (q / 32767.0).astype(float32), tasks/clap_analyzer.py:505, without a division: r0 = x * (1/32767), one FMA
// for the residual, one for the correction.  Equal to the reference's value (float64 quotient cast to float32)
// for ALL 65 536 int16 inputs -- checked exhaustively (tests/test_oracle_golden.py::test_pcm16_scaling_sequence,
// tests/test_gpu_mel.py::test_int16_input_path_equals_float_path); 3 instructions instead of ~10.
__device__ __forceinline__ float pcm16_to_f32(short q) {
  constexpr float kInv = 1.0f / 32767.0f;
  const float x = (float)q;
  const float r0 = __fmul_rn(x, kInv);
  const float e = __fmaf_rn(-32767.0f, r0, x);
  return __fmaf_rn(e, kInv, r0);
}

template <bool kI16>
__device__ __forceinline__ float load_sample(const void* pcm, long long i) {
  if constexpr (kI16) {
    return pcm16_to_f32(((const short*)pcm)[i]);
  } else {
    return ((const float*)pcm)[i];
  }
}

// kK2: number of 32-bin groups of the spectrum that carry mel weight (compile time, so the warp
// shuffles of the real-FFT split sit in straight-line code): 19 for fmax = 14 kHz, 32 = all.
template <bool kI16, int kK2>
__global__ void __launch_bounds__(kThreads, 2)
mel_kernel(const void* __restrict__ pcm, int n_samples, int hop, int T, int n_mels, int max_bin,
           int transpose, int frame_len, int bin_shift, int nnz, int center, int log_mode, MelTables tb,
           float* __restrict__ out) {
  // frame_len = cfg.n_fft in {2048, 1024, 512}.  Shorter frames are transformed as 2048-point frames whose tail
  // is zero (the window table is zero there): X_2048[k << bin_shift] == X_nfft[k] exactly, so the mel filters
  // read every (1 << bin_shift)-th bin.  max_bin is in 2048-point bins.
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n_stage = (kFramesPerCta - 1) * hop + kNfft;
  float* s_x = reinterpret_cast<float*>(smem_raw);                        // [n_stage] (even count)
  float* s_win = s_x + ((n_stage + 3) & ~3);                              // [2048]
  float2* s_tw = reinterpret_cast<float2*>(s_win + kNfft);                // [1024]
  float* s_tr = reinterpret_cast<float*>(s_tw + 32 * 32);                 // [8][32*33]
  float* s_out = s_tr + kWarps * 32 * kTrStride;                          // [n_mels][17]
  // mel filters in CSR form, staged per CTA: every lane walks a different band, so from global memory each
  // weight load touched 32 sectors (12 % of the kernel's stall samples sat on them)
  float* s_wt = s_out + n_mels * (kFramesPerCta + 1);                     // [nnz]
  int* s_band = reinterpret_cast<int*>(s_wt + nnz);                       // [3][n_mels]: start, len, offset

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kFramesPerCta;
  const int nf = min(kFramesPerCta, T - t0);
  const long long seg_base = (long long)b * n_samples;

  // ---- stage samples (reflect padding of n_fft/2 resolved here) and tables
  const int count = (nf - 1) * hop + frame_len;
  const int p0 = t0 * hop - (center ? frame_len / 2 : 0);  // index into the unpadded window of the first sample
  bool staged = false;
  if constexpr (kI16) {
    // interior tiles: 16-byte vector loads (8 samples), all issued before the first use, so one
    // memory round trip covers the whole stage instead of ~9 dependent ones
    const short* src16 = reinterpret_cast<const short*>(pcm) + seg_base + p0;
    if (p0 >= 0 && p0 + count <= n_samples && (count & 7) == 0 &&
        (reinterpret_cast<uintptr_t>(src16) & 15) == 0) {
      const int nvec = count >> 3;
      constexpr int kMaxIt = 5;  // 5 * 256 * 8 = 10240 >= (16-1)*hop + 2048 for hop <= 546
      if (nvec <= kMaxIt * kThreads) {
        int4 v[kMaxIt];
#pragma unroll
        for (int it = 0; it < kMaxIt; ++it) {
          const int vi = tid + it * kThreads;
          if (vi < nvec) v[it] = __ldg(reinterpret_cast<const int4*>(src16) + vi);
        }
#pragma unroll
        for (int it = 0; it < kMaxIt; ++it) {
          const int vi = tid + it * kThreads;
          if (vi < nvec) {
            const short* q = reinterpret_cast<const short*>(&v[it]);
            float4 lo, hi;
            lo.x = pcm16_to_f32(q[0]); lo.y = pcm16_to_f32(q[1]);
            lo.z = pcm16_to_f32(q[2]); lo.w = pcm16_to_f32(q[3]);
            hi.x = pcm16_to_f32(q[4]); hi.y = pcm16_to_f32(q[5]);
            hi.z = pcm16_to_f32(q[6]); hi.w = pcm16_to_f32(q[7]);
            reinterpret_cast<float4*>(s_x)[2 * vi] = lo;
            reinterpret_cast<float4*>(s_x)[2 * vi + 1] = hi;
          }
        }
        staged = true;
      }
    }
  }
  if (!staged) {
    for (int i = tid; i < count; i += kThreads) {
      int src = p0 + i;
      if (src < 0) src = -src;
      if (src >= n_samples) src = 2 * (n_samples - 1) - src;
      s_x[i] = load_sample<kI16>(pcm, seg_base + src);
    }
  }
  for (int i = tid; i < kNfft - frame_len; i += kThreads) s_x[count + i] = 0.f;  // finite tail under the zero window
  {
    // window (2048 floats) and twiddles (1024 float2): 16-byte loads, all in flight before the first store
    static_assert(kNfft == 8 * kThreads && 32 * 32 * 2 == 8 * kThreads, "table staging assumes 256 threads");
    const float4* gw = reinterpret_cast<const float4*>(tb.window);
    const float4* gt = reinterpret_cast<const float4*>(tb.fft_tw);
    const float4 w0 = __ldg(gw + tid), w1 = __ldg(gw + tid + kThreads);
    const float4 t0v = __ldg(gt + tid), t1v = __ldg(gt + tid + kThreads);
    reinterpret_cast<float4*>(s_win)[tid] = w0;
    reinterpret_cast<float4*>(s_win)[tid + kThreads] = w1;
    reinterpret_cast<float4*>(s_tw)[tid] = t0v;
    reinterpret_cast<float4*>(s_tw)[tid + kThreads] = t1v;
  }
  for (int i = tid; i < nnz; i += kThreads) s_wt[i] = tb.weights[i];
  for (int i = tid; i < n_mels; i += kThreads) {
    s_band[i] = tb.band_start[i];
    s_band[n_mels + i] = tb.band_len[i];
    s_band[2 * n_mels + i] = tb.band_off[i];
  }
  __syncthreads();

  float* tr = s_tr + warp * 32 * kTrStride;
  const int n_band_iter = (n_mels + 31) >> 5;

  for (int f = warp; f < nf; f += kWarps) {
    float re[32], im[32];
    // ---- z[n] = x[2n]w[2n] + i x[2n+1]w[2n+1];  lane = n2, element n1 holds z[32*n1 + n2]
    const float2* xf = reinterpret_cast<const float2*>(s_x + f * hop);
    const float2* wf = reinterpret_cast<const float2*>(s_win);
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
      const float2 x = xf[32 * n1 + lane];
      const float2 w = wf[32 * n1 + lane];
      re[n1] = x.x * w.x;
      im[n1] = x.y * w.y;
    }
    fft32(re, im);  // element i = Y[k1 = rev5(i)] for this n2
    // ---- twiddle W_1024^(n2*k1) and transpose to lane = k1, element = n2
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int k1 = rev5(i);
      const float2 w = s_tw[k1 * 32 + lane];
      const float r = re[i], q = im[i];
      re[i] = fmaf(r, w.x, -q * w.y);
      im[i] = fmaf(r, w.y, q * w.x);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) tr[rev5(i) * kTrStride + lane] = re[i];
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) re[n2] = tr[lane * kTrStride + n2];
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 32; ++i) tr[rev5(i) * kTrStride + lane] = im[i];
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) im[n2] = tr[lane * kTrStride + n2];
    __syncwarp();
    fft32(re, im);  // element i = Z[k1 + 32*k2], k1 = lane, k2 = rev5(i)

    // ---- real-FFT split + power:  X[k] = (Z[k]+Z*[N-k])/2 - (i/2) W_2048^k (Z[k]-Z*[N-k])
    const int partner = (32 - lane) & 31;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int k2 = rev5(i);
      if (k2 < kK2) {  // compile time
        float pr = __shfl_sync(0xffffffffu, re[31 - i], partner);
        float pi = __shfl_sync(0xffffffffu, im[31 - i], partner);
        if (lane == 0) {  // N-k = 32*(32-k2): same lane, element rev5((32-k2)&31)
          pr = re[rev5((32 - k2) & 31)];
          pi = im[rev5((32 - k2) & 31)];
        }
        const int k = lane + 32 * k2;
        const float2 w = __ldg(&tb.post_tw[k]);  // (cos, -sin)
        const float er = re[i] + pr, ei = im[i] - pi;
        const float orr = re[i] - pr, oi = im[i] + pi;
        const float xr = 0.5f * (er + fmaf(w.x, oi, w.y * orr));
        const float xi = 0.5f * (ei - fmaf(w.x, orr, -w.y * oi));
        tr[k] = fmaf(xr, xr, xi * xi);
      }
    }
    if (max_bin >= kNc && lane == 0) {  // Nyquist bin: X[1024] = Re Z[0] - Im Z[0]
      const float ny = re[0] - im[0];
      tr[kNc] = ny * ny;
    }
    __syncwarp();

    // ---- triangular mel filters (CSR), ascending-bin summation, then dB
    for (int j = 0; j < n_band_iter; ++j) {
      const int m = lane + 32 * j;
      if (m < n_mels) {
        const int st = s_band[m], len = s_band[n_mels + m];
        const float* wt = s_wt + s_band[2 * n_mels + m];
        float acc = 0.0f;
        for (int q = 0; q < len; ++q) acc = fmaf(wt[q], tr[(st + q) << bin_shift], acc);
        s_out[m * (kFramesPerCta + 1) + f] = log_mode ? log10f(fmaf(10000.0f, acc, 1.0f)) : 10.0f * log10f(fmaxf(acc, 1e-10f));
      }
    }
    __syncwarp();
  }
  __syncthreads();

  // ---- write the tile
  if (!transpose) {
    float* o = out + (long long)b * n_mels * T;
    for (int i = tid; i < n_mels * kFramesPerCta; i += kThreads) {
      const int m = i / kFramesPerCta, tl = i % kFramesPerCta;
      if (tl < nf) o[(long long)m * T + t0 + tl] = s_out[m * (kFramesPerCta + 1) + tl];
    }
  } else {
    float* o = out + (long long)b * T * n_mels;
    for (int i = tid; i < n_mels * kFramesPerCta; i += kThreads) {
      const int tl = i / n_mels, m = i % n_mels;
      if (tl < nf) o[(long long)(t0 + tl) * n_mels + m] = s_out[m * (kFramesPerCta + 1) + tl];
    }
  }
}

static size_t mel_smem_bytes(int hop, int n_mels, int nnz) {
  const int n_stage = (kFramesPerCta - 1) * hop + kNfft;
  size_t floats = ((n_stage + 3) & ~3) + kNfft + 2 * 32 * 32 + (size_t)kWarps * 32 * kTrStride +
                  (size_t)n_mels * (kFramesPerCta + 1) + (size_t)nnz + 3 * (size_t)n_mels;
  return floats * sizeof(float);
}

int mel_plan_hop(const am_mel_plan* plan) { return plan->cfg.hop; }

static int validate_cfg(const am_mel_cfg* c) {
  AM_CHECK(c != nullptr, "mel cfg is NULL");
  AM_CHECK(c->n_fft == 2048 || c->n_fft == 1024 || c->n_fft == 512, "mel: n_fft must be 2048, 1024 or 512 (got %d)",
           c->n_fft);
  AM_CHECK(c->hop > 0 && (c->hop % 2) == 0 && c->hop <= kNfft, "mel: hop must be even, in (0, 2048]");
  AM_CHECK(c->n_mels > 0 && c->n_mels <= 256, "mel: n_mels must be in [1, 256]");
  AM_CHECK(c->sr > 0, "mel: sr must be positive");
  return AM_OK;
}

}  // namespace am

using namespace am;

extern "C" int am_mel_num_frames(const am_mel_cfg* cfg, int n_samples) {
  if (!cfg || cfg->hop <= 0 || n_samples < 0) return AM_ERR_INVALID;
  return 1 + n_samples / cfg->hop;
}

// host-only helper (no GPU): the filterbank the plan uploads, dense f32[n_mels, n_fft/2+1]
extern "C" int am_mel_filterbank(const am_mel_cfg* cfg, float* out) {
  AM_CHECK(cfg && out, "am_mel_filterbank: NULL argument");
  std::vector<float> w;
  AM_TRY(build_filterbank(*cfg, w));
  std::memcpy(out, w.data(), w.size() * sizeof(float));
  return AM_OK;
}

extern "C" int am_mel_plan_create(const am_mel_cfg* cfg, am_mel_plan** out) {
  AM_CHECK(out != nullptr, "am_mel_plan_create: out is NULL");
  *out = nullptr;
  AM_TRY(validate_cfg(cfg));
  AM_TRY(ensure_init());
  std::vector<float> fb;
  AM_TRY(build_filterbank(*cfg, fb));
  const int bins = cfg->n_fft / 2 + 1, nm = cfg->n_mels;
  std::vector<int> st(nm), len(nm), off(nm);
  std::vector<float> wts;
  int max_bin = 0;
  for (int m = 0; m < nm; ++m) {
    int lo = -1, hi = -1;
    for (int k = 0; k < bins; ++k)
      if (fb[(size_t)m * bins + k] != 0.0f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    st[m] = lo < 0 ? 0 : lo;
    len[m] = lo < 0 ? 0 : hi - lo + 1;
    off[m] = (int)wts.size();
    for (int k = 0; k < len[m]; ++k) wts.push_back(fb[(size_t)m * bins + st[m] + k]);
    if (hi > max_bin) max_bin = hi;
  }
  // periodic Hann of the frame length; zero beyond it (frames shorter than 2048 are zero-padded transforms)
  std::vector<float> win(kNfft, 0.0f);
  for (int n = 0; n < cfg->n_fft; ++n) win[n] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * n / cfg->n_fft));
  std::vector<float2> ftw, ptw;
  fill_fft_twiddles(ftw, ptw);
  auto* plan = new am_mel_plan();
  plan->cfg = *cfg;
  plan->max_bin = max_bin;
  plan->nnz = (int)wts.size();
  // one allocation, 256-byte aligned slices
  size_t o_win = 0, o_ftw = round_up(o_win + win.size() * 4, 256),
         o_ptw = round_up(o_ftw + ftw.size() * 8, 256), o_st = round_up(o_ptw + ptw.size() * 8, 256),
         o_len = round_up(o_st + nm * 4, 256), o_off = round_up(o_len + nm * 4, 256),
         o_w = round_up(o_off + nm * 4, 256), total = round_up(o_w + wts.size() * 4 + 4, 256);
  int s = plan->storage.alloc(total);
  if (s != AM_OK) {
    delete plan;
    return s;
  }
  char* base = plan->storage.p;
  std::vector<char> host(total, 0);
  std::memcpy(host.data() + o_win, win.data(), win.size() * 4);
  std::memcpy(host.data() + o_ftw, ftw.data(), ftw.size() * 8);
  std::memcpy(host.data() + o_ptw, ptw.data(), ptw.size() * 8);
  std::memcpy(host.data() + o_st, st.data(), nm * 4);
  std::memcpy(host.data() + o_len, len.data(), nm * 4);
  std::memcpy(host.data() + o_off, off.data(), nm * 4);
  std::memcpy(host.data() + o_w, wts.data(), wts.size() * 4);
  cudaError_t e = cudaMemcpy(base, host.data(), total, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    delete plan;
    return cuda_fail(e, "cudaMemcpy(mel tables)", __FILE__, __LINE__);
  }
  plan->t.window = reinterpret_cast<float*>(base + o_win);
  plan->t.fft_tw = reinterpret_cast<float2*>(base + o_ftw);
  plan->t.post_tw = reinterpret_cast<float2*>(base + o_ptw);
  plan->t.band_start = reinterpret_cast<int*>(base + o_st);
  plan->t.band_len = reinterpret_cast<int*>(base + o_len);
  plan->t.band_off = reinterpret_cast<int*>(base + o_off);
  plan->t.weights = reinterpret_cast<float*>(base + o_w);
  const size_t smem = mel_smem_bytes(cfg->hop, cfg->n_mels, plan->nnz);
  e = cudaFuncSetAttribute(mel_kernel<true, 19>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(mel_kernel<false, 19>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(mel_kernel<true, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(mel_kernel<false, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    delete plan;
    return cuda_fail(e, "cudaFuncSetAttribute(mel)", __FILE__, __LINE__);
  }
  *out = plan;
  return AM_OK;
}

extern "C" void am_mel_plan_free(am_mel_plan* plan) { delete plan; }

// same tables, other framing / compression: center = 0 (librosa center=False), log_mode = 1 (log10(1 + 10000 x)) is
// the MusiCNN front end of tasks/analysis.py:371-375
extern "C" int am_mel_plan_create_ex(const am_mel_cfg* cfg, int center, int log_mode, am_mel_plan** out) {
  AM_CHECK((center == 0 || center == 1) && (log_mode == 0 || log_mode == 1), "am_mel_plan_create_ex: bad mode");
  AM_TRY(am_mel_plan_create(cfg, out));
  (*out)->center = center;
  (*out)->log_mode = log_mode;
  return AM_OK;
}

extern "C" int am_mel_num_frames_ex(const am_mel_cfg* cfg, int center, int n_samples) {
  if (!cfg || cfg->hop <= 0) return 0;
  return center ? 1 + n_samples / cfg->hop : (n_samples >= cfg->n_fft ? 1 + (n_samples - cfg->n_fft) / cfg->hop : 0);
}

extern "C" int am_mel_batch_dev(const am_mel_plan* plan, const void* pcm_dev, int pcm_is_i16, int B,
                                int n_samples, float* out_dev, void* stream) {
  AM_CHECK(plan && pcm_dev && out_dev, "am_mel_batch_dev: NULL argument");
  AM_CHECK(B >= 0, "am_mel_batch_dev: negative batch");
  AM_CHECK(plan->center ? n_samples > plan->cfg.n_fft / 2 : n_samples >= plan->cfg.n_fft,
           "mel: window of %d samples is shorter than %s", n_samples, plan->center ? "the reflect pad" : "one frame");
  if (B == 0) return AM_OK;
  const am_mel_cfg& c = plan->cfg;
  const int T = plan->center ? 1 + n_samples / c.hop : 1 + (n_samples - c.n_fft) / c.hop;
  const size_t smem = mel_smem_bytes(c.hop, c.n_mels, plan->nnz);
  cudaStream_t st = (cudaStream_t)stream;
  for (int b0 = 0; b0 < B; b0 += 65535) {  // gridDim.y limit
    const int nb = std::min(65535, B - b0);
    dim3 grid(ceil_div(T, kFramesPerCta), nb);
    const char* in = (const char*)pcm_dev + (size_t)b0 * n_samples * (pcm_is_i16 ? 2 : 4);
    float* o = out_dev + (size_t)b0 * c.n_mels * T;
    const int shift = c.n_fft == 2048 ? 0 : (c.n_fft == 1024 ? 1 : 2);
    const int max_bin = plan->max_bin << shift;  // in 2048-point bins
    const bool narrow = max_bin < 19 * 32;  // student config: highest weighted bin is 597
    if (pcm_is_i16) {
      if (narrow) {
        AM_LAUNCH((mel_kernel<true, 19>), grid, kThreads, smem, st, in, n_samples, c.hop, T, c.n_mels, max_bin,
                  c.transpose, c.n_fft, shift, plan->nnz, plan->center, plan->log_mode, plan->t, o);
      } else {
        AM_LAUNCH((mel_kernel<true, 32>), grid, kThreads, smem, st, in, n_samples, c.hop, T, c.n_mels, max_bin,
                  c.transpose, c.n_fft, shift, plan->nnz, plan->center, plan->log_mode, plan->t, o);
      }
    } else {
      if (narrow) {
        AM_LAUNCH((mel_kernel<false, 19>), grid, kThreads, smem, st, in, n_samples, c.hop, T, c.n_mels, max_bin,
                  c.transpose, c.n_fft, shift, plan->nnz, plan->center, plan->log_mode, plan->t, o);
      } else {
        AM_LAUNCH((mel_kernel<false, 32>), grid, kThreads, smem, st, in, n_samples, c.hop, T, c.n_mels, max_bin,
                  c.transpose, c.n_fft, shift, plan->nnz, plan->center, plan->log_mode, plan->t, o);
      }
    }
  }
  return AM_OK;
}

static int mel_batch_host(const void* pcm, int is_i16, int B, int n_samples, const am_mel_cfg* cfg,
                          float* out, int center = 1, int log_mode = 0) {
  AM_CHECK(pcm && out, "am_mel_batch: NULL buffer");
  AM_TRY(validate_cfg(cfg));
  AM_CHECK(B >= 0 && cfg && (center ? n_samples > cfg->n_fft / 2 : n_samples >= cfg->n_fft),
           "am_mel_batch: bad shape B=%d n_samples=%d", B, n_samples);
  if (B == 0) return AM_OK;
  am_mel_plan* plan = nullptr;
  AM_TRY(am_mel_plan_create_ex(cfg, center, log_mode, &plan));
  const int T = am_mel_num_frames_ex(cfg, center, n_samples);
  const size_t in_bytes = (size_t)B * n_samples * (is_i16 ? 2 : 4);
  const size_t out_elems = (size_t)B * cfg->n_mels * T;
  DevBuf<char> d_in;
  DevBuf<float> d_out;
  Stream st;
  int s = d_in.alloc(in_bytes);
  if (s == AM_OK) s = d_out.alloc(out_elems);
  if (s == AM_OK) s = st.create();
  if (s == AM_OK) {
    cudaError_t e = cudaMemcpyAsync(d_in.p, pcm, in_bytes, cudaMemcpyHostToDevice, st.s);
    if (e != cudaSuccess) s = cuda_fail(e, "H2D pcm", __FILE__, __LINE__);
  }
  if (s == AM_OK) s = am_mel_batch_dev(plan, d_in.p, is_i16, B, n_samples, d_out.p, st.s);
  if (s == AM_OK) {
    cudaError_t e = cudaMemcpyAsync(out, d_out.p, out_elems * 4, cudaMemcpyDeviceToHost, st.s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st.s);
    if (e != cudaSuccess) s = cuda_fail(e, "D2H mel", __FILE__, __LINE__);
  }
  am_mel_plan_free(plan);
  return s;
}

extern "C" int am_mel_batch(const float* pcm, int B, int n_samples, const am_mel_cfg* cfg, float* out) {
  return mel_batch_host(pcm, 0, B, n_samples, cfg, out);
}
extern "C" int am_mel_batch_i16(const int16_t* pcm, int B, int n_samples, const am_mel_cfg* cfg,
                                float* out) {
  return mel_batch_host(pcm, 1, B, n_samples, cfg, out);
}
extern "C" int am_mel_batch_ex(const float* pcm, int B, int n_samples, const am_mel_cfg* cfg, int center, int log_mode,
                               float* out) {
  AM_CHECK((center == 0 || center == 1) && (log_mode == 0 || log_mode == 1), "am_mel_batch_ex: bad mode");
  return mel_batch_host(pcm, 0, B, n_samples, cfg, out, center, log_mode);
}

// tasks/clap_analyzer.py:502-523 (host side: decode stays on the host, SURVEY 8(a))
extern "C" int am_pcm_to_segments(const float* audio, int64_t L, int16_t* seg, int max_seg, int* n_seg) {
  AM_CHECK(n_seg != nullptr, "am_pcm_to_segments: n_seg is NULL");
  AM_CHECK(L >= 0 && (audio != nullptr || L == 0), "am_pcm_to_segments: bad audio buffer");
  constexpr int64_t SEG = 480000, HOP = 240000;
  std::vector<int64_t> starts;
  if (L <= SEG) {
    starts.push_back(0);
  } else {
    for (int64_t s = 0; s + SEG <= L; s += HOP) starts.push_back(s);
    if ((int64_t)starts.size() * HOP < L) starts.push_back(L - SEG);
  }
  *n_seg = (int)starts.size();
  if (seg == nullptr) return AM_OK;
  AM_CHECK(max_seg >= *n_seg, "am_pcm_to_segments: need room for %d windows, got %d", *n_seg, max_seg);
  for (size_t i = 0; i < starts.size(); ++i) {
    int16_t* dst = seg + i * SEG;
    const int64_t s0 = starts[i];
    const int64_t n = std::min<int64_t>(SEG, L - s0);
    for (int64_t j = 0; j < n; ++j) {
      float v = audio[s0 + j];
      v = v < -1.0f ? -1.0f : (v > 1.0f ? 1.0f : v);   // np.clip
      dst[j] = (int16_t)(v * 32767.0f);                // float32 product, C truncation (astype(int16))
    }
    for (int64_t j = n; j < SEG; ++j) dst[j] = 0;      // zero right-pad of a short track
  }
  return AM_OK;
}
