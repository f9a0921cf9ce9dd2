// Register FFT helpers shared by the STFT kernels (mel.cu, track_features.cu), sm_100a.
//
// A 2048-point real frame is transformed as a 1024-point complex FFT laid out 32 x 32 over one warp: each lane runs
// fft32 on its column, applies W_1024^(n2*k1) from the table fft_tw, transposes through shared memory, runs fft32
// again, and the real-FFT split X[k] = (Z[k]+Z*[N-k])/2 - (i/2) W_2048^k (Z[k]-Z*[N-k]) uses the table post_tw.
#pragma once

#include <cuda_runtime.h>

#include <cmath>
#include <vector>

namespace am {

// host: the two twiddle tables of the layout above.  ftw[k1*32 + n2] = W_1024^(n2*k1), ptw[k] = W_2048^k, stored as
// (cos, -sin) in float32 from float64 angles.
inline void fill_fft_twiddles(std::vector<float2>& ftw, std::vector<float2>& ptw) {
  ftw.assign(32 * 32, make_float2(0.f, 0.f));
  ptw.assign(1024, make_float2(0.f, 0.f));
  for (int k1 = 0; k1 < 32; ++k1)
    for (int n2 = 0; n2 < 32; ++n2) {
      const double a = 2.0 * M_PI * (double)(n2 * k1) / 1024;
      ftw[k1 * 32 + n2] = make_float2((float)std::cos(a), (float)-std::sin(a));
    }
  for (int k = 0; k < 1024; ++k) {
    const double a = 2.0 * M_PI * k / 2048;
    ptw[k] = make_float2((float)std::cos(a), (float)-std::sin(a));
  }
}

// ---------------------------------------------------------------- device: 32-point FFT
__device__ __forceinline__ float cos32(int i) {  // cos(2*pi*i/32), i in [0,16)
  switch (i) {
    case 0: return 1.0f;
    case 1: return 0.98078528040323044913f;
    case 2: return 0.92387953251128675613f;
    case 3: return 0.83146961230254523708f;
    case 4: return 0.70710678118654752440f;
    case 5: return 0.55557023301960222474f;
    case 6: return 0.38268343236508977173f;
    case 7: return 0.19509032201612826785f;
    case 8: return 0.0f;
    case 9: return -0.19509032201612826785f;
    case 10: return -0.38268343236508977173f;
    case 11: return -0.55557023301960222474f;
    case 12: return -0.70710678118654752440f;
    case 13: return -0.83146961230254523708f;
    case 14: return -0.92387953251128675613f;
    default: return -0.98078528040323044913f;
  }
}
// sin(2*pi*i/32) for i in [0,16): sin(x) = cos(x - pi/2) -> index i-8; cos is even.
__device__ __forceinline__ float sin32i(int i) {
  int j = i - 8;
  if (j < 0) j = -j;
  return cos32(j);
}

__host__ __device__ constexpr int rev5(int i) {
  return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4);
}

// In-place radix-2 decimation-in-frequency, forward (e^{-i...}).  Input natural order,
// output bit-reversed: X[k] is left in element rev5(k).  Fully unrolled; all indices and
// twiddles are compile-time, trivial twiddles cost no multiplies.
__device__ __forceinline__ void fft32(float (&re)[32], float (&im)[32]) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
#pragma unroll
    for (int base = 0; base < 32; base += 2 * half) {
#pragma unroll
      for (int j = 0; j < half; ++j) {
        const int a = base + j, b = a + half;
        const float ar = re[a], ai = im[a], br = re[b], bi = im[b];
        re[a] = ar + br;
        im[a] = ai + bi;
        const float dr = ar - br, di = ai - bi;
        const int idx = j * (16 / half);  // twiddle W_32^idx = cos - i sin
        if (idx == 0) {
          re[b] = dr;
          im[b] = di;
        } else if (idx == 8) {  // * (-i)
          re[b] = di;
          im[b] = -dr;
        } else if (idx == 4) {  // * (1 - i)/sqrt2
          re[b] = (dr + di) * 0.70710678118654752440f;
          im[b] = (di - dr) * 0.70710678118654752440f;
        } else if (idx == 12) {  // * (-1 - i)/sqrt2
          re[b] = (di - dr) * 0.70710678118654752440f;
          im[b] = -(dr + di) * 0.70710678118654752440f;
        } else {
          const float c = cos32(idx), s = sin32i(idx);
          re[b] = fmaf(dr, c, di * s);
          im[b] = fmaf(di, c, -dr * s);
        }
      }
    }
  }
}

}  // namespace am
