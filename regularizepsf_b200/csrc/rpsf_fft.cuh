// rpsf_fft.cuh — register-resident and thread-cooperative complex FFTs for sm_100a.
//
// The correction path (reference: regularizepsf/transform.py:163-164, scipy.fft.fft2 /
// ifft2 over (N,P,P) patches) needs only power-of-two lengths P in {16..512}.  A length-P
// transform is split P = N1 * N2 and run by N1 cooperating threads:
//
//   pass A   each thread owns the N2 samples  x[n1 + N1*j]  and runs an N2-point FFT in
//            registers (fully unrolled radix-2 DIF, compile-time twiddles that become FFMA
//            immediates), then scales by the inter-pass twiddle  w_P^(n1*k2);
//   exchange an N1 x N2 transpose through shared memory (layout chosen by the caller);
//   pass B   each thread runs N2/N1 (1 or 2) N1-point FFTs; bin  k = k2 + N2*k1.
//
// The inverse runs the same passes backwards with conjugated twiddles, so forward output
// order == inverse input order and no bit-reversal pass ever touches memory.  No scaling
// is applied in either direction (the 1/P^2 of ifft2 is folded into the stored kernel).
#pragma once
#include <cuda_runtime.h>
#include <type_traits>

namespace rpsf {

template <typename T> struct Vec2;
template <> struct Vec2<float>  { using type = float2;  };
template <> struct Vec2<double> { using type = double2; };
template <typename T> using cplx = typename Vec2<T>::type;

template <typename T> __host__ __device__ __forceinline__ cplx<T> mk(T re, T im) { cplx<T> r; r.x = re; r.y = im; return r; }

// ---- packed pair arithmetic ------------------------------------------------------------------
// A complex number is an aligned (re, im) register pair.  sm_100a has packed fp32 instructions
// (FADD2 / FMUL2 / FFMA2: one issue slot for both halves) whose operands take free modifiers:
// negate, swap halves (.LO_HI), swap-and-negate-one (.LO_HI.NP) and scalar / immediate broadcast.
// Written as make_float2(...) shuffles around the intrinsics below, ptxas folds all of them into
// the instruction, so a complex add is ONE instruction, a complex multiply TWO and a multiply by
// +-i none at all.  double has no packed form; the same expressions compile to scalar DADD/DFMA.
__device__ __forceinline__ float2 padd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 pmul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ double2 padd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 pmul(double2 a, double2 b) { return make_double2(a.x * b.x, a.y * b.y); }
__device__ __forceinline__ double2 pfma(double2 a, double2 b, double2 c) {
  return make_double2(fma(a.x, b.x, c.x), fma(a.y, b.y, c.y));
}
template <typename C> __device__ __forceinline__ C cadd(C a, C b) { return padd(a, b); }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { C n; n.x = -b.x; n.y = -b.y; return padd(a, n); }
// a * b = a * b.re + (a.im, a.re) * (-b.im, b.im)
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
  C sw, im, re; sw.x = a.y; sw.y = a.x; im.x = -b.y; im.y = b.y; re.x = b.x; re.y = b.x;
  return pfma(a, re, pmul(sw, im));
}
// a * conj(b)
template <typename C> __device__ __forceinline__ C cmulc(C a, C b) {
  C sw, im, re; sw.x = a.y; sw.y = a.x; im.x = b.y; im.y = -b.y; re.x = b.x; re.y = b.x;
  return pfma(a, re, pmul(sw, im));
}
// a * s for a real scalar s
template <typename C, typename T> __device__ __forceinline__ C cscale(C a, T s) { C b; b.x = s; b.y = s; return pmul(a, b); }
// a * s rounded on its own, never contracted with the add that consumes it (the row window the readers of the band
// buffer apply must round exactly as the product stored by the row pass once did).  Scalar __fmul_rn: ptxas was seen
// to fuse the packed __fmul2_rn into the FFMA2 of the first butterfly.
__device__ __forceinline__ float2 cscale_rn(float2 a, float s) { return make_float2(__fmul_rn(a.x, s), __fmul_rn(a.y, s)); }
__device__ __forceinline__ double2 cscale_rn(double2 a, double s) { return make_double2(__dmul_rn(a.x, s), __dmul_rn(a.y, s)); }

// ---- compile-time twiddles: cos(2*pi*m/64), m = 0..16, correctly rounded doubles ----------
__host__ __device__ constexpr double cos64_table(int m) {
  constexpr double t[17] = {
      1.0, 0.9951847266721969, 0.9807852804032304, 0.9569403357322088, 0.9238795325112867,
      0.881921264348355, 0.8314696123025452, 0.773010453362737, 0.7071067811865476,
      0.6343932841636455, 0.5555702330196022, 0.47139673682599764, 0.3826834323650898,
      0.2902846772544624, 0.19509032201612828, 0.0980171403295606, 0.0};
  return t[m];
}
// cos / sin of 2*pi*m/64 for m in [0, 32]
__host__ __device__ constexpr double cos64(int m) { return m <= 16 ? cos64_table(m) : -cos64_table(32 - m); }
__host__ __device__ constexpr double sin64(int m) { return m <= 16 ? cos64_table(16 - m) : cos64_table(m - 16); }

template <int B, int E, typename F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(f);
  }
}

// d * w_SPAN^J (forward: w = exp(-2*pi*i/SPAN); inverse: conjugate).  0 <= J < SPAN/2.
template <int SPAN, int J, bool INV, typename T>
__device__ __forceinline__ cplx<T> twiddle_mul(cplx<T> d) {
  static_assert(SPAN <= 64 && J >= 0 && 2 * J < SPAN, "twiddle out of table range");
  const cplx<T> rot = INV ? mk<T>(-d.y, d.x) : mk<T>(d.y, -d.x);      // d * (+-i): an operand modifier
  if constexpr (J == 0) {
    return d;
  } else if constexpr (4 * J == SPAN) {          // -i (fwd) / +i (inv)
    return rot;
  } else if constexpr (8 * J == SPAN) {          // (1 -/+ i)/sqrt2
    constexpr T h = T(0.7071067811865476);
    return cscale(padd(d, rot), h);
  } else if constexpr (8 * J == 3 * SPAN) {      // (-1 -/+ i)/sqrt2
    constexpr T h = T(0.7071067811865476);
    return cscale(padd(rot, mk<T>(-d.x, -d.y)), h);
  } else {
    constexpr int m = 64 / SPAN * J;
    constexpr T c = T(cos64(m));
    constexpr T s = T(sin64(m));
    // d * (c -/+ i s) = d * c + rot * s
    return pfma(d, mk<T>(c, c), cscale(rot, s));
  }
}

__host__ __device__ constexpr int bitrev(int v, int bits) {
  int r = 0;
  for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1) << (bits - 1 - i);
  return r;
}
__host__ __device__ constexpr int ilog2(int n) { return n <= 1 ? 0 : 1 + ilog2(n >> 1); }

// In-register N-point DFT, natural order in and out, N in {1,2,4,8,16,32}.  Unnormalised.
template <int N, bool INV, typename T>
__device__ __forceinline__ void fft_reg(cplx<T> (&v)[N]) {
  if constexpr (N > 1) {
    // radix-2 decimation in frequency: span = N, N/2, ..., 2
    static_for<0, ilog2(N)>([&](auto stage) {
      constexpr int span = N >> decltype(stage)::value;
      constexpr int half = span / 2;
      static_for<0, N / span>([&](auto blk) {
        constexpr int base = decltype(blk)::value * span;
        static_for<0, half>([&](auto jj) {
          constexpr int j = decltype(jj)::value;
          const cplx<T> a = v[base + j];
          const cplx<T> b = v[base + j + half];
          v[base + j] = cadd(a, b);
          v[base + j + half] = twiddle_mul<span, j, INV, T>(csub(a, b));
        });
      });
    });
    // bit-reversal is a compile-time register renaming
    cplx<T> t[N];
    static_for<0, N>([&](auto i) { t[decltype(i)::value] = v[bitrev(decltype(i)::value, ilog2(N))]; });
    static_for<0, N>([&](auto i) { v[decltype(i)::value] = t[decltype(i)::value]; });
  }
}

// ---- split of a length-P transform over N1 threads x N2 registers --------------------------
template <int P> struct Split;
template <> struct Split<16>  { static constexpr int N1 = 4,  N2 = 4;  };
template <> struct Split<32>  { static constexpr int N1 = 4,  N2 = 8;  };
template <> struct Split<64>  { static constexpr int N1 = 8,  N2 = 8;  };
template <> struct Split<128> { static constexpr int N1 = 8,  N2 = 16; };
template <> struct Split<256> { static constexpr int N1 = 16, N2 = 16; };
template <> struct Split<512> { static constexpr int N1 = 16, N2 = 32; };

// Cooperative forward FFT.
//   in : v[j]            = x[t + N1*j]                       (t = this thread's index in the team)
//   out: v[m*N1 + k1]    = X[(t + N1*m) + N2*k1]             (m < N2/N1, k1 < N1)
// `ex(k2, n1)` maps an exchange slot to a shared-memory index private to this team,
// `sync()` orders the team's writes before its reads (and is called once more before return
// so the caller may reuse the buffer).  tw[k2*N1 + n1] = exp(-2*pi*i*n1*k2/P).
// `done()` runs after the last read of the exchange buffer (the two-argument form passes `sync`).
template <int P, typename T, typename Ex, typename Sync, typename Done>
__device__ __forceinline__ void coop_fft_forward(cplx<T> (&v)[Split<P>::N2], int t, cplx<T>* smem,
                                                 const cplx<T>* __restrict__ tw, Ex ex, Sync sync, Done done) {
  constexpr int N1 = Split<P>::N1, N2 = Split<P>::N2, R = N2 / N1;
  fft_reg<N2, false, T>(v);
  static_for<1, N2>([&](auto kk) {
    constexpr int k2 = decltype(kk)::value;
    v[k2] = cmul(v[k2], tw[k2 * N1 + t]);
  });
  static_for<0, N2>([&](auto kk) { smem[ex(decltype(kk)::value, t)] = v[decltype(kk)::value]; });
  sync();
  static_for<0, R>([&](auto mm) {
    constexpr int m = decltype(mm)::value;
    cplx<T> y[N1];
    static_for<0, N1>([&](auto nn) { y[decltype(nn)::value] = smem[ex(t + N1 * m, decltype(nn)::value)]; });
    fft_reg<N1, false, T>(y);
    static_for<0, N1>([&](auto nn) { v[m * N1 + decltype(nn)::value] = y[decltype(nn)::value]; });
  });
  done();
}
template <int P, typename T, typename Ex, typename Sync>
__device__ __forceinline__ void coop_fft_forward(cplx<T> (&v)[Split<P>::N2], int t, cplx<T>* smem,
                                                 const cplx<T>* __restrict__ tw, Ex ex, Sync sync) {
  coop_fft_forward<P, T>(v, t, smem, tw, ex, sync, sync);
}

// Cooperative inverse FFT: exact reverse of the forward (conjugate twiddles, unnormalised).
//   in : v[m*N1 + k1] = X[(t + N1*m) + N2*k1]
//   out: v[j]         = x[t + N1*j]
// `done()` runs after the last read of the exchange buffer (pass `sync` unless the caller orders
// the buffer's next use itself).
template <int P, typename T, typename Ex, typename Sync, typename Done>
__device__ __forceinline__ void coop_fft_inverse(cplx<T> (&v)[Split<P>::N2], int t, cplx<T>* smem,
                                                 const cplx<T>* __restrict__ tw, Ex ex, Sync sync, Done done) {
  constexpr int N1 = Split<P>::N1, N2 = Split<P>::N2, R = N2 / N1;
  static_for<0, R>([&](auto mm) {
    constexpr int m = decltype(mm)::value;
    cplx<T> y[N1];
    static_for<0, N1>([&](auto nn) { y[decltype(nn)::value] = v[m * N1 + decltype(nn)::value]; });
    fft_reg<N1, true, T>(y);
    static_for<0, N1>([&](auto nn) { smem[ex(t + N1 * m, decltype(nn)::value)] = y[decltype(nn)::value]; });
  });
  sync();
  static_for<0, N2>([&](auto kk) { v[decltype(kk)::value] = smem[ex(decltype(kk)::value, t)]; });
  static_for<1, N2>([&](auto kk) {
    constexpr int k2 = decltype(kk)::value;
    v[k2] = cmulc(v[k2], tw[k2 * N1 + t]);
  });
  done();
  fft_reg<N2, true, T>(v);
}
template <int P, typename T, typename Ex, typename Sync>
__device__ __forceinline__ void coop_fft_inverse(cplx<T> (&v)[Split<P>::N2], int t, cplx<T>* smem,
                                                 const cplx<T>* __restrict__ tw, Ex ex, Sync sync) {
  coop_fft_inverse<P, T>(v, t, smem, tw, ex, sync, sync);
}

}  // namespace rpsf
