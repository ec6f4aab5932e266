// rpsf_construct_grad.cuh — vector-Jacobian products of construct (transform.py:78-82) and of the PSF FFT cube
// (psf.py:216-219), so that a gradient reaches the PSF values, alpha and epsilon (DESIGN.md section 6).
//
// construct: K = conj(S) T f with a = |S|, b = |T|, c = eps b, D = a^(alpha+1) + c^(alpha+1), f = a^(alpha-1) / D.
// With G the incoming gradient of K (PyTorch's convention, dL/dRe + i dL/dIm) and w = Re(G S conj(T)):
//   grad_S = f conj(G) T + w a^(alpha-3) ((alpha-1) c^(alpha+1) - 2 a^(alpha+1)) / D^2 S
//   grad_T = f G S       - w (alpha+1) eps^(alpha+1) a^(alpha-1) b^(alpha-1) / D^2 T
//   grad_alpha =  sum w a^(alpha-1) c^(alpha+1) ln(a/c) / D^2
//   grad_eps   = -sum w (alpha+1) eps^alpha a^(alpha-1) b^(alpha+1) / D^2
// evaluated as u = a^(alpha+1) / D, v = c^(alpha+1) / D, w/a, S/a, w/b, T/b, which stay bounded where the closed form
// has 0 * inf products (|w| <= |G| a b).  Special bins: G = 0 gives exact zeros in all four outputs whatever S and T
// hold; where K is finite those products take their limit 0 (the second terms at a = 0 and b = 0, the grad_alpha term
// at a = 0 or c = 0, the grad_eps term at eps = 0); where K is not finite and G != 0 both cube outputs are NaN and so
// are the two sums.
//
// PSF FFT: X = fft2(x) with x real, so grad_x = Re(fft2(conj(G))): a row pass that conjugates on load, then a column
// pass that keeps the real part, both on the coop_fft_forward machinery of fft2_rows / fft2_cols.
#pragma once
#include "rpsf_kernels.cuh"

namespace rpsf {

// one wave of 8 CTAs of 256 threads on the 148 SMs of a B200; a constant, so that the partition of the bins over the
// CTAs, and with it the summation order of grad_alpha and grad_eps, does not depend on the device
constexpr int CGRAD_THREADS = 256;
constexpr int CGRAD_MAX_CTAS = 148 * 8;

// Elementwise over `count` bins.  gS / gT may be null (not computed, not written).  partial (nullable): one
// (grad_alpha, grad_eps) pair per CTA, summed in double in a fixed order (grid-stride per thread, then a fixed tree).
// DEV: alpha and epsilon come from two device doubles (`ae`), loaded once per CTA (construct_transfer_kernel's DEV).
template <typename T, bool DEV = false>
__global__ void __launch_bounds__(CGRAD_THREADS)
construct_transfer_kernel_backward(const cplx<T>* __restrict__ S, const cplx<T>* __restrict__ Tg,
                                   const cplx<T>* __restrict__ G, long long count, T alpha, T epsilon,
                                   cplx<T>* __restrict__ gS, cplx<T>* __restrict__ gT, double2* __restrict__ partial,
                                   const double* __restrict__ ae = nullptr) {
  if constexpr (DEV) {
    __shared__ T scalars[2];
    if (threadIdx.x == 0) { scalars[0] = T(ae[0]); scalars[1] = T(ae[1]); }
    __syncthreads();
    alpha = scalars[0];
    epsilon = scalars[1];
  }
  double acc_alpha = 0.0, acc_eps = 0.0;
  const T nan = T(NAN);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const cplx<T> g = G[i];
    if (g.x == T(0) && g.y == T(0)) {
      if (gS) gS[i] = mk<T>(T(0), T(0));
      if (gT) gT[i] = mk<T>(T(0), T(0));
      continue;
    }
    const cplx<T> s = S[i], tg = Tg[i];
    const T a = hypot(s.x, s.y), b = hypot(tg.x, tg.y), c = epsilon * b;
    // the forward's arithmetic (construct_transfer_kernel), to find the bins where K is not finite
    const T pw = pow_like_numpy<T>(a, alpha - T(1));
    const T ap = pow_like_numpy<T>(a, alpha + T(1)), cp = pow_like_numpy<T>(c, alpha + T(1));
    const T den = ap + cp;
    const T nx = s.x * pw, ny = -s.y * pw;
    T qx, qy;
    if (den == T(0)) { qx = nx / fabs(den); qy = ny / fabs(den); }
    else { const T scl = T(1) / den; qx = nx * scl; qy = ny * scl; }
    if (!isfinite(qx * tg.x - qy * tg.y) || !isfinite(qx * tg.y + qy * tg.x)) {
      if (gS) gS[i] = mk<T>(nan, nan);
      if (gT) gT[i] = mk<T>(nan, nan);
      acc_alpha += double(nan);
      acc_eps += double(nan);
      continue;
    }
    const T f = pw / den, u = ap / den, v = cp / den;
    // G S, and w = Re(G S conj(T))
    const T gsx = g.x * s.x - g.y * s.y, gsy = g.x * s.y + g.y * s.x;
    const T w = gsx * tg.x + gsy * tg.y;
    if (gS) {
      // f conj(G) T
      T rx = f * (g.x * tg.x + g.y * tg.y), ry = f * (g.x * tg.y - g.y * tg.x);
      if (a > T(0)) {
        const T sx = s.x / a, sy = s.y / a;
        const T k = f * ((alpha - T(1)) * v - T(2) * u) * (w / a);
        rx += k * sx; ry += k * sy;
      }
      gS[i] = mk<T>(rx, ry);
    }
    if (gT) {
      T rx = f * gsx, ry = f * gsy;
      if (b > T(0)) {
        const T tx = tg.x / b, ty = tg.y / b;
        const T k = (alpha + T(1)) * f * v * (w / b);
        rx -= k * tx; ry -= k * ty;
      }
      gT[i] = mk<T>(rx, ry);
    }
    if (partial) {
      const T fvw = f * v * w;
      if (a > T(0) && c > T(0)) acc_alpha += double(fvw * (log(a) - log(c)));
      if (epsilon > T(0)) acc_eps += double(-(alpha + T(1)) * fvw / epsilon);
    }
  }
  if (!partial) return;
  // fixed-order block reduction: butterfly within each warp, then warp 0 over the warps' sums
  __shared__ double red[2][CGRAD_THREADS / 32];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    acc_alpha += __shfl_xor_sync(0xffffffffu, acc_alpha, off);
    acc_eps += __shfl_xor_sync(0xffffffffu, acc_eps, off);
  }
  const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;
  if (lane == 0) { red[0][warp] = acc_alpha; red[1][warp] = acc_eps; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double sa = 0.0, se = 0.0;
    for (int k = 0; k < CGRAD_THREADS / 32; ++k) { sa += red[0][k]; se += red[1][k]; }
    partial[blockIdx.x] = make_double2(sa, se);
  }
}

// One CTA of THREADS threads: out = (sum of partial[.].x, sum of partial[.].y), in a fixed order.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
construct_grad_sum(const double2* __restrict__ partial, int n, double* __restrict__ out) {
  double sa = 0.0, se = 0.0;
  for (int k = threadIdx.x; k < n; k += THREADS) { sa += partial[k].x; se += partial[k].y; }
  __shared__ double red[2][THREADS];
  red[0][threadIdx.x] = sa; red[1][threadIdx.x] = se;
  __syncthreads();
  for (int half = THREADS / 2; half > 0; half >>= 1) {
    if ((int)threadIdx.x < half) {
      red[0][threadIdx.x] += red[0][threadIdx.x + half];
      red[1][threadIdx.x] += red[1][threadIdx.x + half];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[0] = red[0][0]; out[1] = red[1][0]; }
}

// ---- PSF FFT adjoint: values_grad = Re(fft2(conj(spectrum_grad))) ----------------------------------------------
// rows: fft2_rows with the complex input conjugated on load, into a complex scratch cube
template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::ROW_THREADS)
fft2_rows_conj(const cplx<T>* __restrict__ in, cplx<T>* __restrict__ out, const cplx<T>* __restrict__ tw_g,
               long long n_rows) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* scratch_all = tw + P;
  for (int i = threadIdx.x; i < P; i += blockDim.x) tw[i] = tw_g[i];
  __syncthreads();
  const int team = threadIdx.x / N1, t = threadIdx.x % N1;
  cplx<T>* scr = scratch_all + team * TL::SCR;
  const long long row = (long long)blockIdx.x * TL::TEAMS + team;
  if (row >= n_rows) return;
  const unsigned mask = team_mask(N1);
  auto ex = [](int k2, int n1) { return k2 * TL::EX_STRIDE + n1; };
  auto sync = [mask]() { __syncwarp(mask); };
  cplx<T> v[N2];
  static_for<0, N2>([&](auto jj) {
    constexpr int j = decltype(jj)::value;
    const cplx<T> z = in[row * P + t + N1 * j];
    v[j] = mk<T>(z.x, -z.y);
  });
  coop_fft_forward<P, T>(v, t, scr, tw, ex, sync);
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    scr[(t + N1 * (e / N1)) + N2 * (e % N1)] = v[e];
  });
  sync();
#pragma unroll
  for (int i = 0; i < P / N1; ++i) out[row * P + t + N1 * i] = scr[t + N1 * i];
}

// columns: fft2_cols reading the scratch cube and writing only the real part into the real (n, P, P) output
template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::K2_THREADS)
fft2_cols_real(const cplx<T>* __restrict__ data, T* __restrict__ out, const cplx<T>* __restrict__ tw_g,
               long long n_patches) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, C = TL::C;
  constexpr int NT = P / C;                                  // tiles across the full width
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* xbuf = tw + P;
  for (int i = threadIdx.x; i < P; i += blockDim.x) tw[i] = tw_g[i];
  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const long long sitem = (long long)blockIdx.x * TL::SLOTS + slot;
  const bool valid = sitem < n_patches * NT;
  const long long n = valid ? sitem / NT : 0;
  const int tile = valid ? int(sitem % NT) : 0;
  const long long offset = n * P * P + tile * C + c;
  cplx<T> v[N2];
  static_for<0, N2>([&](auto jj) {
    constexpr int j = decltype(jj)::value;
    v[j] = valid ? data[offset + (long long)(n1 + N1 * j) * P] : mk<T>(T(0), T(0));
  });
  __syncthreads();
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };
  auto sync = []() { __syncthreads(); };
  coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync);
  if (valid) {
    static_for<0, N2>([&](auto ee) {
      constexpr int e = decltype(ee)::value;
      out[offset + (long long)((n1 + N1 * (e / N1)) + N2 * (e % N1)) * P] = v[e].x;
    });
  }
}

}  // namespace rpsf
