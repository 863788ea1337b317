// Calculated particle images (bioem_b200_render_maps): the inverse of the forward r2c transform of
// bioem_kernels.cuh, applied to convolved spectra V = P_o conj(K_c) and written out as real images
//
//      out[item][x][y] = norm * R0[(x - cx) mod N][(y - cy) mod N] + mu,   R0 = c2r(V) / N^2
//
// so that sum R0 = sumC and sum_q out(q) I(q) at norm = 1, mu = 0 is the correlation value lCC / N^2 the likelihood
// uses at the displacement (-cx, -cy) (gen_corr_kernel: lCC[d] = sum_q R0(q + d) I(q)).  A c2r transform sees only the
// Hermitian part of the two self-conjugate columns ky = 0 and ky = N/2 (quirk Q1): on the fused path ctf_conv_kernel
// has already stored that part, and both paths take the real part of those columns after the kx transform, which is
// the same thing.  sum R0^2 is therefore sumsquareC less the energy of the anti-Hermitian part of those columns,
// which the reference's Parseval sum counts and no real image carries.
//
//   render_cols_kernel<N> / render_rows_kernel<N>   fused edges: Lay<N> packed spectrum -> kx inverse (complex,
//                                                   per ky column) -> global scratch [item][x][N/2+1] -> c2r rows,
//                                                   two real rows per complex transform -> shifted, scaled image
//   gen_render_cols_kernel / gen_render_rows_kernel other edges: the same two passes as direct DFTs (reference layout)
#pragma once
#include "bioem_kernels.cuh"

namespace bioem
{

// one calculated image: conv spectrum slot of the batch, image slot of the batch's output, circular shift in [0, N),
// scale and offset
struct RenderItem
{
  int slot, out, sx, sy;
  float norm, mu;
};

// inverse transform along kx of columns [ky0, ky0 + KC) of one packed spectrum -> scratch[item][x][ky] (row-major,
// N/2+1 complex per row): the mirror of fft_cols_kernel, same split N = R1 * R2, twiddles exp(+2 pi i n2 k1 / N)
template <int N>
__global__ void __launch_bounds__(NT) render_cols_kernel(const float4 *__restrict__ convs, const RenderItem *__restrict__ items,
                                                         const float2 *__restrict__ tw_inv, float2 *__restrict__ scratch)
{
  using L = Lay<N>;
  constexpr int R1 = L::R1, R2 = L::R2, KC = L::FKC;
  constexpr int NC1 = N / 2 + 1;
  extern __shared__ __align__(16) unsigned char smem_rcols[];
  float2 *E = reinterpret_cast<float2 *>(smem_rcols); // [KC * N]
  float2 *TW = E + KC * N;                            // [N]
  const int tid = threadIdx.x;
  const int img = blockIdx.y;
  const int ky0 = blockIdx.x * KC;
  const int ncol = min(KC, NC1 - ky0);
  for (int i = tid; i < N; i += NT)
    TW[i] = tw_inv[i];
  const float2 *src2 = reinterpret_cast<const float2 *>(convs + (size_t) items[img].slot * L::MAP4);
  float2 *dst = scratch + (size_t) img * N * NC1;
  __syncthreads();
  for (int item = tid; item < R2 * KC; item += NT)
  {
    const int n2 = item / KC, kyl = item % KC;
    if (kyl < ncol)
    {
      const int ky = ky0 + kyl;
      float2 x[R1];
#pragma unroll
      for (int n1 = 0; n1 < R1; n1++)
      {
        // spectrum element kx = n1 * R2 + n2 of column ky in the packed layout
        const size_t f4 = ky < L::NCOL ? (size_t) L::main_idx(ky / L::KC, n1 / 2, n2, ky % L::KC)
                                       : (size_t) L::MAIN4 + (n1 / 2) * R2 + n2;
        x[n1] = src2[f4 * 2 + (n1 & 1)];
      }
      bfft::Dft<R1, 1>::run(x);
#pragma unroll
      for (int k1 = 1; k1 < R1; k1++)
        x[k1] = bfft::cmul(x[k1], TW[n2 * R1 + k1]);
#pragma unroll
      for (int k1 = 0; k1 < R1; k1++)
        E[(k1 * R2 + n2) * KC + kyl] = x[k1];
    }
  }
  __syncthreads();
  for (int item = tid; item < R1 * KC; item += NT)
  {
    const int k1 = item / KC, kyl = item % KC;
    if (kyl < ncol)
    {
      float2 y[R2];
#pragma unroll
      for (int n2 = 0; n2 < R2; n2++)
        y[n2] = E[(k1 * R2 + n2) * KC + kyl];
      bfft::Dft<R2, 1>::run(y);
#pragma unroll
      for (int k2 = 0; k2 < R2; k2++)
        dst[(size_t) (k1 + R1 * k2) * NC1 + ky0 + kyl] = y[k2];
    }
  }
}

// c2r along y of rows [2 p0, 2 (p0 + PC)) of one item, two real rows per complex transform (the mirror of
// fft_rows_kernel's packing: Z[k] = A[k] + i B[k] over the full length, A and B extended by Hermitian symmetry, so
// the inverse of Z is a + i b), then the shift as an index remap and norm / mu at write-out
template <int N>
__global__ void __launch_bounds__(NT) render_rows_kernel(const float2 *__restrict__ scratch, const RenderItem *__restrict__ items,
                                                         const float2 *__restrict__ tw_inv, float *__restrict__ out)
{
  using L = Lay<N>;
  constexpr int R1 = L::R1, R2 = L::R2, PC = L::PC;
  constexpr int NPAIR = N / 2;
  constexpr int NC1 = N / 2 + 1;
  __shared__ float2 E[PC * N];
  __shared__ float2 TW[N];
  const int tid = threadIdx.x;
  const int img = blockIdx.y;
  const int p0 = blockIdx.x * PC;
  const int npl = min(PC, NPAIR - p0);
  for (int i = tid; i < N; i += NT)
    TW[i] = tw_inv[i];
  const float2 *src = scratch + (size_t) img * N * NC1;
  for (int i = tid; i < npl * N; i += NT)
  {
    const int pl = i / N, k = i % N;
    const float2 *ra = src + (size_t) (2 * (p0 + pl)) * NC1;
    const float2 *rb = ra + NC1;
    float2 a, b;
    if (k <= N / 2)
    {
      a = ra[k];
      b = rb[k];
      if (k == 0 || k == N / 2) // self-conjugate columns: their real part only
        a.y = b.y = 0.f;
    }
    else
    {
      a = ra[N - k];
      b = rb[N - k];
      a.y = -a.y;
      b.y = -b.y;
    }
    E[pl * N + k] = make_float2(a.x - b.y, a.y + b.x);
  }
  __syncthreads();
  // pass 1: length-R1 transforms over n1 (stride R2), twiddle, skewed store as fft_rows_kernel
  {
    const int pl = tid / R2, n2 = tid % R2;
    const bool act = pl < npl;
    float2 x[R1];
    if (act)
    {
#pragma unroll
      for (int n1 = 0; n1 < R1; n1++)
        x[n1] = E[pl * N + n1 * R2 + n2];
    }
    __syncthreads();
    if (act)
    {
      bfft::Dft<R1, 1>::run(x);
#pragma unroll
      for (int k1 = 1; k1 < R1; k1++)
        x[k1] = bfft::cmul(x[k1], TW[n2 * R1 + k1]);
#pragma unroll
      for (int k1 = 0; k1 < R1; k1++)
        E[pl * N + k1 * R2 + ((n2 + k1) % R2)] = x[k1];
    }
  }
  __syncthreads();
  // pass 2: length-R2 transforms, natural order (npl * R1 <= NT: one item per thread)
  {
    const int item = tid;
    const bool act = item < npl * R1;
    const int pl = act ? item / R1 : 0, k1 = act ? item % R1 : 0;
    float2 y[R2];
    if (act)
    {
#pragma unroll
      for (int n2 = 0; n2 < R2; n2++)
        y[n2] = E[pl * N + k1 * R2 + ((n2 + k1) % R2)];
      bfft::Dft<R2, 1>::run(y);
    }
    __syncthreads();
    if (act)
    {
#pragma unroll
      for (int k2 = 0; k2 < R2; k2++)
        E[pl * N + k1 + R1 * k2] = y[k2];
    }
  }
  __syncthreads();
  const RenderItem it = items[img];
  const float invNN = 1.0f / (float) (N * N);
  float *o = out + (size_t) it.out * N * N;
  for (int i = tid; i < npl * N; i += NT)
  {
    const int pl = i / N, c = i % N;
    const int r = 2 * (p0 + pl);
    const float2 z = E[pl * N + c];
    int xr = r + it.sx;
    xr -= xr >= N ? N : 0;
    int xr1 = xr + 1;
    xr1 -= xr1 >= N ? N : 0;
    int yc = c + it.sy;
    yc -= yc >= N ? N : 0;
    o[(size_t) xr * N + yc] = __fmaf_rn(it.norm, __fmul_rn(z.x, invNN), it.mu);
    o[(size_t) xr1 * N + yc] = __fmaf_rn(it.norm, __fmul_rn(z.y, invNN), it.mu);
  }
  static_assert(PC * R2 <= NT && PC * R1 <= NT, "one item per thread in both passes");
}

#ifndef BIOEM_LIK_ONLY
// direct-DFT path, kx inverse: scratch[item][x][k1] = sum_k0 V[k0][k1] exp(+2 pi i k0 x / N); grid (x, item)
__global__ void __launch_bounds__(256) gen_render_cols_kernel(const float2 *__restrict__ convs, size_t S,
                                                              const RenderItem *__restrict__ items, const float2 *__restrict__ tw,
                                                              int N, float2 *__restrict__ scratch)
{
  extern __shared__ float2 g_sm[];
  float2 *TW = g_sm; // [N]
  const int NC = N / 2 + 1;
  const int img = blockIdx.y, x = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < N; i += blockDim.x)
    TW[i] = tw[i];
  __syncthreads();
  const float2 *V = convs + (size_t) items[img].slot * S;
  for (int k1 = tid; k1 < NC; k1 += blockDim.x)
  {
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int k0 = 0; k0 < N; k0++)
    {
      const float2 w = TW[idx], v = V[(size_t) k0 * NC + k1];
      re += v.x * w.x - v.y * w.y;
      im += v.x * w.y + v.y * w.x;
      idx += x;
      if (idx >= N)
        idx -= N;
    }
    scratch[((size_t) img * N + x) * NC + k1] = make_float2(re, im);
  }
}

// direct-DFT path, c2r along y: R0[x][y] = sum_k1 w(k1) Re(T[x][k1] exp(+2 pi i k1 y / N)) / N^2 with w = 1 for the
// self-conjugate columns and 2 otherwise (as gen_corr_kernel), shifted, scaled; grid (x, item)
__global__ void __launch_bounds__(256) gen_render_rows_kernel(const float2 *__restrict__ scratch, const RenderItem *__restrict__ items,
                                                              const float2 *__restrict__ tw, int N, float *__restrict__ out)
{
  extern __shared__ float2 g_sm[];
  const int NC = N / 2 + 1;
  float2 *TW = g_sm;    // [N]
  float2 *T = g_sm + N; // [NC]
  const int img = blockIdx.y, x = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < N; i += blockDim.x)
    TW[i] = tw[i];
  for (int i = tid; i < NC; i += blockDim.x)
    T[i] = scratch[((size_t) img * N + x) * NC + i];
  __syncthreads();
  const RenderItem it = items[img];
  const float invNN = 1.0f / (float) (N * N);
  int xr = x + it.sx;
  xr -= xr >= N ? N : 0;
  float *o = out + ((size_t) it.out * N + xr) * N;
  for (int y = tid; y < N; y += blockDim.x)
  {
    float s = 0.f;
    int idx = 0;
    for (int k1 = 0; k1 < NC; k1++)
    {
      const float2 t = T[k1], w = TW[idx];
      const float term = t.x * w.x - t.y * w.y;
      s += (k1 == 0 || 2 * k1 == N) ? term : 2.f * term;
      idx += y;
      if (idx >= N)
        idx -= N;
    }
    int yc = y + it.sy;
    yc -= yc >= N ? N : 0;
    o[yc] = __fmaf_rn(it.norm, __fmul_rn(s, invNN), it.mu);
  }
}
#endif // BIOEM_LIK_ONLY

} // namespace bioem
