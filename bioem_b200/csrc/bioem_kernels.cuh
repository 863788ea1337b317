// sm_100a kernels for the BioEM likelihood path.
//
//   stage 1  project_kernel        createProjection        (reference bioem.cpp:1604-1818)
//            fft_rows_kernel /     forward r2c 2-D FFT     (reference bioem.cpp:1848)
//            fft_cols_kernel
//   stage 2  ctf_conv_kernel       createConvolutedProjectionMap (bioem.cpp:1855-1923)
//   stage 3-5 likelihood_kernel    calculateCCFFT + doRefMapFFT + calProb, fused
//                                  (bioem.cpp:1435-1459, bioem_algorithm.h:18-198)
//            merge_partials_kernel / finalize_kernel
//
// Data layout in HBM ("packed half-spectrum"): a real N x N image has the
// half-spectrum A[kx][ky], kx < N, ky <= N/2.  With N = R1*R2 (bfft::Geo<N>),
// NCOL = N/2 and KC columns per chunk, element (kx = n1*R2 + n2, ky = ch*KC + kyl)
// with ky < NCOL lives in float4 number
//      ((ch*(R1/2) + n1/2)*KC + kyl)*R2 + n2 ,   .xy if n1 even, .zw if n1 odd,
// i.e. exactly the order in which the column pass of the fused kernel reads it
// (lane = kyl*R2 + n2: one fully coalesced LDG.128 per thread per two points).  The Nyquist column
// ky = N/2 is a tail of N/2 float4: tail[(n1/2)*R2 + n2].
#pragma once
#include "fft_regs.cuh"
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace bioem
{

constexpr int NT = 256; // threads per CTA for the FFT kernels

constexpr int largest_divisor_leq(int n, int lim)
{
  int best = 1;
  for (int d = 1; d <= lim; d++)
    if (n % d == 0)
      best = d;
  return best;
}

template <int N> struct Lay
{
  using G = bfft::Geo<N>;
  static constexpr int R1 = G::R1, R2 = G::R2, PC = G::PC;
  static constexpr int NCOL = N / 2;
  // columns per chunk of the packed layout = columns one warp transforms at a time in the
  // fused kernel (lanes = R2 sub-sequences x KC columns)
  static constexpr int KC = largest_divisor_leq(NCOL, (32 / R2) > 0 ? (32 / R2) : 1);
  static constexpr int FKC = G::KC; // columns per CTA chunk of the forward column-FFT kernel
  static constexpr int NCH = NCOL / KC;
  static constexpr int MAIN4 = NCOL * N / 2;
  static constexpr int TAIL4 = N / 2;
  static constexpr int MAP4 = MAIN4 + TAIL4;
  static_assert(PC * R2 <= NT && PC * R1 <= NT, "row-pass chunk must fit one item per thread");
  __host__ __device__ static constexpr int main_idx(int ch, int n1p, int n2, int kyl)
  {
    return ((ch * (R1 / 2) + n1p) * KC + kyl) * R2 + n2;
  }
  // inverse of main_idx / of the tail numbering: float4 index i -> (n1p, n2, ky)
  __host__ __device__ static void decode(int i, int &n1p, int &n2, int &ky)
  {
    if (i < MAIN4)
    {
      n2 = i % R2;
      int t = i / R2;
      const int kyl = t % KC;
      t /= KC;
      n1p = t % (R1 / 2);
      ky = (t / (R1 / 2)) * KC + kyl;
    }
    else
    {
      const int t = i - MAIN4;
      n2 = t % R2;
      n1p = t / R2;
      ky = NCOL;
    }
  }
};

struct ConvParam
{
  float sumC;
  float sumsqC;
  double Bterm; // (Nt/2-2)*log((Nt-2)*ForLogProb) - prior(c)   (bioem_algorithm.h:42-67)
};

// best-so-far record of one image (bioem_Probability_map + what is needed to
// finish norm/mu later)
struct Running
{
  double Const;
  double Total;
  float lpf; // float-narrowed logpro of the current maximum
  int orient;
  int conv;
  int lin; // displacement enumeration index wx*nw + wy
  float v; // correlation value at the maximum
  float sumC;
  float sumsqC;
  int pad;
};

struct ProbMapOut // == bioem_Probability_map, include/map.h:116-129 (40 bytes)
{
  double Total;
  double Constoadd;
  int max_prob_cent_x, max_prob_cent_y, max_prob_orient, max_prob_conv;
  float max_prob_norm, max_prob_mu;
};
struct ProbAngleOut // == bioem_Probability_angle, include/map.h:131-135
{
  double forAngles;
  double ConstAngle;
};

constexpr double kMinProb = -999999.; // defs.h:65

__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }

// ===========================================================================
// layout conversion: standard [N][N/2+1] interleaved complex <-> packed
// ===========================================================================
template <int N>
__global__ void pack_kernel(const float2 *__restrict__ std_maps, float4 *__restrict__ packed, int nmaps)
{
  using L = Lay<N>;
  const int map = blockIdx.y;
  if (map >= nmaps)
    return;
  const float2 *src = std_maps + (size_t) map * N * (N / 2 + 1);
  float4 *dst = packed + (size_t) map * L::MAP4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L::MAP4; i += gridDim.x * blockDim.x)
  {
    int n1p, n2, ky;
    L::decode(i, n1p, n2, ky);
    const int kx0 = (2 * n1p) * L::R2 + n2, kx1 = (2 * n1p + 1) * L::R2 + n2;
    float2 a = src[(size_t) kx0 * (N / 2 + 1) + ky], b = src[(size_t) kx1 * (N / 2 + 1) + ky];
    dst[i] = make_float4(a.x, a.y, b.x, b.y);
  }
}

template <int N>
__global__ void unpack_kernel(const float4 *__restrict__ packed, float2 *__restrict__ std_maps, int nmaps)
{
  using L = Lay<N>;
  const int map = blockIdx.y;
  if (map >= nmaps)
    return;
  float2 *dst = std_maps + (size_t) map * N * (N / 2 + 1);
  const float4 *src = packed + (size_t) map * L::MAP4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L::MAP4; i += gridDim.x * blockDim.x)
  {
    int n1p, n2, ky;
    L::decode(i, n1p, n2, ky);
    const int kx0 = (2 * n1p) * L::R2 + n2, kx1 = (2 * n1p + 1) * L::R2 + n2;
    float4 v = src[i];
    dst[(size_t) kx0 * (N / 2 + 1) + ky] = make_float2(v.x, v.y);
    dst[(size_t) kx1 * (N / 2 + 1) + ky] = make_float2(v.z, v.w);
  }
}

// ===========================================================================
// stage 1a: projection (rotate, rasterise).  One CTA per (orientation, band of
// image rows); the band lives in shared memory; inside the CTA every warp owns a
// contiguous sub-band and walks ALL model points in order, so each pixel receives
// its contributions in model-point order exactly like the reference's sequential
// loop (deterministic, no atomics).  FP32 operations are written with explicit
// round-to-nearest intrinsics in the reference's evaluation order so that the
// pixel a point lands on and the weight it adds are those of the CPU code.
// ===========================================================================
struct ProjParams
{
  const float4 *xyzr; // model points: x, y, z, radius
  const float *dens;  // density
  const float4 *angles;
  float *proj;      // [OB][N*N]
  double *tempden;  // [OB][nbands]
  int *skipped;     // [O] points out of frame per orientation (absolute index), optional
  int A;
  int N;
  int band_rows;
  int nbands;
  int o_base; // first orientation of the batch (index into angles)
  int doquater;
  int shiftX, shiftY;
  float pixelSize;
};

#ifndef BIOEM_LIK_ONLY // non-template kernels: defined once, in bioem_b200.cu
__global__ void __launch_bounds__(256) project_kernel(ProjParams p)
{
  extern __shared__ float band[]; // band_rows * N
  const int N = p.N;
  const int ob = blockIdx.x, b = blockIdx.y;
  const int r0 = b * p.band_rows;
  const int r1 = min(N, r0 + p.band_rows);
  const int rows = r1 - r0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  for (int i = tid; i < rows * N; i += blockDim.x)
    band[i] = 0.f;

  // rotation matrix, reference evaluation order (bioem.cpp:1638-1672)
  const float4 q = p.angles[p.o_base + ob];
  float m00, m01, m02, m10, m11, m12;
  if (p.doquater)
  {
    const float q0 = q.x, q1 = q.y, q2 = q.z, q3 = q.w;
    m00 = __fsub_rn(__fsub_rn(1.f, __fmul_rn(__fmul_rn(2.f, q1), q1)), __fmul_rn(__fmul_rn(2.f, q2), q2));
    m10 = __fmul_rn(2.f, __fsub_rn(__fmul_rn(q0, q1), __fmul_rn(q2, q3)));
    m01 = __fmul_rn(2.f, __fadd_rn(__fmul_rn(q0, q1), __fmul_rn(q2, q3)));
    m11 = __fsub_rn(__fsub_rn(1.f, __fmul_rn(__fmul_rn(2.f, q0), q0)), __fmul_rn(__fmul_rn(2.f, q2), q2));
    m02 = __fmul_rn(2.f, __fsub_rn(__fmul_rn(q0, q2), __fmul_rn(q1, q3)));
    m12 = __fmul_rn(2.f, __fadd_rn(__fmul_rn(q1, q2), __fmul_rn(q0, q3)));
  }
  else
  {
    const float al = q.x, be = q.y, ga = q.z;
    const float ca = cosf(al), sa = sinf(al), cb = cosf(be), sb = sinf(be), cg = cosf(ga), sg = sinf(ga);
    m00 = __fsub_rn(__fmul_rn(cg, ca), __fmul_rn(__fmul_rn(cb, sa), sg));
    m01 = __fadd_rn(__fmul_rn(cg, sa), __fmul_rn(__fmul_rn(cb, ca), sg));
    m02 = __fmul_rn(sg, sb);
    m10 = __fsub_rn(__fmul_rn(-sg, ca), __fmul_rn(__fmul_rn(cb, sa), cg));
    m11 = __fadd_rn(__fmul_rn(-sg, sa), __fmul_rn(__fmul_rn(cb, ca), cg));
    m12 = __fmul_rn(cg, sb);
  }
  __syncthreads();

  // this warp's rows
  const int h = (rows + nwarps - 1) / nwarps;
  const int wr0 = r0 + warp * h;
  const int wr1 = min(r1, wr0 + h);
  const float px = p.pixelSize;
  const float half = __fdiv_rn((float) N, 2.0f);
  float td = 0.f; // per-lane share of tempden
  int nskip = 0;
  // Model points are taken in tiles of PT.  Phase A: warp w rotates the points [w*SEG, (w+1)*SEG) of the tile, 32
  // consecutive points per trip, and keeps -- in order, compacted with a ballot -- only those whose footprint
  // touches THIS CTA's band of rows (s_pt[w*SEG ..], s_cnt[w]); with a 48^3 voxel model that is ~3 % of the
  // 110,592 points.  Phase B: every warp walks the kept points of all segments in order, 32 at a time: one ballot
  // tells which of them touch the warp's own rows, and only those are rasterised, lowest index first -- the order
  // of the reference's loop over the model points, so every pixel receives its contributions in model order
  // (deterministic, no atomics).
  constexpr int PT = 1024;
  __shared__ int4 s_pt[PT]; // i, j, radius bits, density bits
  __shared__ int s_cnt[8];
  const int SEG = PT / nwarps; // nwarps is 1, 2, 4 or 8
  for (int n0 = 0; n0 < p.A; n0 += PT)
  {
    int cnt = 0;
    for (int kk = 0; kk < SEG; kk += 32)
    {
      const int k = warp * SEG + kk + lane;
      bool keep = false, out = false;
      int4 e = make_int4(0, 0, 0, 0);
      if (n0 + k < p.A)
      {
        const float4 pt = __ldg(&p.xyzr[n0 + k]);
        const float den = __ldg(&p.dens[n0 + k]);
        const float rx = __fadd_rn(__fadd_rn(__fadd_rn(0.f, __fmul_rn(m00, pt.x)), __fmul_rn(m01, pt.y)), __fmul_rn(m02, pt.z));
        const float ry = __fadd_rn(__fadd_rn(__fadd_rn(0.f, __fmul_rn(m10, pt.x)), __fmul_rn(m11, pt.y)), __fmul_rn(m12, pt.z));
        int i = (int) floorf(__fadd_rn(__fadd_rn(__fdiv_rn(rx, px), half), 0.5f));
        int j = (int) floorf(__fadd_rn(__fadd_rn(__fdiv_rn(ry, px), half), 0.5f));
        const float radius = pt.w;
        if (radius <= px)
        {
          out = i < 0 || j < 0 || i >= N || j >= N;
          keep = !out && i >= r0 && i < r1;
        }
        else
        {
          i -= p.shiftX;
          j -= p.shiftY;
          const int irad = (int) __fdiv_rn(radius, px) + 1;
          out = i < irad || j < irad || i >= N - irad || j >= N - irad;
          keep = !out && !(i + irad < r0 || i - irad >= r1);
        }
        e = make_int4(i, j, __float_as_int(radius), __float_as_int(den));
      }
      nskip += __popc(__ballot_sync(0xffffffffu, out));
      const unsigned km = __ballot_sync(0xffffffffu, keep);
      if (keep)
        s_pt[warp * SEG + cnt + __popc(km & ((1u << lane) - 1u))] = e;
      cnt += __popc(km);
    }
    if (lane == 0)
      s_cnt[warp] = cnt;
    __syncthreads();
    for (int ws = 0; ws < nwarps; ws++)
    {
      const int nt = s_cnt[ws];
      for (int k0 = 0; k0 < nt; k0 += 32)
      {
        int4 e = make_int4(0, 0, 0, 0);
        bool hit = false;
        if (k0 + lane < nt)
        {
          e = s_pt[ws * SEG + k0 + lane];
          const float radius = __int_as_float(e.z);
          if (radius <= px)
            hit = e.x >= wr0 && e.x < wr1;
          else
          {
            const int irad = (int) __fdiv_rn(radius, px) + 1;
            hit = !(e.x + irad < wr0 || e.x - irad >= wr1);
          }
        }
        unsigned todo = __ballot_sync(0xffffffffu, hit);
        while (todo)
        {
          const int src = __ffs(todo) - 1;
          todo &= todo - 1;
          const int i = __shfl_sync(0xffffffffu, e.x, src), j = __shfl_sync(0xffffffffu, e.y, src);
          const float radius = __int_as_float(__shfl_sync(0xffffffffu, e.z, src));
          const float den = __int_as_float(__shfl_sync(0xffffffffu, e.w, src));
          if (radius <= px)
          {
            if (lane == 0)
            {
              band[(i - r0) * N + j] = __fadd_rn(band[(i - r0) * N + j], den);
              td = __fadd_rn(td, den);
            }
          }
          else
          {
            const int irad = (int) __fdiv_rn(radius, px) + 1;
            const float rad2 = __fmul_rn(radius, radius);
            const int S = 2 * irad + 1;
            const double denom = 4 * 3.14159265358979323846 * (double) radius * (double) rad2;
            // lanes cover only the footprint rows this warp owns (one trip for the usual 7 x 7 footprint of a
            // voxel model and a warp of one to four rows), in the reference's ii-outer / jj-inner order
            const int d_lo = max(-irad, wr0 - i), d_hi = min(irad, wr1 - 1 - i);
            const int cells = (d_hi - d_lo + 1) * S;
            for (int idx = lane; idx < cells; idx += 32)
            {
              const int di = idx / S + d_lo, dj = idx % S - irad;
              const int ii = i + di, jj = j + dj;
              // dist = ((float)(di)*di + dj*dj) * px * px
              const float dist = __fmul_rn(__fmul_rn(__fadd_rn(__fmul_rn((float) di, (float) di), (float) (dj * dj)), px), px);
              if (dist < rad2)
              {
                const float num = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(px, px), 2.f), sqrtf(__fsub_rn(rad2, dist))), den), 3.f);
                const double w = (double) num / denom;
                float *px_ = &band[(ii - r0) * N + jj];
                *px_ = (float) ((double) *px_ + w);
                td = (float) ((double) td + w);
              }
            }
          }
          // the next point may touch the same pixels from other lanes: order the read-modify-writes
          __syncwarp();
        }
      }
    }
    __syncthreads();
  }
  __syncthreads();
  float *out = p.proj + (size_t) ob * N * N + (size_t) r0 * N;
  for (int i = tid; i < rows * N; i += blockDim.x)
    out[i] = band[i];
  // deterministic reduction of the tempden shares: lanes then warps, fixed order
  __shared__ float s_td[256];
  s_td[tid] = td;
  if (lane == 0)
    s_cnt[warp] = nskip; // out-of-frame points of the segments this warp rotated
  __syncthreads();
  if (tid == 0)
  {
    double t = 0.0;
    for (int k = 0; k < (int) blockDim.x; k++)
      t += (double) s_td[k];
    p.tempden[(size_t) ob * p.nbands + b] = t;
    if (p.skipped && b == 0)
    {
      int ns = 0;
      for (int w = 0; w < nwarps; w++)
        ns += s_cnt[w];
      p.skipped[p.o_base + ob] = ns; // every band rotates the whole model: band 0 reports
    }
  }
}

#endif // BIOEM_LIK_ONLY

// ===========================================================================
// stage 1b: forward 2-D r2c FFT of real images -> packed half-spectrum.
// rows pass (two real rows per complex transform) to a row-major scratch
// [img][N][N/2+1], then column pass into the packed layout.
// scale[img] (optional): multiply the image by NormDen / sum_b tempden[img][b]
// (bioem.cpp:1808-1818) while loading.
// ===========================================================================
template <int N>
__global__ void __launch_bounds__(NT) fft_rows_kernel(const float *__restrict__ imgs, const double *__restrict__ tempden,
                                                      int nbands, float normDen, const float2 *__restrict__ tw_fwd,
                                                      float2 *__restrict__ scratch)
{
  using L = Lay<N>;
  constexpr int R1 = L::R1, R2 = L::R2, PC = L::PC;
  constexpr int NPAIR = N / 2;
  __shared__ float2 E[PC * N];
  __shared__ float2 TW[N];
  const int tid = threadIdx.x;
  const int img = blockIdx.y;
  const int p0 = blockIdx.x * PC;
  const int npl = min(PC, NPAIR - p0);
  for (int i = tid; i < N; i += NT)
    TW[i] = tw_fwd[i];
  float scale = 1.f;
  if (tempden)
  {
    double t = 0.0;
    for (int b = 0; b < nbands; b++)
      t += tempden[(size_t) img * nbands + b];
    scale = __fdiv_rn(normDen, (float) t);
  }
  const float *src = imgs + (size_t) img * N * N;
  __syncthreads();
  // pass 1
  {
    const int pl = tid / R2, n2 = tid % R2;
    if (pl < npl)
    {
      const float *ra = src + (size_t) (2 * (p0 + pl)) * N;
      const float *rb = ra + N;
      float2 x[R1];
#pragma unroll
      for (int n1 = 0; n1 < R1; n1++)
        x[n1] = make_float2(__fmul_rn(ra[n1 * R2 + n2], scale), __fmul_rn(rb[n1 * R2 + n2], scale));
      bfft::Dft<R1, -1>::run(x);
#pragma unroll
      for (int k1 = 1; k1 < R1; k1++)
        x[k1] = bfft::cmul(x[k1], TW[n2 * R1 + k1]);
#pragma unroll
      for (int k1 = 0; k1 < R1; k1++)
        E[pl * N + k1 * R2 + ((n2 + k1) % R2)] = x[k1];
    }
  }
  __syncthreads();
  // pass 2 (results kept in registers across the barrier, then written back in natural order)
  for (int base = 0; base < npl * R1; base += NT)
  {
    const int item = base + tid;
    const bool act = item < npl * R1;
    const int pl = act ? item / R1 : 0, k1 = act ? item % R1 : 0;
    float2 y[R2];
    if (act)
    {
#pragma unroll
      for (int n2 = 0; n2 < R2; n2++)
        y[n2] = E[pl * N + k1 * R2 + ((n2 + k1) % R2)];
      bfft::Dft<R2, -1>::run(y);
    }
    __syncthreads();
    if (act)
    {
#pragma unroll
      for (int k2 = 0; k2 < R2; k2++)
        E[pl * N + k1 + R1 * k2] = y[k2];
    }
    // (npl*R1 <= NT always holds for the shipped geometries, so one trip)
  }
  __syncthreads();
  // separate the two real rows: A = (Z[k] + conj Z[N-k])/2, B = (Z[k] - conj Z[N-k])/(2i)
  float2 *dst = scratch + (size_t) img * N * (N / 2 + 1);
  for (int i = tid; i < npl * (N / 2 + 1); i += NT)
  {
    const int pl = i / (N / 2 + 1), k = i % (N / 2 + 1);
    const float2 z = E[pl * N + k], zc = E[pl * N + ((N - k) % N)];
    const float2 a = make_float2(0.5f * (z.x + zc.x), 0.5f * (z.y - zc.y));
    const float2 bb = make_float2(0.5f * (z.y + zc.y), -0.5f * (z.x - zc.x));
    dst[(size_t) (2 * (p0 + pl)) * (N / 2 + 1) + k] = a;
    dst[(size_t) (2 * (p0 + pl) + 1) * (N / 2 + 1) + k] = bb;
  }
}

template <int N>
__global__ void __launch_bounds__(NT) fft_cols_kernel(const float2 *__restrict__ scratch, const float2 *__restrict__ tw_fwd,
                                                      float4 *__restrict__ packed)
{
  using L = Lay<N>;
  constexpr int R1 = L::R1, R2 = L::R2, KC = L::FKC;
  constexpr int NC1 = N / 2 + 1;
  extern __shared__ __align__(16) unsigned char smem_cols[];
  float2 *E = reinterpret_cast<float2 *>(smem_cols); // [KC * N]
  float2 *TW = E + KC * N;                           // [N]
  const int tid = threadIdx.x;
  const int img = blockIdx.y;
  const int ky0 = blockIdx.x * KC; // chunks cover ky = 0 .. N/2 (the last one may be partial)
  const int ncol = min(KC, NC1 - ky0);
  for (int i = tid; i < N; i += NT)
    TW[i] = tw_fwd[i];
  const float2 *src = scratch + (size_t) img * N * NC1;
  float2 *dst2 = reinterpret_cast<float2 *>(packed + (size_t) img * L::MAP4);
  __syncthreads();
  for (int item = tid; item < R2 * KC; item += NT)
  {
    const int n2 = item / KC, kyl = item % KC;
    if (kyl < ncol)
    {
      float2 x[R1];
#pragma unroll
      for (int n1 = 0; n1 < R1; n1++)
        x[n1] = src[(size_t) (n1 * R2 + n2) * NC1 + ky0 + kyl];
      bfft::Dft<R1, -1>::run(x);
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
      bfft::Dft<R2, -1>::run(y);
      const int ky = ky0 + kyl;
#pragma unroll
      for (int k2 = 0; k2 < R2; k2++)
      {
        const int kx = k1 + R1 * k2;
        const int n1 = kx / R2, m2 = kx % R2;
        size_t f4;
        if (ky < L::NCOL)
          f4 = (size_t) L::main_idx(ky / L::KC, n1 / 2, m2, ky % L::KC);
        else
          f4 = (size_t) L::MAIN4 + (n1 / 2) * R2 + m2;
        dst2[f4 * 2 + (n1 & 1)] = y[k2];
      }
    }
  }
}

#ifndef BIOEM_LIK_ONLY // non-template kernels: defined once, in bioem_b200.cu
// per-image sum and sum of squares, strictly sequential float accumulation in
// row-major order like the reference (bioem.cpp:2087-2107); one-off input prep.
__global__ void image_sums_kernel(const float *__restrict__ imgs, int n2, int M, float *__restrict__ sum,
                                  float *__restrict__ sumsq)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  const float *p = imgs + (size_t) m * n2;
  float s = 0.f, ss = 0.f;
  for (int i = 0; i < n2; i++)
  {
    const float v = p[i];
    s = __fadd_rn(s, v);
    ss = __fadd_rn(ss, __fmul_rn(v, v));
  }
  sum[m] = s;
  sumsq[m] = ss;
}

// MRC particle ingest (reference map.cpp:811-845): per-image mean and deviation accumulated in
// FILE order with float accumulators (sequential, like the reader's loop), then the image is
// stored transposed (maps[i*N + j] = file[j*N + i]) and, unless NO_MAP_NORM, scaled to zero mean
// / unit deviation with the reference's expression  x / st2 - st / st2.
__global__ void mrc_stats_kernel(const float *__restrict__ raw, int n2, int M, float *__restrict__ mean,
                                 float *__restrict__ dev)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  const float *p = raw + (size_t) m * n2;
  float st = 0.f, st2 = 0.f;
  for (int i = 0; i < n2; i++)
  {
    const float v = p[i];
    st = __fadd_rn(st, v);
    st2 = __fadd_rn(st2, __fmul_rn(v, v));
  }
  st = __fdiv_rn(st, (float) n2);
  st2 = __fsqrt_rn(__fsub_rn(__fdiv_rn(st2, (float) n2), __fmul_rn(st, st)));
  mean[m] = st;
  dev[m] = st2;
}

__global__ void mrc_transpose_kernel(const float *__restrict__ raw, const float *__restrict__ mean,
                                     const float *__restrict__ dev, int N, int normalise, float *__restrict__ maps)
{
  __shared__ float tile[32][33];
  const int m = blockIdx.z;
  const float *src = raw + (size_t) m * N * N;
  float *dst = maps + (size_t) m * N * N;
  const int j0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y)
  {
    const int j = j0 + r, i = i0 + threadIdx.x;
    if (j < N && i < N)
      tile[r][threadIdx.x] = src[(size_t) j * N + i];
  }
  __syncthreads();
  const float st = normalise ? mean[m] : 0.f, st2 = normalise ? dev[m] : 1.f;
  for (int r = threadIdx.y; r < 32; r += blockDim.y)
  {
    const int i = i0 + r, j = j0 + threadIdx.x;
    if (i < N && j < N)
    {
      const float v = tile[threadIdx.x][r];
      dst[(size_t) i * N + j] = normalise ? __fsub_rn(__fdiv_rn(v, st2), __fdiv_rn(st, st2)) : v;
    }
  }
}

#endif // BIOEM_LIK_ONLY

// ===========================================================================
// stage 2: V = P * conj(K_c) on packed maps, sumC, sumsquareC, and the
// displacement-independent part of the log-posterior.
// ===========================================================================
template <int N>
__global__ void __launch_bounds__(NT) ctf_conv_kernel(const float4 *__restrict__ proj, const float4 *__restrict__ ctf,
                                                      const double *__restrict__ prior, float4 *__restrict__ conv,
                                                      ConvParam *__restrict__ cpar, int C, float Ntotpi,
                                                      const int4 *__restrict__ sel)
{
  using L = Lay<N>;
  // regular launch: grid (C, orientations of the batch), output slot ob*C + c.  With a selection list (exact
  // arg-max pass): grid (1, items), item b convolves projection sel[b].y with CTF sel[b].z into slot b.
  const int tid = threadIdx.x;
  const int c = sel ? sel[blockIdx.y].z : blockIdx.x;
  const int ob = sel ? sel[blockIdx.y].y : blockIdx.y;
  const size_t oslot = sel ? (size_t) blockIdx.y : (size_t) ob * C + c;
  const float4 *P = proj + (size_t) ob * L::MAP4;
  const float4 *K = ctf + (size_t) c * L::MAP4;
  // (conv == nullptr: cached-product mode of the fused kernel, which never reads a convolved spectrum -- only
  // sumC, sumsquareC and the displacement-independent term are needed)
  float4 *V = conv ? conv + oslot * L::MAP4 : nullptr;
  float acc = 0.f;
  float sumC = 0.f;
  for (int i = tid; i < L::MAP4; i += NT)
  {
    const float4 a = P[i], k = K[i];
    float4 v;
    v.x = a.x * k.x + a.y * k.y;
    v.y = a.y * k.x - a.x * k.y;
    v.z = a.z * k.z + a.w * k.w;
    v.w = a.w * k.z - a.z * k.w;
    // Hermitian weights (bioem.cpp:1893-1914): 1 for ky = 0 and ky = N/2, else 2
    float w = 2.f;
    const bool tail = i >= L::MAIN4;
    int n1p, n2, ky;
    L::decode(i, n1p, n2, ky);
    const bool dc = ky == 0;
    if (tail || dc)
      w = 1.f;
    float4 vs = v;
    if (conv && (tail || dc))
    {
      // The reference's CTF table is not Hermitian along kx (quirk Q1), so neither is V in
      // the two self-conjugate columns ky = 0 and ky = N/2.  A c2r transform (FFTW) only sees
      // the Hermitian part of these columns: Re of their kx-transform.  Store that part,
      // V_sym[kx] = (V[kx] + conj V[-kx]) / 2, so that the fused kernel can pack the two
      // columns into one complex transform.  sumC / sumsquareC use the unsymmetrised V.
      float pv[4];
#pragma unroll
      for (int e = 0; e < 2; e++)
      {
        const int kx = (2 * n1p + e) * L::R2 + n2;
        const int kxp = (N - kx) % N;
        const int m1 = kxp / L::R2, m2 = kxp % L::R2;
        const int ip = tail ? L::MAIN4 + (m1 / 2) * L::R2 + m2 : L::main_idx(0, m1 / 2, m2, 0);
        const float4 ap = P[ip], kp = K[ip];
        if (m1 & 1)
        {
          pv[2 * e] = ap.z * kp.z + ap.w * kp.w;
          pv[2 * e + 1] = ap.w * kp.z - ap.z * kp.w;
        }
        else
        {
          pv[2 * e] = ap.x * kp.x + ap.y * kp.y;
          pv[2 * e + 1] = ap.y * kp.x - ap.x * kp.y;
        }
      }
      vs.x = 0.5f * (v.x + pv[0]);
      vs.y = 0.5f * (v.y - pv[1]);
      vs.z = 0.5f * (v.z + pv[2]);
      vs.w = 0.5f * (v.w - pv[3]);
    }
    if (conv)
      V[i] = vs;
    acc += w * (v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w);
    if (i == 0)
      sumC = v.x; // kx = 0, ky = 0
  }
  __shared__ float red[NT];
  red[tid] = acc;
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1)
  {
    if (tid < s)
      red[tid] += red[tid + s];
    __syncthreads();
  }
  if (tid == 0)
  {
    const float ssC = __fdiv_rn(red[0], (float) (N * N));
    ConvParam cp;
    cp.sumC = sumC;
    cp.sumsqC = ssC;
    const float fl = __fsub_rn(__fmul_rn(ssC, Ntotpi), __fmul_rn(sumC, sumC));
    cp.Bterm = ((double) Ntotpi * 0.5 - 2.0) * log((double) __fsub_rn(Ntotpi, 2.f) * (double) fl) - prior[c];
    cpar[oslot] = cp;
  }
}

// Stage 2 of a grouped CTF table (cached-product mode, G x C rows): only sumC, sumsquareC and the B-term, for every
// (orientation, row) pair of the batch.  ctf_conv_kernel makes one pass over a projection and a table row per pair;
// here a CTA takes SUMS_CB rows x SUMS_OB orientations and loads every float4 of them once for all SUMS_CB x SUMS_OB
// pairs (the G x C rows do not fit L2; the table is read OBcur / SUMS_OB times per batch instead of OBcur times).
// Each pair's sum runs in exactly the order of ctf_conv_kernel (same per-thread stride, same tree), so cpar is
// bit-identical to what ctf_conv_kernel writes for the same row.  Output slot ob*GC + row.
constexpr int SUMS_CB = 4, SUMS_OB = 8;
template <int N>
__global__ void __launch_bounds__(NT) ctf_sums_kernel(const float4 *__restrict__ proj, const float4 *__restrict__ ctf,
                                                      const double *__restrict__ prior, ConvParam *__restrict__ cpar,
                                                      int GC, int OBcur, float Ntotpi)
{
  using L = Lay<N>;
  const int tid = threadIdx.x;
  const int c0 = blockIdx.x * SUMS_CB, o0 = blockIdx.y * SUMS_OB;
  const float4 *K[SUMS_CB];
  const float4 *P[SUMS_OB];
#pragma unroll
  for (int j = 0; j < SUMS_CB; j++)
    K[j] = ctf + (size_t) min(c0 + j, GC - 1) * L::MAP4; // (past the end: a valid row, never written out)
#pragma unroll
  for (int b = 0; b < SUMS_OB; b++)
    P[b] = proj + (size_t) min(o0 + b, OBcur - 1) * L::MAP4;
  __shared__ float red[SUMS_OB * SUMS_CB][NT];
  __shared__ float s_sumC[SUMS_OB * SUMS_CB]; // kx = 0, ky = 0 of every pair
  float acc[SUMS_OB][SUMS_CB];
#pragma unroll
  for (int b = 0; b < SUMS_OB; b++)
#pragma unroll
    for (int j = 0; j < SUMS_CB; j++)
      acc[b][j] = 0.f;
  for (int i = tid; i < L::MAP4; i += NT)
  {
    float w = 2.f;
    const bool tail = i >= L::MAIN4;
    int n1p, n2, ky;
    L::decode(i, n1p, n2, ky);
    if (tail || ky == 0)
      w = 1.f;
    float4 k[SUMS_CB];
#pragma unroll
    for (int j = 0; j < SUMS_CB; j++)
      k[j] = K[j][i];
#pragma unroll
    for (int b = 0; b < SUMS_OB; b++)
    {
      const float4 a = P[b][i];
#pragma unroll
      for (int j = 0; j < SUMS_CB; j++)
      {
        float4 v;
        v.x = a.x * k[j].x + a.y * k[j].y;
        v.y = a.y * k[j].x - a.x * k[j].y;
        v.z = a.z * k[j].z + a.w * k[j].w;
        v.w = a.w * k[j].z - a.z * k[j].w;
        acc[b][j] += w * (v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w);
        if (i == 0)
          s_sumC[b * SUMS_CB + j] = v.x;
      }
    }
  }
#pragma unroll
  for (int b = 0; b < SUMS_OB; b++)
#pragma unroll
    for (int j = 0; j < SUMS_CB; j++)
      red[b * SUMS_CB + j][tid] = acc[b][j];
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1)
  {
    if (tid < s)
#pragma unroll
      for (int q = 0; q < SUMS_OB * SUMS_CB; q++)
        red[q][tid] += red[q][tid + s];
    __syncthreads();
  }
  if (tid == 0)
#pragma unroll
    for (int b = 0; b < SUMS_OB; b++)
#pragma unroll
      for (int j = 0; j < SUMS_CB; j++)
      {
        const int c = c0 + j, ob = o0 + b;
        if (c >= GC || ob >= OBcur)
          continue;
        const float ssC = __fdiv_rn(red[b * SUMS_CB + j][0], (float) (N * N));
        const float sC = s_sumC[b * SUMS_CB + j];
        ConvParam cp;
        cp.sumC = sC;
        cp.sumsqC = ssC;
        const float fl = __fsub_rn(__fmul_rn(ssC, Ntotpi), __fmul_rn(sC, sC));
        cp.Bterm = ((double) Ntotpi * 0.5 - 2.0) * log((double) __fsub_rn(Ntotpi, 2.f) * (double) fl) - prior[c];
        cpar[(size_t) ob * GC + c] = cp;
      }
}

struct LikParams
{
  const float4 *convs; // [OBcur*C][MAP4]
  const float4 *refs;  // [M][MAP4]
  const ConvParam *cpar;
  const float *sumRef;
  const float *sumsqRef;
  const float2 *tw_inv;      // [N]  exp(+2 pi i n2*k1/N) at [n2*R1 + k1]
  const unsigned char *wtab; // [N]  window index of a raw displacement, 255 = outside
  Running *partials;         // [NG][M]
  ProbAngleOut *angles;      // [O][M] or null
  float *dbg_values;         // optional [OBcur*C][M][nw*nw] correlation values ([CTA][nw*nw] with pairs)
  // optional work list (exact arg-max pass): CTA b evaluates the single likelihood of particle pairs[b].x
  // against conv spectrum b of the batch (launched with C = 1, OG = 1: the spectra were gathered per item);
  // its partial goes to partials[b], its correlation window to dbg_values[b]
  const int4 *pairs;
  // cached-product mode (likelihood_kernel<N, W, true>, chosen by zmode != 0; needs REAL CTF kernels, i.e. CTFs given
  // in Fourier space, param.cpp:1540-1570): conv * conj(particle) = (projection * conj(particle)) * K_c.  The CTA
  // forms Z = projection * conj(particle) once per orientation into its private scratch map and streams Z and the
  // real table K_c per CTF: 3/4 of the operand bytes and half of the multiplies of the complex path.
  const float4 *projs; // [OBcur][MAP4] projection spectra of the batch
  const float4 *kreal; // [C][kr4] real CTF tables in column-pass order (KLay<N>)
  float4 *zbuf;        // [nslots][MAP4] scratch maps, one per resident CTA
  int *zflags;         // [nslots] 0 = free
  int nslots, kr4, zmode;
  int M, C, OBcur, OG, o_base;
  int nw;  // window points per axis
  int nwp; // nw rounded up to even
  float Ntotpi;
  float invNN;
  float ex2coef; // (3 - Nt)/2 * log2(e): sum of exp over the window runs in base 2
  double acoef_d;
  // grouped CTF table (likelihood_kernel<N, W, true, true>, chosen by group != nullptr; cached-product mode only):
  // kreal / cpar hold GC = G x C rows, particle m integrates over the C rows [group[m]*C, group[m]*C + C) of them;
  // CTA b takes particle perm[b % M] (particles ordered by group, so the resident CTAs share few groups' tables)
  const int *group; // [M]
  const int *perm;  // [M]
  int GC;
};

// Real CTF table of the cached-product mode, per CTF, in the order the column pass consumes it: lane
// (c, n2) of column chunk ch reads KQ float4 holding K(kx = n1*R2 + n2, ky = ch*KC + c) for n1 = 4q .. 4q+3 at
// [(ch*KQ + q)*KC*R2 + lane]; the Nyquist column follows as [MAINK4 + q*R2 + n2].  The two self-conjugate columns
// ky = 0 and N/2 hold (K(kx) + K(N-kx))/2: the c2r transform only sees the Hermitian part of these columns
// (quirk Q1, see ctf_conv_kernel), and for Hermitian projection / particle columns that part is Z * K_sym.
template <int N> struct KLay
{
  using L = Lay<N>;
  static constexpr int KQ = (L::R1 + 3) / 4;
  static constexpr int KCR2 = L::KC * L::R2;
  static constexpr int MAINK4 = L::NCH * KQ * KCR2;
  static constexpr int KR4 = MAINK4 + KQ * L::R2;
};

#ifndef BIOEM_LIK_ONLY
template <int N>
__global__ void kreal_kernel(const float4 *__restrict__ ctf, float4 *__restrict__ kreal, int C)
{
  using L = Lay<N>;
  using K = KLay<N>;
  const int c = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K::KR4 || c >= C)
    return;
  const float4 *T = ctf + (size_t) c * L::MAP4;
  int ch, q, n2, kyl;
  const bool tail = i >= K::MAINK4;
  if (!tail)
  {
    const int lane = i % K::KCR2;
    q = (i / K::KCR2) % K::KQ;
    ch = i / (K::KCR2 * K::KQ);
    kyl = lane / L::R2;
    n2 = lane % L::R2;
  }
  else
  {
    const int t = i - K::MAINK4;
    n2 = t % L::R2;
    q = t / L::R2;
    ch = 0;
    kyl = 0;
  }
  // real part of the table at (kx, this column)
  auto at = [&](int kx) {
    const int n1 = kx / L::R2, m2 = kx % L::R2;
    const float4 v = T[tail ? L::MAIN4 + (n1 / 2) * L::R2 + m2 : L::main_idx(ch, n1 / 2, m2, kyl)];
    return (n1 & 1) ? v.z : v.x;
  };
  const bool selfconj = tail || (ch == 0 && kyl == 0);
  float out[4];
#pragma unroll
  for (int e = 0; e < 4; e++)
  {
    const int n1 = 4 * q + e;
    float v = 0.f;
    if (n1 < L::R1)
    {
      const int kx = n1 * L::R2 + n2;
      v = at(kx);
      if (selfconj)
        v = 0.5f * (v + at((N - kx) % N));
    }
    out[e] = v;
  }
  kreal[(size_t) c * K::KR4 + i] = make_float4(out[0], out[1], out[2], out[3]);
}
#endif

// number of leading (= trailing) radix-R2 output groups that can hold a displacement of
// [-maxD, maxD]: raw index k = k1 + R1*k2, k <= maxD or k >= N - maxD
template <int N> __host__ __device__ constexpr int lik_window_groups(int maxD)
{
  using L = Lay<N>;
  constexpr int HALF = L::R2 / 2;
  if (L::G::GENERIC)
    return HALF; // rule-generated split: only the unpruned variant exists
  const int need = maxD / L::R1 + 1;
  return (need <= 7 && need < HALF) ? need : HALF;
}

// Shared-memory plan of the fused kernel (W = window groups, NK = kept radix-R2 outputs).
//   Y   [NK*R1][YS] float2: rows of the column-transformed spectrum that can hold window
//       displacements, row slot = j*R1 + k1 for raw row k1 + R1*k2(j).  After a row pair has been
//       consumed by the row pass its two slots are reused for the pair's firstele values
//       (FE, NK*R1 floats per window row).
//   E   per warp [R1][ES] float2: the exchange tile between the two radix passes
//   WT  [N] window table, RS [256] window row -> row slot
// Shared-memory geometry of the fused kernel (see LikSmem below) as free functions, so that the
// warp count can be chosen from it.
template <int N> struct LikGeo
{
  using L = Lay<N>;
  static constexpr int KC = L::KC;
  // Exchange tile E[k1][c][n2] (float2): pass 1 stores with lane = c*R2 + n2 at k1*ES + c*CS + n2
  // (contiguous per half warp), pass 2 loads with lane = k1*KC + c at the same address for
  // n2 = 0..R2-1: conflict-free when c*CS == c and k1*ES == k1*KC (mod 16 bank pairs).
  // With two columns of sixteen sub-sequences per warp (N = 128 .. 320) pass 2 loads pairs of
  // values as 128-bit words: c*CS and k1*ES are then multiples of two float2 whose halves run
  // through all eight 16-byte bank groups of a quarter warp (CS = 18, ES = 36).
  static constexpr bool WIDE = (KC == 2 && L::R2 == 16);
  static constexpr int CS = WIDE ? 18 : ((L::R2 - 1 + 15) / 16) * 16 + 1;
  static constexpr int ES = WIDE ? 36 : KC * CS + ((KC - KC * CS) % 16 + 16) % 16;
  static constexpr int YS0 = L::NCOL + ((KC - L::NCOL) % 16 + 16) % 16;
  static constexpr int YS = YS0 > L::NCOL ? YS0 : YS0 + 16; // index NCOL of a row must exist
  static constexpr int EW = L::R1 * ES;                     // float2 per warp
  // W = R2/2 is the "keep everything" variant (lik_window_groups only returns it as the fall-back): all R2 output
  // groups, also the middle one of an odd R2
  __host__ __device__ static constexpr int nk(int W) { return W >= L::R2 / 2 ? L::R2 : 2 * W; }
  // Above N = 224 one CTA fills an SM and the warp count is what the shared memory leaves: Y then
  // holds exactly the window rows (slot = window row index, nwp of them) instead of whole radix
  // output groups, which buys two more warps at N = 320 / 360 and the 24 x 16 split at N = 384.
  static constexpr bool COMPACT = N > 224 || L::G::GENERIC;
  __host__ __device__ static constexpr int rows(int W, int nwp) { return COMPACT ? nwp : nk(W) * L::R1; }
  // BIOEM_TMA (measured variant, profiles/r02_tma_variant.md): one staging slot per warp for the conv and the
  // particle chunk of its next column task, filled by cp.async.bulk
  static constexpr int CHUNK4 = (L::R1 / 2) * KC * L::R2; // float4 per operand chunk (contiguous in the packed layout)
#ifdef BIOEM_TMA
  static constexpr size_t OPS_BYTES = 2 * (size_t) CHUNK4 * 16;
#else
  static constexpr size_t OPS_BYTES = 0;
#endif
  __host__ __device__ static constexpr size_t dyn_bytes(int W, int nwarp, int nwp)
  {
    return ((size_t) rows(W, nwp) * YS + (size_t) nwarp * EW) * sizeof(float2) + ((N + 15) & ~15) + 256 + nwarp * OPS_BYTES;
  }
};
template <int N> __host__ __device__ constexpr int lik_window_groups(int maxD);

// likelihoods whose double-precision bookkeeping is deferred, then done by that many lanes of warp 0
// at once (32: one per lane -- the double-precision log / exp sequence costs warp 0 the same ~1,700 instructions
// whether 16 or 32 lanes are busy, and the other warps end up waiting for it at the next barrier)
#ifndef BIOEM_NPEND
#define BIOEM_NPEND 32
#endif
template <int N> __host__ __device__ constexpr int lik_pending() { return BIOEM_NPEND; }

// warps per CTA of the fused kernel.  From N = 160 to 224 two CTAs of 8 warps share an SM.  Measured
// on B200 at N = 224 (tools/build_variant.py): 8 warps 55.1 ns/likelihood, 7 warps (which would
// divide both the 56 column chunks and the 21 row tasks evenly) 58.1 ns -- registers are granted
// in units of 4 warps, so 7 warps buy nothing.  Above, one CTA fills the SM (its row slots need
// more than half of the shared memory): as many warps (12, 10 or 8) as fit next to the row slots
// of the production window DISPLACE_CENTER 40 (N = 360: 8 warps 248.7, 12 warps 204.7 ns).
template <int N> __host__ __device__ constexpr int lik_warps()
{
#ifdef BIOEM_LW
  return BIOEM_LW;
#else
  // small images: four CTAs of 4 warps per SM -- the row slots are small, and the finer barrier
  // domains lose less to the uneven last round of row tasks (measured with the N/4 window:
  // N = 64 8.0 -> 6.1, N = 96 19.1 -> 15.5, N = 128 27.6 -> 23.0 ns/likelihood; N = 160 / 192 are
  // slower that way, their row slots allow only two or three such CTAs)
  if (N <= 128)
    return 4;
  if (N <= 224)
    return 8;
  constexpr size_t budget = 227 * 1024 - 1024;
  for (int nw = 12; nw > 8; nw -= 2)
    if (LikGeo<N>::dyn_bytes(lik_window_groups<N>(40), nw, 82) + (size_t) lik_pending<N>() * nw * 8 + 512 <= budget)
      return nw;
  return 8;
#endif
}
template <int N> struct LikSmem
{
  using L = Lay<N>;
  using G = LikGeo<N>;
  static constexpr int NWARP = lik_warps<N>();
  static constexpr int LNT = 32 * NWARP; // threads per CTA
  // registers per thread: two CTAs per SM up to N = 224 (registers are granted to a CTA in units
  // of 4 warps, so 7 warps cost as many as 8), one CTA per SM above
#ifdef BIOEM_MAXREG
  static constexpr int MAXREG = BIOEM_MAXREG;
#else
  static constexpr int MAXREG = N <= 224 ? 128 : (65536 / (32 * ((NWARP + 3) / 4 * 4))) / 8 * 8 > 255 ? 255 : (65536 / (32 * ((NWARP + 3) / 4 * 4))) / 8 * 8;
#endif
  static constexpr int KC = G::KC, CS = G::CS, ES = G::ES, YS = G::YS, EW = G::EW;
  static constexpr bool WIDE = G::WIDE;
  __host__ __device__ static constexpr int nk(int W) { return G::nk(W); }
  __host__ __device__ static constexpr size_t bytes(int W, int nwp) { return G::dyn_bytes(W, NWARP, nwp); }
};
template <int N> __host__ __device__ constexpr size_t lik_smem_bytes(int maxD, int nwp)
{
  return LikSmem<N>::bytes(lik_window_groups<N>(maxD), nwp);
}

// 64-bit shared store straight from the register pair that holds the value (with a plain C++
// store ptxas stages five of the six row-slot stores of a column item through one register pair:
// two MOVs each, serialised on the previous store's operand read)
__device__ __forceinline__ void sts_f2(float2 *dst, float2 v)
{
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"((unsigned) __cvta_generic_to_shared(dst)), "f"(v.x), "f"(v.y));
}

__device__ __forceinline__ float rcp_approx(float x)
{
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 2^x, one MUFU.EX2 (results below the normal range flush to zero)
__device__ __forceinline__ float ex2_ftz(float x)
{
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m)
{
  unsigned lo = (unsigned) v, hi = (unsigned) (v >> 32);
  lo = __shfl_xor_sync(0xffffffffu, lo, m);
  hi = __shfl_xor_sync(0xffffffffu, hi, m);
  return ((unsigned long long) hi << 32) | lo;
}

// sentinels of the running minimum of firstele (real values are many orders of magnitude smaller):
// outputs that are no window displacement carry FE_INVALID, a thread that has seen nothing FE_NONE
constexpr float FE_INVALID = 1e36f, FE_NONE = 1e35f;

// monotone map float -> unsigned (a < b  <=>  ord(a) < ord(b))
__device__ __forceinline__ unsigned float_ordered(float f)
{
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// running per-image state of one CTA (kept in shared memory, touched by warp 0 only)
struct BookState
{
  double Const, Total, anConst, anTotal;
  float lpf, v, sC, ssC;
  int o, c, lin;
};

// ===========================================================================
// stages 3-5 fused.  One CTA owns one particle image m and a group of
// orientations of the current batch; for every (orientation, CTF) pair it
//   * streams the conv spectrum (L2) and the particle spectrum (L2/HBM) with fully
//     coalesced 128-bit loads (one 512-byte line per warp instruction) and multiplies
//     conv * conj(particle) in registers,
//   * column pass of the inverse 2-D FFT, WARP-SYNCHRONOUS: each warp owns KC columns at a
//     time (lanes = KC columns x R2 sub-sequences), radix-R1 in registers, twiddle (lane
//     constants held in registers), exchange through the warp's private shared-memory tile
//     (only __syncwarp), radix-R2 in registers; only the output groups that can hold window
//     displacements are formed (output pruning) and stored, unconditionally, as rows of Y,
//   * row pass, same structure: two real rows per complex transform, through the same tile,
//   * the displacement-dependent factor of the analytic log-posterior (firstele, FP32,
//     reference operation order, two displacements per packed instruction) straight out of
//     the FFT registers; every thread keeps an ONLINE (min firstele <=> max logpro, sum of exp
//     relative to that minimum, re-based when the minimum moves); a REDUX minimum and a shuffle
//     sum combine the lanes into one ring entry per warp,
//   * the bookkeeping (double-precision log, float narrowing, log-sum-exp fold into the image's
//     running state, arg-max (orientation, CTF)) is deferred: warp 0 does it for lik_pending<N>()
//     = 16 likelihoods at once, one per lane.  The displacement of the arg-max is NOT tracked here:
//     exact_argmax_kernel re-evaluates every particle's winning likelihood at download.
// All butterflies run on packed FP32x2 instructions.  Per likelihood one CTA barrier (columns
// -> rows) and one split-phase mbarrier (rows -> next columns: arrive, run the first radix pass
// of the next likelihood's first chunk, wait); no correlation map ever leaves the SM.
// ===========================================================================
template <int N, int W, bool ZM, bool GR = false>
__global__ void __launch_bounds__(LikSmem<N>::LNT) __maxnreg__(LikSmem<N>::MAXREG) likelihood_kernel(LikParams p)
{
  using KL = KLay<N>;
  using L = Lay<N>;
  using SM = LikSmem<N>;
  constexpr int NK = SM::nk(W); // radix-R2 output groups kept
  constexpr int R1 = L::R1, R2 = L::R2, KC = L::KC, NCH = L::NCH;
  constexpr int ES = SM::ES, CS = SM::CS, YS = SM::YS, NWARP = SM::NWARP;
  constexpr bool COMPACT = SM::G::COMPACT;
  constexpr int P2 = (KC * R1 + 31) / 32; // pass-2 trips
  constexpr int NPEND = lik_pending<N>();
  // window mask folded into the last term of firstele instead of FSEL (P2 * NK more registers).  Measured at N = 224:
  // 47.2 ns with, 46.7 ns without (fewer instructions, but the extra live registers cost more) -- off.
#ifndef BIOEM_AMASK
#define BIOEM_AMASK 0
#endif
  constexpr bool AMASK = BIOEM_AMASK && P2 * NK <= 8;
  auto k2_of = [](int j) { return (NK == R2) ? j : (j < W ? j : R2 - NK + j); };

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *Y = reinterpret_cast<float2 *>(smem_raw); // [NROWS][YS]
  float2 *Eall = Y + (size_t) SM::G::rows(W, p.nwp) * YS;
  unsigned char *WT = reinterpret_cast<unsigned char *>(Eall + (size_t) NWARP * SM::EW);
  unsigned char *RS = WT + ((N + 15) & ~15);
#ifdef BIOEM_TMA
  constexpr int CHUNK4 = SM::G::CHUNK4;
  constexpr unsigned CHUNKB = CHUNK4 * 16;
  float4 *OPS = reinterpret_cast<float4 *>(RS + 256) + (size_t) (threadIdx.x >> 5) * 2 * CHUNK4; // [conv chunk][particle chunk]
  __shared__ unsigned long long s_tbar[NWARP];
#endif
  // ring of likelihoods waiting for their bookkeeping, one entry per warp and likelihood: the warp's minimum of
  // firstele (bit pattern: positive floats order like their bits) and its sum of exp relative to that minimum
  __shared__ unsigned s_wk[NPEND][NWARP];
  __shared__ float s_ws[NPEND][NWARP];
  __shared__ int s_poc[NPEND];
  __shared__ unsigned long long s_mbar; // closing barrier of a likelihood (one arrival per warp)
  __shared__ BookState s_bk;
  __shared__ int s_zslot;

  const int nw = p.nw, nwp = p.nwp;
  const int tid = threadIdx.x;
  int warp = tid >> 5;
  int lane = tid & 31;
  // (cached-product variant: with one more operand stream the register allocator sits at its 128-register cap and
  // would rather re-derive the lane number from the thread-id register inside every column task -- a long-latency
  // S2R in front of the operand loads -- than keep it; an opaque move makes it keep it)
#ifndef BIOEM_ZV
#define BIOEM_ZV 27
#endif
  // (measured at N = 224, ns per likelihood: none 46.2, lane 45.9, + scratch offset 45.6, + table offset 45.4,
  // + warp number 45.1; the same moves make the complex-path kernel spill, so they are this variant's only)
  constexpr int RV = ZM ? BIOEM_ZV : 0;
  constexpr bool LATE_SUMS = (RV & 4) != 0;
  if constexpr ((RV & 1) != 0)
    asm volatile("" : "+r"(lane));
  if constexpr ((RV & 16) != 0)
    asm volatile("" : "+r"(warp));
  float2 *E = Eall + (size_t) warp * SM::EW;
  static_assert(ZM || !GR, "grouped CTF tables are real: cached-product mode only");
  const int m = GR ? p.perm[blockIdx.x % p.M] : (p.pairs ? p.pairs[blockIdx.x].x : blockIdx.x % p.M);
  // (grouped table: first row of this particle's group; the work-list path indexes rows directly and is never grouped)
  const int cb = GR ? p.group[m] * p.C : 0;
  const int g = p.pairs ? blockIdx.x : blockIdx.x / p.M;
  const int o_lo = g * p.OG;
  const int o_hi = min(p.OBcur, o_lo + p.OG);

  for (int i = tid; i < N; i += SM::LNT)
  {
    const unsigned w = p.wtab[i];
    WT[i] = (unsigned char) w;
    if (w != 255u)
    {
      const int k2 = i / R1, k1 = i % R1;
      const int j = (NK == R2) ? k2 : (k2 < W ? k2 : k2 - (R2 - NK));
      const int rs = COMPACT ? (int) w : j * R1 + k1;
      RS[w] = (unsigned char) rs;
      if ((int) w == nw - 1)
        RS[nw] = (unsigned char) rs; // padding row of an odd window: any valid slot
    }
  }
  const unsigned mbar_addr = (unsigned) __cvta_generic_to_shared(&s_mbar);
  unsigned mbar_parity = 0;
#ifdef BIOEM_TMA
  const unsigned tbar_addr = (unsigned) __cvta_generic_to_shared(&s_tbar[warp]);
  const unsigned ops_addr = (unsigned) __cvta_generic_to_shared(OPS);
  unsigned tbar_parity = 0;
  if (lane == 0)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tbar_addr), "r"(1) : "memory");
#endif
  if (tid == 0)
  {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar_addr), "r"(NWARP) : "memory");
    s_bk.Const = kMinProb;
    s_bk.Total = 0.0;
    s_bk.lpf = 0.f;
    s_bk.v = s_bk.sC = s_bk.ssC = 0.f;
    s_bk.o = s_bk.c = s_bk.lin = 0;
    if constexpr (ZM)
    {
      // a private scratch map for this CTA's cached product: first free slot, starting at this SM's own (there are as
      // many slots as CTAs can be resident, so the search ends at once; it would also end with fewer)
      unsigned smid, nsm;
      asm("mov.u32 %0, %%smid;" : "=r"(smid));
      asm("mov.u32 %0, %%nsmid;" : "=r"(nsm));
      const unsigned per_sm = max(1u, (unsigned) p.nslots / max(1u, nsm));
      int sl = (int) ((smid * per_sm) % (unsigned) p.nslots);
      while (atomicCAS(p.zflags + sl, 0, 1) != 0)
        sl = sl + 1 == p.nslots ? 0 : sl + 1;
      s_zslot = sl;
    }
  }
  __syncthreads();
  float4 *zs = ZM ? p.zbuf + (size_t) s_zslot * L::MAP4 : nullptr;
  // this lane's float4 of column chunk 0 in the scratch maps (kept, not re-derived, for the same reason)
  int zoff = ZM ? s_zslot * L::MAP4 + lane : 0;
  if constexpr (ZM && (BIOEM_ZV & 2))
    asm volatile("" : "+r"(zoff));
  float4 *const zs_l = p.zbuf + zoff;

  // lane roles (fixed for the whole kernel).  Pass 1 of both transforms: lane = c*R2 + n2
  // (c = column / row pair within the warp's task, n2 = sub-sequence).  Pass 2: item = k1*KC + c.
  const int a_c = lane / R2, a_n2 = lane % R2;
  const bool a_act = lane < KC * R2;
  float2 tw[R1]; // exp(+2 pi i n2*k1/N), k1 >= 1
#pragma unroll
  for (int k1 = 1; k1 < R1; k1++)
    tw[k1] = p.tw_inv[a_n2 * R1 + k1];
  // bit t*NK + j: output j of this lane's pass-2 item t is a window displacement (the others are
  // computed too, but enter the minimum / sum as FE_INVALID)
  unsigned vmask = 0;
#pragma unroll
  for (int t = 0; t < P2; t++)
  {
    const int item = lane + 32 * t;
    const int k1 = (item / KC) % R1;
    bfft::static_for<0, NK>([&](auto j_) {
      constexpr int j = decltype(j_)::value;
      if (WT[k1 + R1 * k2_of(j)] != 255)
        vmask |= 1u << (t * NK + j);
    });
  }
  static_assert(P2 * NK <= 32, "validity mask must fit one register");
  // compact row slots: byte j of cslot[t] = slot of output j of this lane's pass-2 item t in the
  // column pass (255: not a window row, not stored)
  constexpr int CSW = COMPACT ? (NK + 3) / 4 : 1;
  unsigned cslot[P2][CSW];
  if constexpr (COMPACT)
  {
#pragma unroll
    for (int t = 0; t < P2; t++)
    {
      const int k1 = ((lane + 32 * t) / KC) % R1;
#pragma unroll
      for (int q = 0; q < CSW; q++)
        cslot[t][q] = 0;
      bfft::static_for<0, NK>([&](auto j_) {
        constexpr int j = decltype(j_)::value;
        cslot[t][j / 4] |= (unsigned) WT[k1 + R1 * k2_of(j)] << (8 * (j % 4));
      });
    }
  }
  // exp(a*log1p(t)) = 2^(t*(c1 + t*(c2 + t*c3))), a = (3 - Nt)/2, for the tiny t >= 0 that matter;
  // decreasing in t and 0 for huge t
  const float c1 = p.ex2coef, c2 = -0.5f * p.ex2coef, c3 = p.ex2coef * (1.f / 3.f);
  auto expa1p = [&](float t) { return ex2_ftz(t * fmaf(t, fmaf(t, c3, c2), c1)); };

  const float4 *ref = p.refs + (size_t) m * L::MAP4;
  // first column chunk of this warp.  Chunk 0 (which also carries the Nyquist column: half as many
  // loads and multiplies again) goes to the last warp, which has the fewest row tasks: its first
  // radix pass runs in that warp's slack before the closing barrier.
  const int ch0 = (warp + 1) % NWARP;
  // (the particle's sums and the conv spectrum's sums are only needed in the row pass: they are read there, behind
  // the column -> row barrier, instead of living in registers through the column pass, where every register counts)
  __shared__ float s_sr[2];
  float sR0 = 0.f, ssR0 = 0.f;
  if constexpr (LATE_SUMS)
  {
    if (tid == 0)
    {
      s_sr[0] = p.sumRef[m];
      s_sr[1] = p.sumsqRef[m];
    }
  }
  else
    sR0 = p.sumRef[m], ssR0 = p.sumsqRef[m];
  const float Nt = p.Ntotpi;
  int slot = 0; // likelihoods in the ring (uniform over the CTA)

  // Bookkeeping of the npend ring entries (bioem_algorithm.h:84-141), by warp 0: lane l takes
  // entry l -- the two double-precision logs, the exact first-of-ties rule over its near-minimum
  // candidates -- then the entries are folded in enumeration order semantics: the running maximum
  // only moves on a strictly greater float-narrowed logpro, so the FIRST maximum wins.
  auto flush = [&](int npend) {
    __syncwarp();
    const bool act = lane < npend;
    float lpf = __int_as_float(0xff800000), S = 0.f;
    int oc = 0;
    ConvParam cpl;
    cpl.sumC = cpl.sumsqC = 0.f;
    if (act)
    {
      unsigned fbmin = 0xffffffffu;
#pragma unroll
      for (int w = 0; w < NWARP; w++)
        fbmin = min(fbmin, s_wk[lane][w]);
      oc = s_poc[lane];
      cpl = p.cpar[oc];
      const float fmin = __uint_as_float(fbmin);
      const float inv = __fdiv_rn(1.f, fmin);
      lpf = (float) __fma_rn(p.acoef_d, log((double) fmin), cpl.Bterm);
#pragma unroll 1
      for (int w = 0; w < NWARP; w++)
        S += s_ws[lane][w] * expa1p((__uint_as_float(s_wk[lane][w]) - fmin) * inv);
    }
    // (WHICH displacement attains the maximum is not tracked: logpro is narrowed to float before it is compared, so
    // displacements tie and the first in enumeration order keeps the record, bioem_algorithm.h:84-96 -- the exact pass
    // at download, exact_argmax_kernel, applies that rule to the whole window of every particle's winning likelihood)
    // arg-max of the batch: greatest lpf, lowest lane (= first in enumeration order) on ties
    unsigned long long key = ((unsigned long long) float_ordered(lpf) << 32) | (unsigned) (31 - lane);
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1)
    {
      const unsigned long long o = shfl_xor_u64(key, sft);
      key = o > key ? o : key;
    }
    const int lbest = 31 - (int) (key & 31u);
    const float lpfmax = __shfl_sync(0xffffffffu, lpf, lbest);
    double e = act ? (double) S * exp((double) lpf - (double) lpfmax) : 0.0;
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1)
      e += __longlong_as_double((long long) shfl_xor_u64((unsigned long long) __double_as_longlong(e), sft));
    if (lane == lbest)
    {
      if (s_bk.Const < (double) lpfmax)
      {
        s_bk.Total = s_bk.Total * exp(s_bk.Const - (double) lpfmax) + e;
        s_bk.Const = (double) lpfmax;
        s_bk.lpf = lpfmax;
        s_bk.o = p.o_base + oc / (GR ? p.GC : p.C);
        s_bk.c = oc % (GR ? p.GC : p.C); // (grouped: the row of the whole table)
        s_bk.lin = 0; // displacement index and correlation value: filled in by the exact pass
        s_bk.v = 0.f;
        s_bk.sC = cpl.sumC;
        s_bk.ssC = cpl.sumsqC;
      }
      else
        s_bk.Total += e * exp((double) lpfmax - s_bk.Const);
      if (p.angles)
      {
        if (s_bk.anConst < (double) lpfmax)
        {
          s_bk.anTotal = s_bk.anTotal * exp(s_bk.anConst - (double) lpfmax) + e;
          s_bk.anConst = (double) lpfmax;
        }
        else
          s_bk.anTotal += e * exp((double) lpfmax - s_bk.anConst);
      }
    }
    __syncwarp();
  };

  // The two radix passes of one column chunk (KC columns) of the current warp.
  //   col1: loads, conv * conj(particle), radix-R1, twiddle -> the warp's exchange tile
  //   col2: radix-R2 (pruned) from the tile -> row slots of Y
  // (FIRST: chunk 0, which also carries the Nyquist column -- a separate instance, so that the
  // other 55 chunks do not pay the register moves that merge the two paths)
#ifdef BIOEM_TMA
  // one elected lane asks the copy engine for the conv and the particle chunk of a column task: two contiguous
  // 3.5 KB blocks of the packed layout -> this warp's staging slot, completion counted on the warp's mbarrier
  auto tma_issue = [&](int ch, const float4 *conv) {
    if (lane == 0)
    {
      const float4 *gc = conv + (size_t) ch * CHUNK4, *gr = ref + (size_t) ch * CHUNK4;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tbar_addr), "r"(2u * CHUNKB) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ops_addr),
                   "l"(gc), "r"(CHUNKB), "r"(tbar_addr)
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ops_addr + CHUNKB),
                   "l"(gr), "r"(CHUNKB), "r"(tbar_addr)
                   : "memory");
    }
  };
#endif
  // (more: another likelihood follows the one conv belongs to -- only the staging variant needs to know)
  // the radix-R1 butterflies, the inter-pass twiddles and the store into the warp's exchange tile
  auto col1_finish = [&](float2(&x)[R1]) {
    bfft::Dft<R1, 1>::run(x);
#pragma unroll
    for (int k1 = 1; k1 < R1; k1++)
      x[k1] = bfft::cmul(x[k1], tw[k1]);
#pragma unroll
    for (int k1 = 0; k1 < R1; k1++)
      E[k1 * ES + a_c * CS + a_n2] = x[k1];
  };
  // Cached-product mode: Z = projection * conj(particle) of the current orientation, this warp's column chunks, into
  // the CTA's scratch map.  Every lane later reads back exactly the float4 it stored here (same chunk -> warp -> lane
  // assignment as col1), so the scratch needs no synchronisation at all; it stays in L2.
  auto zpass = [&](int pidx) {
    if constexpr (ZM)
    {
      const float4 *P = p.projs + (size_t) pidx * L::MAP4;
      if (a_act)
      {
        for (int ch = ch0; ch < NCH; ch += NWARP)
        {
          const int base = ch * (R1 / 2) * KC * R2 + lane;
#pragma unroll
          for (int n1p = 0; n1p < R1 / 2; n1p++)
          {
            const float4 r = ldg4(ref + base + n1p * KC * R2);
            const float4 v = ldg4(P + base + n1p * KC * R2);
            const float2 za = bfft::cmulc(make_float2(v.x, v.y), make_float2(r.x, r.y));
            const float2 zb = bfft::cmulc(make_float2(v.z, v.w), make_float2(r.z, r.w));
            zs_l[base - lane + n1p * KC * R2] = make_float4(za.x, za.y, zb.x, zb.y);
          }
          if (ch == 0 && a_c == 0)
          {
#pragma unroll
            for (int n1p = 0; n1p < R1 / 2; n1p++)
            {
              const float4 r = ldg4(ref + L::MAIN4 + n1p * R2 + a_n2);
              const float4 v = ldg4(P + L::MAIN4 + n1p * R2 + a_n2);
              const float2 za = bfft::cmulc(make_float2(v.x, v.y), make_float2(r.x, r.y));
              const float2 zb = bfft::cmulc(make_float2(v.z, v.w), make_float2(r.z, r.w));
              zs[L::MAIN4 + n1p * R2 + a_n2] = make_float4(za.x, za.y, zb.x, zb.y);
            }
          }
        }
      }
      __syncwarp();
    }
  };
  // (conv: the conv spectrum of the likelihood -- in cached-product mode the real table of its CTF)
  auto col1_ = [&](int ch, const float4 *conv, bool more, auto first_) {
    constexpr bool FIRST = decltype(first_)::value;
    if constexpr (ZM)
    {
      if (a_act)
      {
        float2 x[R1];
        const int base = ch * (R1 / 2) * KC * R2; // (+ lane: in zs_l)
        float kk[4 * KL::KQ];
#pragma unroll
        for (int q = 0; q < KL::KQ; q++)
        {
          const float4 k4 = ldg4(conv + (ch * KL::KQ + q) * KL::KCR2 + lane);
          kk[4 * q] = k4.x, kk[4 * q + 1] = k4.y, kk[4 * q + 2] = k4.z, kk[4 * q + 3] = k4.w;
        }
#pragma unroll
        for (int n1p = 0; n1p < R1 / 2; n1p++)
        {
          const float4 z = zs_l[base + n1p * KC * R2];
          x[2 * n1p] = __fmul2_rn(make_float2(z.x, z.y), make_float2(kk[2 * n1p], kk[2 * n1p]));
          x[2 * n1p + 1] = __fmul2_rn(make_float2(z.z, z.w), make_float2(kk[2 * n1p + 1], kk[2 * n1p + 1]));
        }
        if constexpr (FIRST)
        {
          if (a_c == 0)
          {
            // pack the Nyquist column into the (Hermitian) DC column: Z = X0 + i*X_{N/2}
            float kt[4 * KL::KQ];
#pragma unroll
            for (int q = 0; q < KL::KQ; q++)
            {
              const float4 k4 = ldg4(conv + KL::MAINK4 + q * R2 + a_n2);
              kt[4 * q] = k4.x, kt[4 * q + 1] = k4.y, kt[4 * q + 2] = k4.z, kt[4 * q + 3] = k4.w;
            }
#pragma unroll
            for (int n1p = 0; n1p < R1 / 2; n1p++)
            {
              const float4 z = zs[L::MAIN4 + n1p * R2 + a_n2];
              x[2 * n1p] = bfft::cadd_i(x[2 * n1p], __fmul2_rn(make_float2(z.x, z.y), make_float2(kt[2 * n1p], kt[2 * n1p])));
              x[2 * n1p + 1] =
                bfft::cadd_i(x[2 * n1p + 1], __fmul2_rn(make_float2(z.z, z.w), make_float2(kt[2 * n1p + 1], kt[2 * n1p + 1])));
            }
          }
        }
        col1_finish(x);
      }
      __syncwarp();
    }
    else
    {
#ifdef BIOEM_TMA
    {
      unsigned done;
      do
      {
        // (with a suspend-time hint, like the closing barrier: without it the waiting warps poll through the issue
        // slots of the others -- +13 % warp instructions per likelihood, measured)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2, %3;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(tbar_addr), "r"(tbar_parity), "r"(0x989680u)
                     : "memory");
      } while (!done);
      tbar_parity ^= 1u;
    }
    float2 x[R1];
    if (a_act)
    {
#pragma unroll
      for (int n1p = 0; n1p < R1 / 2; n1p++)
      {
        const float4 v = OPS[n1p * KC * R2 + lane];
        const float4 r = OPS[CHUNK4 + n1p * KC * R2 + lane];
        x[2 * n1p] = bfft::cmulc(make_float2(v.x, v.y), make_float2(r.x, r.y));
        x[2 * n1p + 1] = bfft::cmulc(make_float2(v.z, v.w), make_float2(r.z, r.w));
      }
    }
    // the slot has been consumed (its values are in x): hand it back to the copy engine for this warp's next task
    __syncwarp();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    {
      int nch = ch + NWARP;
      const float4 *nconv = conv;
      bool have = true;
      if (nch >= NCH)
      {
        nch = ch0;
        nconv = conv + L::MAP4;
        have = more;
      }
      if (have)
        tma_issue(nch, nconv);
    }
    if (a_act)
    {
#else
    if (a_act)
    {
      float2 x[R1];
      const int base = ch * (R1 / 2) * KC * R2 + lane; // == main_idx(ch, 0, a_n2, a_c)
#pragma unroll
      for (int n1p = 0; n1p < R1 / 2; n1p++)
      {
        const float4 r = ldg4(ref + base + n1p * KC * R2);
        const float4 v = ldg4(conv + base + n1p * KC * R2);
        x[2 * n1p] = bfft::cmulc(make_float2(v.x, v.y), make_float2(r.x, r.y));
        x[2 * n1p + 1] = bfft::cmulc(make_float2(v.z, v.w), make_float2(r.z, r.w));
      }
#endif
      if constexpr (FIRST)
      {
        if (a_c == 0)
        {
          // pack the Nyquist column into the (Hermitian) DC column: Z = X0 + i*X_{N/2}
#pragma unroll
          for (int n1p = 0; n1p < R1 / 2; n1p++)
          {
            const float4 r = ldg4(ref + L::MAIN4 + n1p * R2 + a_n2);
            const float4 v = ldg4(conv + L::MAIN4 + n1p * R2 + a_n2);
            x[2 * n1p] = bfft::cadd_i(x[2 * n1p], bfft::cmulc(make_float2(v.x, v.y), make_float2(r.x, r.y)));
            x[2 * n1p + 1] = bfft::cadd_i(x[2 * n1p + 1], bfft::cmulc(make_float2(v.z, v.w), make_float2(r.z, r.w)));
          }
        }
      }
      col1_finish(x);
    }
    __syncwarp();
    }
  };
  auto col1 = [&](int ch, const float4 *conv, bool more) {
    if (ch == 0)
      col1_(ch, conv, more, std::true_type{});
    else
      col1_(ch, conv, more, std::false_type{});
  };
  auto col2 = [&](int ch) {
#pragma unroll
    for (int t = 0; t < P2; t++)
    {
      const int item = lane + 32 * t;
      if (item < KC * R1)
      {
        const int k1 = item / KC, cc = item % KC;
        float2 y[R2];
        if constexpr (SM::WIDE)
        {
#pragma unroll
          for (int n2 = 0; n2 < R2; n2 += 2)
          {
            const float4 w = *reinterpret_cast<const float4 *>(&E[k1 * ES + cc * CS + n2]);
            y[n2] = make_float2(w.x, w.y);
            y[n2 + 1] = make_float2(w.z, w.w);
          }
        }
        else
        {
#pragma unroll
          for (int n2 = 0; n2 < R2; n2++)
            y[n2] = E[k1 * ES + cc * CS + n2];
        }
        bfft::Dft<R2, 1>::run(y);
        if constexpr (COMPACT)
        {
          float2 *Ycol = Y + ch * KC + cc;
          bfft::static_for<0, NK>([&](auto j_) {
            constexpr int j = decltype(j_)::value;
            const unsigned sl = (cslot[t][j / 4] >> (8 * (j % 4))) & 255u;
            if (sl != 255u)
            {
              // (direct stores pay up to R1 = 20: N = 320 119.6 -> 116.3 ns; with the 24-point first pass
              // of N = 360 / 384 they cost 4-9 %)
              if constexpr (R1 <= 20)
                sts_f2(Ycol + sl * YS, y[k2_of(j)]);
              else
                Ycol[sl * YS] = y[k2_of(j)];
            }
          });
        }
        else
        {
          float2 *Ycol = Y + k1 * YS + ch * KC + cc;
          bfft::static_for<0, NK>([&](auto j_) {
            constexpr int j = decltype(j_)::value;
            sts_f2(Ycol + j * R1 * YS, y[k2_of(j)]);
          });
        }
      }
    }
    __syncwarp();
  };
  // pass 1 of this warp's first column chunk was already run behind the closing barrier of the
  // previous likelihood
  bool pre_done = false;

#ifdef BIOEM_TMA
  if (o_lo < o_hi)
    tma_issue(ch0, p.convs + (size_t) o_lo * p.C * L::MAP4);
#endif
  if (o_lo < o_hi)
    zpass(p.pairs ? p.pairs[blockIdx.x].y : o_lo);
  for (int ol = o_lo; ol < o_hi; ol++)
  {
    if (tid == 0)
    {
      s_bk.anConst = kMinProb;
      s_bk.anTotal = 0.0;
    }
    for (int c = 0; c < p.C; c++)
    {
      const int oc = ol * p.C + c;
      const int orow = GR ? ol * p.GC + cb + c : oc; // row of cpar (grouped: [OBcur][GC])
      // (cached-product mode: the real table of CTF c, or of the work item's CTF)
      int koff = ZM ? (p.pairs ? p.pairs[blockIdx.x].z : cb + c) * p.kr4 : 0;
      if constexpr (ZM && (BIOEM_ZV & 8))
        asm volatile("" : "+r"(koff));
      const float4 *conv = ZM ? p.kreal + koff : p.convs + (size_t) oc * L::MAP4;
      if (tid == 0)
        s_poc[slot] = orow;
      float sumC, sumsqC;
      if constexpr (!LATE_SUMS)
      {
        const ConvParam cp = p.cpar[orow];
        sumC = cp.sumC, sumsqC = cp.sumsqC;
      }

      // ------------------------------------------------ column pass (along kx), per warp
      // (requesting the operands of the warp's next chunk before the second radix pass of the current one -- the
      // cached-product mode needs 42 operand registers instead of 56 -- still spills: 52.3 ns against 45.1, measured)
      for (int ch = ch0; ch < NCH; ch += NWARP)
      {
        if (!(pre_done && ch == ch0))
          col1(ch, conv, oc + 1 < o_hi * p.C);
        col2(ch);
      }
      pre_done = false;
      __syncthreads(); // all candidate rows of all columns are in Y
      // firstele = Nt*(ssR*ssC - v*v) + 2*sR*sC*v - ssR*sC*sC - sR*sR*ssC   (FP32, source order)
      // (the loads are issued here; their values are first needed in the epilogue of the first row task)
      if constexpr (LATE_SUMS)
        sumC = __ldg(&p.cpar[orow].sumC), sumsqC = __ldg(&p.cpar[orow].sumsqC);
      const float sR = LATE_SUMS ? s_sr[0] : sR0, ssR = LATE_SUMS ? s_sr[1] : ssR0;
      const float f_a = __fmul_rn(ssR, sumsqC);
      const float f_b = __fmul_rn(__fmul_rn(2.f, sR), sumC);
      const float f_c = __fmul_rn(__fmul_rn(ssR, sumC), sumC);
      const float f_d = __fmul_rn(__fmul_rn(sR, sR), sumsqC);
      float mfd[AMASK ? P2 * NK : 1];
      if constexpr (AMASK)
      {
#pragma unroll
        for (int q = 0; q < P2 * NK; q++)
          mfd[q] = ((vmask >> q) & 1u) ? -f_d : FE_INVALID;
      }

      // ------------------------------------------------ row pass (along ky), 2 rows per transform
      // running minimum of firstele of this thread, its enumeration index and correlation value,
      // and the sum of exp(logpro - logpro at that minimum) over everything seen so far
      float bfe = FE_NONE, binv = 1.f / FE_NONE;
      float2 S2 = make_float2(0.f, 0.f);
      const int npairs = nwp / 2;
      for (int p0 = warp * KC; p0 < npairs; p0 += NWARP * KC)
      {
        const int npl = min(KC, npairs - p0);
        if (a_act && a_c < npl)
        {
          const float2 *Ya = Y + (size_t) RS[2 * (p0 + a_c)] * YS;
          const float2 *Yb = Y + (size_t) RS[2 * (p0 + a_c) + 1] * YS;
          float2 x[R1];
#pragma unroll
          for (int n1 = 0; n1 < R1; n1++)
          {
            if (n1 < R1 / 2)
            {
              const float2 a = Ya[n1 * R2 + a_n2], b = Yb[n1 * R2 + a_n2];
              x[n1] = bfft::cadd_i(a, b); // A[n] + i*B[n]
            }
            else
            {
              // n = n1*R2 + n2 >= N/2: A[n] = conj(A[N-n])
              const int nm = (R1 - n1) * R2 - a_n2;
              const float2 a = Ya[nm], b = Yb[nm];
              x[n1] = __fadd2_rn(make_float2(a.x, -a.y), make_float2(b.y, b.x));
            }
          }
          if (a_n2 == 0)
          {
            // DC and Nyquist of the two (real) columns ky = 0 and ky = N/2 share slot 0
            const float2 a = Ya[0], b = Yb[0];
            x[0] = make_float2(a.x, b.x);
            x[R1 / 2] = make_float2(a.y, b.y);
          }
          bfft::Dft<R1, 1>::run(x);
#pragma unroll
          for (int k1 = 1; k1 < R1; k1++)
            x[k1] = bfft::cmul(x[k1], tw[k1]);
#pragma unroll
          for (int k1 = 0; k1 < R1; k1++)
            E[k1 * ES + a_c * CS + a_n2] = x[k1];
        }
        __syncwarp(); // also: every read of this task's Y rows is done, their slots may take FE
#pragma unroll
        for (int t = 0; t < P2; t++)
        {
          const int item = lane + 32 * t;
          const int k1 = item / KC, cc = item % KC;
          if (item < KC * R1 && cc < npl)
          {
            float2 y[R2];
            if constexpr (SM::WIDE)
            {
#pragma unroll
              for (int n2 = 0; n2 < R2; n2 += 2)
              {
                const float4 w = *reinterpret_cast<const float4 *>(&E[k1 * ES + cc * CS + n2]);
                y[n2] = make_float2(w.x, w.y);
                y[n2 + 1] = make_float2(w.z, w.w);
              }
            }
            else
            {
#pragma unroll
              for (int n2 = 0; n2 < R2; n2++)
                y[n2] = E[k1 * ES + cc * CS + n2];
            }
            bfft::Dft<R2, 1>::run(y);
            const int wa = 2 * (p0 + cc);
            const bool vb = wa + 1 < nw;
            // firstele of the item's NK x 2 displacements (.x = row wa, .y = row wa + 1), all at once
            float2 fe[NK];
            bfft::static_for<0, NK>([&](auto j_) {
              constexpr int j = decltype(j_)::value;
              const float2 v = bfft::cscale(y[k2_of(j)], p.invNN);
              float2 f = __fmul2_rn(v, v);
              f = __fadd2_rn(make_float2(f_a, f_a), make_float2(-f.x, -f.y));
              // (one fused multiply-add, spelled out: ptxas contracts the separate multiply and add anyway, and
              // exact_argmax_kernel must repeat this sequence bit for bit.  The reference's own build,
              // -O3 -ffast-math -march=native, is free to contract here too, quirk Q7.)
              f = __ffma2_rn(make_float2(Nt, Nt), f, __fmul2_rn(make_float2(f_b, f_b), v));
              f = __fadd2_rn(f, make_float2(-f_c, -f_c));
              if constexpr (AMASK)
              {
                // the last term doubles as the window mask: -f_d for a window column, FE_INVALID (which swallows the
                // value) for the few outputs of the kept radix groups that lie outside the window.  The padding row of
                // an odd window is a copy of the last row: it cannot move the minimum and is kept out of the sum below.
                f = __fadd2_rn(f, make_float2(mfd[t * NK + j], mfd[t * NK + j]));
                fe[j] = f;
              }
              else
              {
                f = __fadd2_rn(f, make_float2(-f_d, -f_d));
                const bool val = (vmask >> (t * NK + j)) & 1u;
                fe[j].x = val ? f.x : FE_INVALID;
                fe[j].y = (val && vb) ? f.y : FE_INVALID;
              }
            });
            float mn = fminf(fe[0].x, fe[0].y);
#pragma unroll
            for (int j = 1; j < NK; j++)
              mn = fminf(mn, fminf(fe[j].x, fe[j].y));
            // The displacement index of the maximum is not tracked here at all: the exact pass at download
            // (exact_argmax_kernel) re-evaluates the winning likelihood of every particle and applies the reference's
            // first-of-ties rule to its whole window.  Only the running minimum and the sum of exp relative to it remain.
            if (mn < bfe)
            {
              const float old = bfe;
              bfe = mn;
              binv = rcp_approx(bfe); // scales the arguments of the exp-sum only (error 1e-7 relative)
              const float sc = expa1p((old - bfe) * binv);
              S2 = __fmul2_rn(S2, make_float2(sc, sc));
            }
            bfft::static_for<0, NK>([&](auto j_) {
              constexpr int j = decltype(j_)::value;
              const float2 tt = __fmul2_rn(__fadd2_rn(fe[j], make_float2(-bfe, -bfe)), make_float2(binv, binv));
              float2 ll = __ffma2_rn(tt, make_float2(c3, c3), make_float2(c2, c2));
              ll = __ffma2_rn(tt, ll, make_float2(c1, c1));
              ll = __fmul2_rn(tt, ll);
              if constexpr (AMASK)
                S2 = __ffma2_rn(make_float2(ex2_ftz(ll.x), ex2_ftz(ll.y)), make_float2(1.f, vb ? 1.f : 0.f), S2);
              else
                S2 = __fadd2_rn(S2, make_float2(ex2_ftz(ll.x), ex2_ftz(ll.y)));
            });
            if (p.dbg_values)
              bfft::static_for<0, NK>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                if ((vmask >> (t * NK + j)) & 1u)
                {
                  const int wy = WT[k1 + R1 * k2_of(j)];
                  float *dv = p.dbg_values + (p.pairs ? (size_t) oc : (size_t) oc * p.M + m) * nw * nw;
                  dv[wa * nw + wy] = y[k2_of(j)].x * p.invNN;
                  if (vb)
                    dv[(wa + 1) * nw + wy] = y[k2_of(j)].y * p.invNN;
                }
              });
          }
        }
        __syncwarp();
      }

      // ------------------------------------------------ this warp's share of the window
      // (warp-wide integer minima are single REDUX instructions; firstele is positive, so its bit
      // pattern orders like the value)
      const unsigned fb = __float_as_uint(bfe);
      const unsigned wfb = __reduce_min_sync(0xffffffffu, fb);
      const float fw = __uint_as_float(wfb);
      float S = (S2.x + S2.y) * expa1p((bfe - fw) * rcp_approx(fw));
#pragma unroll
      for (int s = 16; s > 0; s >>= 1)
        S += __shfl_xor_sync(0xffffffffu, S, s);
      if (lane == 0)
      {
        s_wk[slot][warp] = wfb;
        s_ws[slot][warp] = S;
      }
      // Closing barrier, split: arrive (this warp is done with Y, its ring entry is written), then
      // -- instead of idling until the slowest warp is through its row tasks -- run the first radix
      // pass of this warp's first column chunk of the NEXT likelihood (it needs neither Y nor the
      // other warps), and only then wait.  Y may be overwritten after the wait.
      __syncwarp();
      if (lane == 0)
        asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(mbar_addr) : "memory");
      if (ch0 < NCH && oc + 1 < o_hi * p.C)
      {
        if constexpr (ZM)
        {
          // the next CTF's table follows this one; after the last CTF the next orientation's product comes first
          // (it, too, needs neither Y nor the other warps)
          const bool last = c == p.C - 1;
          if (last)
            zpass(ol + 1);
          col1(ch0, last ? p.kreal + (size_t) cb * p.kr4 : conv + p.kr4, false);
        }
        else
          col1(ch0, conv + L::MAP4, oc + 2 < o_hi * p.C); // the next conv spectrum of the batch follows this one
        pre_done = true;
      }
      {
        unsigned done;
        do
        {
          // (with a suspend-time hint: the warp sleeps in the barrier unit instead of spinning through
          // the issue slots of the other three warps of its scheduler)
          asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2, %3;\n\t"
                       "selp.u32 %0, 1, 0, p;\n\t}"
                       : "=r"(done)
                       : "r"(mbar_addr), "r"(mbar_parity), "r"(0x989680u)
                       : "memory");
        } while (!done);
        mbar_parity ^= 1u;
      }
      slot++;
      if (slot == NPEND || (p.angles && c == p.C - 1))
      {
        if (warp == 0)
          flush(slot);
        slot = 0;
      }
    }
    if (tid == 0 && p.angles)
    {
      ProbAngleOut a;
      a.forAngles = s_bk.anTotal;
      a.ConstAngle = s_bk.anConst;
      p.angles[(size_t) (p.o_base + ol) * p.M + m] = a;
    }
  }
  if (warp == 0 && slot > 0)
    flush(slot);
  if (tid == 0)
  {
    Running r;
    r.Const = s_bk.Const;
    r.Total = s_bk.Total;
    r.lpf = s_bk.lpf;
    r.orient = s_bk.o;
    r.conv = s_bk.c;
    r.lin = s_bk.lin;
    r.v = s_bk.v;
    r.sumC = s_bk.sC;
    r.sumsqC = s_bk.ssC;
    r.pad = 0;
    p.partials[p.pairs ? (size_t) blockIdx.x : (size_t) g * p.M + m] = r;
    // (every warp is past its last read of the scratch map: their arrivals at the closing barrier of the last
    // likelihood came after their column passes)
    if constexpr (ZM)
      atomicExch(p.zflags + s_zslot, 0);
  }
}


#ifndef BIOEM_LIK_ONLY
// fold the per-group partials of one batch into the running per-image state, in
// orientation order (strict '<' keeps the first maximum, bioem_algorithm.h:96)
__global__ void merge_partials_kernel(const Running *__restrict__ partials, int NG, int M, Running *__restrict__ state)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  Running s = state[m];
  for (int g = 0; g < NG; g++)
  {
    const Running r = partials[(size_t) g * M + m];
    if (r.Total <= 0.0 && r.Const <= kMinProb)
      continue;
    if (s.Const < r.Const)
    {
      const double T = s.Total * exp(s.Const - r.Const) + r.Total;
      s = r;
      s.Total = T;
    }
    else
      s.Total += r.Total * exp(r.Const - s.Const);
  }
  state[m] = s;
}

// Multi-GPU merge over peer memory: the per-image states of up to 16 GPUs of one box are read where they
// lie -- parts.p[r] points into GPU r's memory (peer access over NVLink / NVSwitch; the local GPU's own
// state for r == self) -- and folded in rank order with the rule of merge_partials_kernel.  Gather and
// merge are one kernel: M x 48 bytes per peer cross the switch as plain coalesced loads, nothing is staged.
struct PeerParts
{
  const Running *p[16];
  int n;
};
__global__ void merge_peers_kernel(PeerParts parts, int M, Running *__restrict__ state)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  Running s;
  s.Const = kMinProb;
  s.Total = 0.0;
  s.lpf = 0.f;
  s.orient = s.conv = s.lin = 0;
  s.v = s.sumC = s.sumsqC = 0.f;
  s.pad = 0;
  for (int r = 0; r < parts.n; r++)
  {
    const Running q = parts.p[r][m];
    if (q.Total <= 0.0 && q.Const <= kMinProb)
      continue;
    if (s.Const < q.Const)
    {
      const double T = s.Total * exp(s.Const - q.Const) + q.Total;
      s = q;
      s.Total = T;
    }
    else
      s.Total += q.Total * exp(q.Const - s.Const);
  }
  state[m] = s;
}

__global__ void init_state_kernel(Running *state, int M)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  Running s;
  s.Const = kMinProb;
  s.Total = 0.0;
  s.lpf = 0.f;
  s.orient = 0;
  s.conv = 0;
  s.lin = 0;
  s.v = 0.f;
  s.sumC = 0.f;
  s.sumsqC = 0.f;
  s.pad = 0;
  state[m] = s;
}

__global__ void init_angles_kernel(ProbAngleOut *a, size_t n)
{
  const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  a[i].forAngles = 0.0;
  a[i].ConstAngle = kMinProb;
}

// WRITE_PROB_ANGLES: the K most probable orientations of every particle among the orientations
// [oBegin, oEnd) of the angle table, selected where the table lies (reference: a size-K min-heap of
// (log(forAngles) + ConstAngle, orientation) per particle on the host, bioem.cpp:1254-1290).  One
// thread per particle: consecutive threads read consecutive 16-byte rows of one orientation.
// The list top[m][0..K) is kept sorted in descending (logp, orientation) order, i.e. the order in
// which the reference's heap is finally emptied; a full list only takes a strictly greater logp,
// like the heap (first come stays on equal values).
struct TopAngleOut // == bioem_b200_top_angle
{
  int orient, pad;
  double forAngles, ConstAngle;
};
__global__ void top_angles_kernel(const ProbAngleOut *__restrict__ tab, int M, int oBegin, int oEnd, int K,
                                  double *__restrict__ key, TopAngleOut *__restrict__ top)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  double *kk = key + (size_t) m * K;
  TopAngleOut *tt = top + (size_t) m * K;
  int n = 0;
  for (int o = oBegin; o < oEnd; o++)
  {
    const ProbAngleOut r = tab[(size_t) o * M + m];
    const double lp = log(r.forAngles) + r.ConstAngle;
    if (n == K && !(kk[K - 1] < lp))
      continue;
    // position in descending (logp, orientation) order; o is the largest orientation so far, so
    // the new row goes in front of equal keys
    int pos = (n < K) ? n : K - 1;
    while (pos > 0 && !(kk[pos - 1] > lp))
    {
      kk[pos] = kk[pos - 1];
      tt[pos] = tt[pos - 1];
      pos--;
    }
    kk[pos] = lp;
    tt[pos].orient = o;
    tt[pos].pad = 0;
    tt[pos].forAngles = r.forAngles;
    tt[pos].ConstAngle = r.ConstAngle;
    if (n < K)
      n++;
  }
  for (int i = n; i < K; i++)
  {
    tt[i].orient = -1;
    tt[i].pad = 0;
    tt[i].forAngles = 0.0;
    tt[i].ConstAngle = kMinProb;
  }
}

// Merge of per-rank lists of most probable orientations (WRITE_PROB_ANGLES on several GPUs): lists[r] holds
// rank r's [M][K] rows for ITS block of orientations (blocks ascend with the rank), each sorted as
// top_angles_kernel leaves it.  Feeding a block's rows in ascending orientation order into the same
// insertion rule reproduces what one pass over all orientations would have kept: a row dropped from a
// block's list was beaten by K rows of that block, which also beat it in the global list.
struct PeerLists
{
  const TopAngleOut *p[16];
  int n;
};
__global__ void merge_top_lists_kernel(PeerLists lists, int M, int K, double *__restrict__ key, TopAngleOut *__restrict__ top)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  double *kk = key + (size_t) m * K;
  TopAngleOut *tt = top + (size_t) m * K;
  int n = 0;
  for (int r = 0; r < lists.n; r++)
  {
    const TopAngleOut *src = lists.p[r] + (size_t) m * K;
    // ascending orientation order within the block: repeatedly take the smallest orientation not yet
    // taken (K is small: the reference's WRITE_PROB_ANGLES is typically 10-50)
    int last = -1;
    for (int it = 0; it < K; it++)
    {
      int best = -1, bo = 0x7fffffff;
      for (int i = 0; i < K; i++)
      {
        const int o = src[i].orient;
        if (o > last && o < bo)
        {
          bo = o;
          best = i;
        }
      }
      if (best < 0)
        break;
      last = bo;
      const TopAngleOut row = src[best];
      const double lp = log(row.forAngles) + row.ConstAngle;
      if (n == K && !(kk[K - 1] < lp))
        continue;
      int pos = (n < K) ? n : K - 1;
      while (pos > 0 && !(kk[pos - 1] > lp))
      {
        kk[pos] = kk[pos - 1];
        tt[pos] = tt[pos - 1];
        pos--;
      }
      kk[pos] = lp;
      tt[pos] = row;
      if (n < K)
        n++;
    }
  }
  for (int i = n; i < K; i++)
  {
    tt[i].orient = -1;
    tt[i].pad = 0;
    tt[i].forAngles = 0.0;
    tt[i].ConstAngle = kMinProb;
  }
}

// Exact arg-max displacement of the winning likelihood of every particle (bioem_algorithm.h:84-96: logpro is
// narrowed to float BEFORE the comparison, so neighbouring displacements often tie exactly, quirk Q10, and the
// FIRST one in enumeration order keeps the record).  The fused kernel finds the maximum itself exactly, but
// among the displacements that tie with it only those that were a thread's own minimum are candidates for
// "first".  This pass closes that gap: the correlation window of the winning (orientation, CTF) of each
// particle has been re-evaluated by the same kernel (bit-identical values, LikParams::pairs + dbg_values);
// one CTA per particle evaluates firstele in the same FP32 operation order, the float-narrowed logpro of
// every displacement that can possibly tie, and takes the lowest enumeration index among the equals.
struct RefineItem
{
  int m, slot, conv, pad;
};
__global__ void __launch_bounds__(128) exact_argmax_kernel(const RefineItem *__restrict__ items, const float *__restrict__ values,
                                                           const ConvParam *__restrict__ cpar, const float *__restrict__ sumRef,
                                                           const float *__restrict__ sumsqRef, int C, int nw, float Nt, float invNN,
                                                           double acoef, Running *__restrict__ state, int *__restrict__ counters)
{
  const RefineItem it = items[blockIdx.x];
  const float *v = values + (size_t) blockIdx.x * nw * nw;
  const ConvParam cp = cpar[blockIdx.x]; // the conv spectra of this pass were gathered per item
  const float sR = sumRef[it.m], ssR = sumsqRef[it.m];
  const float f_a = __fmul_rn(ssR, cp.sumsqC);
  const float f_b = __fmul_rn(__fmul_rn(2.f, sR), cp.sumC);
  const float f_c = __fmul_rn(__fmul_rn(ssR, cp.sumC), cp.sumC);
  const float f_d = __fmul_rn(__fmul_rn(sR, sR), cp.sumsqC);
  auto firstele = [&](float raw) {
    // same sequence as the fused kernel's epilogue (value = correlation / N^2 was stored)
    float f = __fmul_rn(raw, raw);
    f = __fadd_rn(f_a, -f);
    f = __fmaf_rn(Nt, f, __fmul_rn(f_b, raw));
    f = __fadd_rn(f, -f_c);
    f = __fadd_rn(f, -f_d);
    return f;
  };
  __shared__ float s_f[128];
  __shared__ int s_l[128];
  const int n = nw * nw, tid = threadIdx.x;
  float fmin = 3.0e38f;
  for (int i = tid; i < n; i += 128)
    fmin = fminf(fmin, firstele(v[i]));
  s_f[tid] = fmin;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1)
  {
    if (tid < s)
      s_f[tid] = fminf(s_f[tid], s_f[tid + s]);
    __syncthreads();
  }
  fmin = s_f[0];
  const float lpf = (float) __fma_rn(acoef, log((double) fmin), cp.Bterm);
  // logpro falls with firstele: whatever narrows to the same float lies within a few ulps of the minimum;
  // 2e-5 relative (~170 ulps) is a safe superset to run the double-precision log on
  const float fthr = fmin + fabsf(fmin) * 2e-5f;
  int best = 0x7fffffff;
  for (int i = tid; i < n; i += 128)
  {
    const float f = firstele(v[i]);
    if (f <= fthr && (float) __fma_rn(acoef, log((double) f), cp.Bterm) == lpf)
      best = min(best, i);
  }
  s_l[tid] = best;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1)
  {
    if (tid < s)
      s_l[tid] = min(s_l[tid], s_l[tid + s]);
    __syncthreads();
  }
  if (tid == 0)
  {
    Running r = state[it.m];
    atomicAdd(&counters[0], 1);
    if (lpf != r.lpf || s_l[0] == 0x7fffffff)
      atomicAdd(&counters[2], 1); // re-evaluation disagrees with the record: leave it alone (never expected)
    else
    {
      if (r.lin != s_l[0])
        atomicAdd(&counters[1], 1);
      r.lin = s_l[0];
      r.v = v[s_l[0]];
      state[it.m] = r;
    }
  }
}

// Running -> bioem_Probability_map (norm / mu as bioem_algorithm.h:106-111)
__global__ void finalize_kernel(const Running *__restrict__ state, const float *__restrict__ sumRef, int M, int nw,
                                int npos, int maxD, int Gs, float Ntotpi, ProbMapOut *__restrict__ out)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M)
    return;
  const Running s = state[m];
  ProbMapOut o;
  o.Total = s.Total;
  o.Constoadd = s.Const;
  o.max_prob_orient = s.orient;
  o.max_prob_conv = s.conv;
  if (s.Const <= kMinProb)
  {
    o.max_prob_cent_x = o.max_prob_cent_y = 0;
    o.max_prob_norm = o.max_prob_mu = 0.f;
  }
  else
  {
    const int wx = s.lin / nw, wy = s.lin % nw;
    // window index -> signed displacement in the reference's enumeration
    // (0, G, .., maxD, then N-maxD, N-maxD+G, ... reported as negative; bioem_algorithm.h:156-197)
    const int dx = wx < npos ? wx * Gs : (wx - npos) * Gs - maxD;
    const int dy = wy < npos ? wy * Gs : (wy - npos) * Gs - maxD;
    o.max_prob_cent_x = -dx;
    o.max_prob_cent_y = -dy;
    const float sR = sumRef[m];
    const float den = __fsub_rn(__fmul_rn(s.sumC, s.sumC), __fmul_rn(s.sumsqC, Ntotpi));
    o.max_prob_norm = __fdiv_rn(-__fadd_rn(__fmul_rn(-s.sumC, sR), __fmul_rn(Ntotpi, s.v)), den);
    o.max_prob_mu = __fdiv_rn(-__fadd_rn(__fmul_rn(-s.sumC, s.v), __fmul_rn(s.sumsqC, sR)), den);
  }
  out[m] = o;
}

#endif // BIOEM_LIK_ONLY

} // namespace bioem
