// Context, batching and the device half of the C ABI (include/bioem_b200.h).
#include "../../include/bioem_b200.h"
#include "bioem_kernels.cuh"
#include "generic_kernels.cuh"
#include "render_kernels.cuh"

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace bioem;

// hand-tuned splits (every pruned variant of the fused kernel) and rule-generated ones (unpruned variant only)
#define BIOEM_SIZES_TUNED(X) X(32) X(36) X(48) X(64) X(96) X(100) X(120) X(128) X(144) X(160) X(192) X(200) X(216) X(224) X(240) X(256) X(288) X(300) X(320) X(336) X(360) X(384) X(400) X(420) X(432) X(448) X(480) X(500) X(512)
#define BIOEM_SIZES_AUTO(X) X(16) X(18) X(20) X(24) X(28) X(30) X(40) X(42) X(50) X(54) X(56) X(60) X(70) X(72) X(80) X(84) X(90) X(98) X(108) X(112) X(126) X(140) X(150) X(162) X(168) X(180) X(196) X(210) X(250) X(252) X(270) X(280) X(294) X(324) X(350) X(378) X(392) X(450) X(486) X(504)
#define BIOEM_SIZES(X) BIOEM_SIZES_TUNED(X) BIOEM_SIZES_AUTO(X)

static thread_local std::string g_err;
static int fail(int code, const std::string &msg)
{
  g_err = msg;
  return code;
}
#define CU(call)                                                                                          \
  do                                                                                                      \
  {                                                                                                       \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess)                                                                                \
      return fail(BIOEM_B200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));               \
  } while (0)

// ---------------------------------------------------------------------------------
// NCCL is bound at run time (dlopen of libnccl.so.2: inside a PyTorch process that is the library torch
// has already loaded; for the stand-alone binary the system one), so the library itself has no link-time
// dependency on it and loads on boxes without NCCL.  Only the prototypes come from <nccl.h>.
// ---------------------------------------------------------------------------------
#include <dlfcn.h>
#include <nccl.h>
struct NcclApi
{
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommCount)(const ncclComm_t, int *) = nullptr;
  ncclResult_t (*CommUserRank)(const ncclComm_t, int *) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi *nccl_api()
{
  static NcclApi api;
  static bool tried = false;
  if (!tried)
  {
    tried = true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *nme : names)
      if ((api.lib = dlopen(nme, RTLD_NOW | RTLD_GLOBAL)))
        break;
    if (api.lib)
    {
      api.GetUniqueId = (decltype(api.GetUniqueId)) dlsym(api.lib, "ncclGetUniqueId");
      api.CommInitRank = (decltype(api.CommInitRank)) dlsym(api.lib, "ncclCommInitRank");
      api.AllGather = (decltype(api.AllGather)) dlsym(api.lib, "ncclAllGather");
      api.CommDestroy = (decltype(api.CommDestroy)) dlsym(api.lib, "ncclCommDestroy");
      api.CommCount = (decltype(api.CommCount)) dlsym(api.lib, "ncclCommCount");
      api.CommUserRank = (decltype(api.CommUserRank)) dlsym(api.lib, "ncclCommUserRank");
      api.GetErrorString = (decltype(api.GetErrorString)) dlsym(api.lib, "ncclGetErrorString");
      if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.CommDestroy || !api.CommCount ||
          !api.CommUserRank || !api.GetErrorString)
        api.lib = nullptr;
    }
  }
  return api.lib ? &api : nullptr;
}
#define NC(call)                                                                                          \
  do                                                                                                      \
  {                                                                                                       \
    ncclResult_t r_ = (call);                                                                             \
    if (r_ != ncclSuccess)                                                                                \
      return fail(BIOEM_B200_ERR_CUDA, std::string(#call) + ": " + nccl_api()->GetErrorString(r_));       \
  } while (0)

struct bioem_b200_context
{
  bioem_b200_config cfg{};
  int device = 0;
  cudaStream_t stream = nullptr;
  int N = 0, nw = 0, nwp = 0, npos = 0;
  size_t map4 = 0; // float4 per packed map
  // inputs
  float4 *d_xyzr = nullptr;
  float *d_dens = nullptr;
  int A = 0;
  float NormDen = 0.f;
  float4 *d_angles = nullptr;
  std::vector<float4> h_angles; // host copy (the exact arg-max pass re-projects the winning orientations)
  int O = 0;
  float4 *d_ctf = nullptr;
  double *d_prior = nullptr;
  int C = 0; // rows of the CTF table (a grouped table: G x Cg)
  // Grouped table (upload_ctf_groups): particle m integrates over the Cg rows [group[m]*Cg, group[m]*Cg + Cg) only.
  // Ungrouped: G = 1, Cg = C and every particle takes every row.
  int G = 1, Cg = 0;
  bool grouped = false;
  bool groups_set = false;                   // set_particle_groups() matches the particles on the handle
  int group_max = -1;                        // largest group number of that list
  int *d_group = nullptr, *d_perm = nullptr; // [M] group of every particle; particles ordered by group
  // cached-product mode of the fused kernel (LikParams::zmode): possible when every CTF kernel is real (CTFs given
  // in Fourier space), chosen in ensure_batch
  bool ctf_is_real = false, zmode = false;
  // direct-DFT path (generic_kernels.cuh) for image edges without an instantiated fused kernel: spectra in the
  // reference's layout, correlation windows of a batch in d_values, window displacements in d_wl
  bool generic = false;
  int *d_wl = nullptr;
  float *d_values = nullptr;
  float4 *d_kreal = nullptr; // [C][kr4] real tables in column-pass order
  float4 *d_zbuf = nullptr;  // [nslots][map4] scratch maps of the resident CTAs
  int *d_zflags = nullptr;
  int nslots = 0;
  size_t kr4 = 0;
  float4 *d_refs = nullptr;
  float *d_sumRef = nullptr, *d_sumsqRef = nullptr;
  int M = 0;
  size_t particle_cap = 0; // images the particle / state buffers were allocated for
  float2 *d_tw_inv = nullptr, *d_tw_fwd = nullptr;
  unsigned char *d_wtab = nullptr;
  // batch buffers
  int OB = 0, OG = 1, nbands = 1, band_rows = 0, proj_threads = 256;
  float *d_proj = nullptr;
  double *d_tempden = nullptr;
  float2 *d_scratch = nullptr;
  float4 *d_projfft = nullptr;
  float4 *d_conv = nullptr;
  ConvParam *d_cpar = nullptr;
  Running *d_partials = nullptr;
  size_t partials_cap = 0;
  // results
  Running *d_state = nullptr;
  ProbAngleOut *d_angtab = nullptr;
  ProbMapOut *d_out = nullptr;
  bool state_ready = false;
  bool argmax_exact = true; // false: likelihoods were folded in since the last exact arg-max pass
  int refine_counts[3] = {0, 0, 0}; // records re-evaluated / displacement corrected / re-evaluation disagreed
  // stats
  long long launches = 0, likelihoods = 0, lik_launches = 0;
  // optional CUDA-event timing of the fused kernel (off unless bioem_b200_set_kernel_timing(h, 1)):
  // recorded pairs wait in lik_events until bioem_b200_kernel_time() reads them; events are recycled
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> lik_events;
  std::vector<cudaEvent_t> event_pool;
  bool time_kernels = false;
  // model points that fell out of the frame, per orientation, since reset (bioem.cpp:1724-1734,1756-1780)
  int *d_skipped = nullptr;
  // multi-GPU merge (NCCL communicator, gather buffers)
  void *nccl_comm = nullptr;
  bool nccl_owned = false;
  int nccl_ranks = 0, nccl_rank = 0;
  Running *d_gather = nullptr;
  size_t gather_cap = 0;
};

// Device buffers come from the device's stream-ordered memory pool (cudaMallocAsync on the
// handle's stream): destroying a handle and creating the next one then costs microseconds per
// buffer instead of the ~20 ms of a cudaFree / cudaMalloc pair (measured: 0.3 s per handle).
static void dfree(bioem_b200_context *h, void *p)
{
  if (p)
    cudaFreeAsync(p, h->stream);
}

// (re)allocate a device array of the handle: the old block is released and the pointer cleared FIRST, so
// that a failed allocation never leaves a dangling pointer behind (the handle stays destroyable)
template <class T> static int dev_realloc(bioem_b200_context *h, T *&p, size_t count)
{
  dfree(h, p);
  p = nullptr;
  if (count == 0)
    return BIOEM_B200_OK;
  CU(cudaMallocAsync((void **) &p, sizeof(T) * count, h->stream));
  return BIOEM_B200_OK;
}

// temporary device buffer of one entry point: released on every return path
struct DevTmp
{
  bioem_b200_context *h;
  void *p = nullptr;
  explicit DevTmp(bioem_b200_context *h_) : h(h_) {}
  DevTmp(const DevTmp &) = delete;
  DevTmp &operator=(const DevTmp &) = delete;
  ~DevTmp()
  {
    if (p)
      cudaFreeAsync(p, h->stream);
  }
  int alloc(size_t bytes)
  {
    CU(cudaMallocAsync(&p, bytes ? bytes : 1, h->stream));
    return BIOEM_B200_OK;
  }
  template <class T> T *as() const { return static_cast<T *>(p); }
};
#define RC(call)                                                                                          \
  do                                                                                                      \
  {                                                                                                       \
    int rc_ = (call);                                                                                     \
    if (rc_ != BIOEM_B200_OK)                                                                             \
      return rc_;                                                                                         \
  } while (0)

static void nccl_release(bioem_b200_context *h)
{
  if (h->nccl_comm && h->nccl_owned && nccl_api())
    nccl_api()->CommDestroy((ncclComm_t) h->nccl_comm);
  h->nccl_comm = nullptr;
  h->nccl_owned = false;
  h->nccl_ranks = 0;
}

static void free_batch(bioem_b200_context *h)
{
  dfree(h, h->d_proj);
  dfree(h, h->d_tempden);
  dfree(h, h->d_scratch);
  dfree(h, h->d_projfft);
  dfree(h, h->d_conv);
  dfree(h, h->d_cpar);
  dfree(h, h->d_partials);
  dfree(h, h->d_zbuf);
  dfree(h, h->d_zflags);
  dfree(h, h->d_values);
  h->d_values = nullptr;
  h->d_zbuf = nullptr;
  h->d_zflags = nullptr;
  h->nslots = 0;
  h->zmode = false;
  h->d_proj = nullptr;
  h->d_tempden = nullptr;
  h->d_scratch = nullptr;
  h->d_projfft = nullptr;
  h->d_conv = nullptr;
  h->d_cpar = nullptr;
  h->d_partials = nullptr;
  h->OB = 0;
  h->partials_cap = 0;
}

template <int N> static size_t map4_of() { return Lay<N>::MAP4; }

static size_t map4_for(int N)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return map4_of<n>();
    BIOEM_SIZES(X)
#undef X
  }
  return 0;
}

// float4 per CTF of the real table, and how many CTAs of the fused kernel one SM can hold (registers, threads and
// shared memory; smem = dynamic + static bytes of one CTA) -- the scratch maps of the cached-product mode are sized by it
template <int N> static void zgeo_of(size_t smem, size_t *kr4, int *ctas)
{
  *kr4 = KLay<N>::KR4;
  const int by_regs = 65536 / (LikSmem<N>::MAXREG * LikSmem<N>::LNT);
  const int by_thr = 2048 / LikSmem<N>::LNT;
  const int by_smem = (int) ((size_t) 228 * 1024 / (smem + 1024));
  *ctas = std::max(1, std::min(std::min(by_regs, by_thr), std::min(by_smem, 32)));
}
static void zgeo_for(int N, size_t smem, size_t *kr4, int *ctas)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    zgeo_of<n>(smem, kr4, ctas);                                                                          \
    return;
    BIOEM_SIZES(X)
#undef X
  }
}
template <int N> static cudaError_t launch_kreal(const float4 *ctf, float4 *kreal, int C, cudaStream_t s)
{
  dim3 g((KLay<N>::KR4 + 255) / 256, C);
  kreal_kernel<N><<<g, 256, 0, s>>>(ctf, kreal, C);
  return cudaGetLastError();
}
static cudaError_t do_kreal(int N, const float4 *ctf, float4 *kreal, int C, cudaStream_t s)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_kreal<n>(ctf, kreal, C, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}

// float4 per map on the direct-DFT path: N x (N/2+1) complex in the reference's layout, rounded up to whole float4
static size_t map4_generic(int N) { return ((size_t) N * (N / 2 + 1) + 1) / 2; }
static bool is_generic(int N) { return map4_for(N) == 0; }

template <int N> static void geo_of(int *r1, int *r2)
{
  *r1 = Lay<N>::R1;
  *r2 = Lay<N>::R2;
}
static void geo_for(int N, int *r1, int *r2)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    geo_of<n>(r1, r2);                                                                                    \
    return;
    BIOEM_SIZES(X)
#undef X
  }
}

// ---------------------------------------------------------------------------------
// per-size launchers
// ---------------------------------------------------------------------------------
template <int N> static cudaError_t launch_pack(const float2 *src, float4 *dst, int nmaps, cudaStream_t s)
{
  dim3 grid(32, nmaps);
  pack_kernel<N><<<grid, 256, 0, s>>>(src, dst, nmaps);
  return cudaGetLastError();
}
template <int N> static cudaError_t launch_unpack(const float4 *src, float2 *dst, int nmaps, cudaStream_t s)
{
  dim3 grid(32, nmaps);
  unpack_kernel<N><<<grid, 256, 0, s>>>(src, dst, nmaps);
  return cudaGetLastError();
}
template <int N>
static cudaError_t launch_fft2d(const float *imgs, const double *tempden, int nbands, float normDen, const float2 *tw_fwd,
                                float2 *scratch, float4 *packed, int nimg, cudaStream_t s)
{
  using L = Lay<N>;
  dim3 g1((N / 2 + L::PC - 1) / L::PC, nimg);
  fft_rows_kernel<N><<<g1, NT, 0, s>>>(imgs, tempden, nbands, normDen, tw_fwd, scratch);
  dim3 g2((N / 2 + 1 + L::FKC - 1) / L::FKC, nimg);
  const size_t smem2 = sizeof(float2) * (size_t) (L::FKC * N + N);
  cudaError_t e = cudaFuncSetAttribute(fft_cols_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem2);
  if (e != cudaSuccess)
    return e;
  fft_cols_kernel<N><<<g2, NT, smem2, s>>>(scratch, tw_fwd, packed);
  return cudaGetLastError();
}
template <int N>
static cudaError_t launch_conv(const float4 *proj, const float4 *ctf, const double *prior, float4 *conv, ConvParam *cpar, int C,
                               int OBcur, float Nt, cudaStream_t s, const int4 *sel, int nsel)
{
  dim3 g(sel ? 1 : C, sel ? nsel : OBcur);
  ctf_conv_kernel<N><<<g, NT, 0, s>>>(proj, ctf, prior, conv, cpar, C, Nt, sel);
  return cudaGetLastError();
}
// dynamic + (an upper bound of the) static shared memory of the fused kernel
template <int N> static size_t lik_smem(int maxD, int nwp)
{
  return lik_smem_bytes<N>(maxD, nwp) + (size_t) lik_pending<N>() * LikSmem<N>::NWARP * 8 + 512;
}

static cudaError_t do_pack(int N, const float2 *src, float4 *dst, int nmaps, cudaStream_t s)
{
  if (is_generic(N)) // the reference's layout is the device layout: a strided copy
  {
    const size_t F = (size_t) N * (N / 2 + 1);
    return cudaMemcpy2DAsync(dst, map4_generic(N) * sizeof(float4), src, F * sizeof(float2), F * sizeof(float2), nmaps,
                             cudaMemcpyDeviceToDevice, s);
  }
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_pack<n>(src, dst, nmaps, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
static cudaError_t do_unpack(int N, const float4 *src, float2 *dst, int nmaps, cudaStream_t s)
{
  if (is_generic(N))
  {
    const size_t F = (size_t) N * (N / 2 + 1);
    return cudaMemcpy2DAsync(dst, F * sizeof(float2), src, map4_generic(N) * sizeof(float4), F * sizeof(float2), nmaps,
                             cudaMemcpyDeviceToDevice, s);
  }
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_unpack<n>(src, dst, nmaps, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
static cudaError_t do_fft2d(int N, const float *imgs, const double *tempden, int nbands, float normDen, const float2 *tw,
                            float2 *scratch, float4 *packed, int nimg, cudaStream_t s)
{
  if (is_generic(N))
  {
    // (tw: exp(+2 pi i j / N) on this path, for both directions)
    gen_dft_rows_kernel<<<dim3(N, nimg), 256, (size_t) N * 12, s>>>(imgs, tempden, nbands, normDen, tw, N, scratch);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
      return e;
    gen_dft_cols_kernel<<<dim3(N, nimg), 256, (size_t) N * 8, s>>>(scratch, tw, N, 2 * map4_generic(N),
                                                                    reinterpret_cast<float2 *>(packed));
    return cudaGetLastError();
  }
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_fft2d<n>(imgs, tempden, nbands, normDen, tw, scratch, packed, nimg, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
template <int N>
static cudaError_t launch_sums(const float4 *proj, const float4 *ctf, const double *prior, ConvParam *cpar, int GC, int OBcur,
                               float Nt, cudaStream_t s)
{
  dim3 g((GC + SUMS_CB - 1) / SUMS_CB, (OBcur + SUMS_OB - 1) / SUMS_OB);
  ctf_sums_kernel<N><<<g, NT, 0, s>>>(proj, ctf, prior, cpar, GC, OBcur, Nt);
  return cudaGetLastError();
}
static cudaError_t do_sums(int N, const float4 *proj, const float4 *ctf, const double *prior, ConvParam *cpar, int GC,
                           int OBcur, float Nt, cudaStream_t s)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_sums<n>(proj, ctf, prior, cpar, GC, OBcur, Nt, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
static cudaError_t do_conv(int N, const float4 *proj, const float4 *ctf, const double *prior, float4 *conv, ConvParam *cpar,
                           int C, int OBcur, float Nt, cudaStream_t s, const int4 *sel = nullptr, int nsel = 0)
{
  if (is_generic(N))
  {
    if (sel || !conv)
      return cudaErrorInvalidValue; // (no exact arg-max pass, no cached-product mode on this path)
    gen_conv_kernel<<<dim3(C, OBcur), 256, 0, s>>>(reinterpret_cast<const float2 *>(proj), reinterpret_cast<const float2 *>(ctf),
                                                   prior, reinterpret_cast<float2 *>(conv), cpar, C, N, 2 * map4_generic(N), Nt);
    return cudaGetLastError();
  }
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_conv<n>(proj, ctf, prior, conv, cpar, C, OBcur, Nt, s, sel, nsel);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
// the fused kernel's variants live in one translation unit per image edge (lik_instance.inl)
#define X(n) extern "C" cudaError_t bioem_lik_launch_##n(const bioem::LikParams *, int, int, cudaStream_t);
BIOEM_SIZES(X)
#undef X
static cudaError_t do_lik(int N, const LikParams &p, int nblocks, int maxD, cudaStream_t s)
{
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return bioem_lik_launch_##n(&p, nblocks, maxD, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
// calculated images of a batch (render_kernels.cuh): conv spectra -> scratch [item][N][N/2+1] -> out [item][N][N]
template <int N>
static cudaError_t launch_render(const float4 *convs, const RenderItem *items, const float2 *tw_inv, float2 *scratch, float *out,
                                 int nitems, cudaStream_t s)
{
  using L = Lay<N>;
  dim3 g1((N / 2 + 1 + L::FKC - 1) / L::FKC, nitems);
  const size_t smem1 = sizeof(float2) * (size_t) (L::FKC * N + N);
  cudaError_t e = cudaFuncSetAttribute(render_cols_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem1);
  if (e != cudaSuccess)
    return e;
  render_cols_kernel<N><<<g1, NT, smem1, s>>>(convs, items, tw_inv, scratch);
  dim3 g2((N / 2 + L::PC - 1) / L::PC, nitems);
  render_rows_kernel<N><<<g2, NT, 0, s>>>(scratch, items, tw_inv, out);
  return cudaGetLastError();
}
static cudaError_t do_render(int N, const float4 *convs, const RenderItem *items, const float2 *tw_inv, float2 *scratch, float *out,
                             int nitems, cudaStream_t s)
{
  if (is_generic(N))
  {
    gen_render_cols_kernel<<<dim3(N, nitems), 256, (size_t) N * sizeof(float2), s>>>(
        reinterpret_cast<const float2 *>(convs), 2 * map4_generic(N), items, tw_inv, N, scratch);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
      return e;
    gen_render_rows_kernel<<<dim3(N, nitems), 256, (size_t) (N + N / 2 + 1) * sizeof(float2), s>>>(scratch, items, tw_inv, N, out);
    return cudaGetLastError();
  }
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return launch_render<n>(convs, items, tw_inv, scratch, out, nitems, s);
    BIOEM_SIZES(X)
#undef X
  }
  return cudaErrorInvalidValue;
}
// dynamic shared memory of gen_corr_kernel: twiddles, T[nw][N/2+1], window list
static size_t gen_corr_smem(int N, int nw) { return ((size_t) N + (size_t) nw * (N / 2 + 1)) * sizeof(float2) + (size_t) nw * 4; }
static size_t smem_for(int N, int maxD, int nwp)
{
  if (is_generic(N))
    return gen_corr_smem(N, nwp) + 64;
  switch (N)
  {
#define X(n)                                                                                              \
  case n:                                                                                                 \
    return lik_smem<n>(maxD, nwp);
    BIOEM_SIZES(X)
#undef X
  }
  return 0;
}

// Gaussian priors on the CTF parameters (bioem_algorithm.h:49-67), per kernel, in double.  A grouped table (G > 1 or
// cent != nullptr) has G groups of C / G rows, and group r's defocus prior is centred on cent[r] (nullptr: the config's
// centre for all).
static int set_ctf_priors(bioem_b200_context *h, const float *CtfParam4, int C, int G = 1, const float *cent = nullptr,
                          bool grouped = false)
{
  std::vector<double> prior(C);
  const bioem_b200_config &p = h->cfg;
  const int Cg = C / G;
  for (int c = 0; c < C; c++)
  {
    const float amp = CtfParam4[4 * c], pha = CtfParam4[4 * c + 1], env = CtfParam4[4 * c + 2];
    const float dcen = cent ? cent[c / Cg] : p.Priordefcent;
    double pr;
    if (!p.tousepsf)
    {
      pr = env * env / 2. / p.sigmaPriorbctf / p.sigmaPriorbctf -
           (pha - dcen) * (pha - dcen) / 2. / p.sigmaPriordefo / p.sigmaPriordefo -
           (amp - p.Priorampcent) * (amp - p.Priorampcent) / 2. / p.sigmaPrioramp / p.sigmaPrioramp;
    }
    else
    {
      // PSF parameters are mapped to their Fourier-space counterparts first (bioem_algorithm.h:59-66)
      const double envF = 4. * M_PI * M_PI * env / (env * env + pha * pha);
      const double phaF = 4. * M_PI * M_PI * pha / (env * env + pha * pha);
      pr = envF * envF / 2. / p.sigmaPriorbctf / p.sigmaPriorbctf -
           (phaF - p.Priordefcent) * (phaF - p.Priordefcent) / 2. / p.sigmaPriordefo / p.sigmaPriordefo -
           (amp - p.Priorampcent) * (amp - p.Priorampcent) / 2. / p.sigmaPrioramp / p.sigmaPrioramp;
    }
    prior[c] = pr;
  }
  const int Cold = h->C;
  h->C = 0; // stays 0 (run() refuses) unless everything below succeeds
  h->state_ready = false;
  (void) Cold;
  free_batch(h); // (also when C is unchanged: a real / complex table decides the mode of the fused kernel)
  // an ungrouped table drops the particle groups; a grouped one keeps them while they name groups it has
  h->groups_set = grouped && h->groups_set && h->group_max < G;
  h->grouped = false;
  RC(dev_realloc(h, h->d_prior, (size_t) C));
  CU(cudaMemcpyAsync(h->d_prior, prior.data(), sizeof(double) * C, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->G = G;
  h->Cg = Cg;
  h->grouped = grouped;
  h->C = C;
  return BIOEM_B200_OK;
}

// ---------------------------------------------------------------------------------
extern "C" {

const char *bioem_b200_last_error(void) { return g_err.c_str(); }
int bioem_b200_version(void) { return 100; }
int bioem_b200_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return n;
}
int bioem_b200_supported_size(int N) { return map4_for(N) != 0; }

// number of displacement-window points per axis as the reference's Algo 1 enumerates them
// (bioem_algorithm.h:156-197): 0, G, 2G, .. <= maxD, then N - maxD, N - maxD + G, .. < N, i.e.
// floor(maxD/G) + 1 non-negative and ceil(maxD/G) negative displacements (quirk Q3: when G does not
// divide maxD this is NOT the symmetric set NxDisp = 2*(maxD/G)+1 of param.cpp:1614-1617).
static void window_counts(int maxD, int G, int *npos, int *nneg)
{
  *npos = maxD / G + 1;
  *nneg = (maxD + G - 1) / G;
}

static int create_impl(bioem_b200_context *h, const bioem_b200_config *cfg)
{
  const int N = h->N;
  CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  {
    // keep freed blocks in the pool instead of returning them to the driver at every synchronisation
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, h->device) == cudaSuccess)
    {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  // twiddles (double -> float) at [n2*R1 + k1], and the displacement-window table
  int R1 = 0, R2 = 0;
  geo_for(N, &R1, &R2);
  std::vector<float2> twi(N), twf(N);
  if (h->generic)
  {
    // direct-DFT path: one table exp(+2 pi i j / N) for both directions, and the window displacements in
    // enumeration order (the inverse of the window table below)
    for (int j = 0; j < N; j++)
    {
      const double ang = 2.0 * M_PI * (double) j / (double) N;
      twi[j] = twf[j] = make_float2((float) cos(ang), (float) sin(ang));
    }
    std::vector<int> wl(h->nw);
    for (int k = 0; k < h->npos; k++)
      wl[k] = k * cfg->GridSpaceCenter;
    for (int k = 0; k < h->nw - h->npos; k++)
      wl[h->npos + k] = N - cfg->maxDisplaceCenter + k * cfg->GridSpaceCenter;
    RC(dev_realloc(h, h->d_wl, (size_t) h->nw));
    CU(cudaMemcpyAsync(h->d_wl, wl.data(), sizeof(int) * h->nw, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  for (int n2 = 0; n2 < R2; n2++)
    for (int k1 = 0; k1 < R1; k1++)
    {
      const long long pr = ((long long) n2 * k1) % N;
      const double ang = 2.0 * M_PI * (double) pr / (double) N;
      twi[n2 * R1 + k1] = make_float2((float) cos(ang), (float) sin(ang));
      twf[n2 * R1 + k1] = make_float2((float) cos(ang), (float) -sin(ang));
    }
  std::vector<unsigned char> wt(N, 255);
  for (int k = 0; k < h->npos; k++)
    wt[k * cfg->GridSpaceCenter] = (unsigned char) k;
  for (int k = 0; k < h->nw - h->npos; k++)
    wt[N - cfg->maxDisplaceCenter + k * cfg->GridSpaceCenter] = (unsigned char) (h->npos + k);
  RC(dev_realloc(h, h->d_tw_inv, (size_t) N));
  RC(dev_realloc(h, h->d_tw_fwd, (size_t) N));
  RC(dev_realloc(h, h->d_wtab, (size_t) N));
  CU(cudaMemcpyAsync(h->d_tw_inv, twi.data(), sizeof(float2) * N, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpyAsync(h->d_tw_fwd, twf.data(), sizeof(float2) * N, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpyAsync(h->d_wtab, wt.data(), N, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

int bioem_b200_create(const bioem_b200_config *cfg, int device, bioem_b200_handle *out)
{
  if (!cfg || !out)
    return fail(BIOEM_B200_ERR_INVALID, "null argument");
  *out = nullptr;
  const int N = cfg->NumberPixels;
  // (edges without an instantiated fused kernel -- odd, prime factors above 7, above 512 -- run on the direct-DFT
  // path; the reference accepts any edge, param.cpp:140-152)
  if (N < 2 || N > 4096)
    return fail(BIOEM_B200_ERR_INVALID, "NUMBER_PIXELS " + std::to_string(N) + " is out of range (2..4096)");
  if (cfg->GridSpaceCenter < 1 || cfg->maxDisplaceCenter < 0)
    return fail(BIOEM_B200_ERR_INVALID, "DISPLACE_CENTER: grid spacing must be >= 1 and the maximum displacement >= 0");
  if (2 * cfg->maxDisplaceCenter + 1 > N)
    return fail(BIOEM_B200_ERR_INVALID, "DISPLACE_CENTER: window larger than the image");
  int npos, nneg;
  window_counts(cfg->maxDisplaceCenter, cfg->GridSpaceCenter, &npos, &nneg);
  const int nw = npos + nneg;
  if (nw > 254)
    return fail(BIOEM_B200_ERR_INVALID, "displacement window has more than 254 points per axis");
  int ndev = bioem_b200_device_count();
  if (ndev == 0)
    return fail(BIOEM_B200_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev)
    return fail(BIOEM_B200_ERR_INVALID, "bad device index");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (smem_for(N, cfg->maxDisplaceCenter, nw + (nw & 1)) > (size_t) prop.sharedMemPerBlockOptin)
    return fail(BIOEM_B200_ERR_INVALID, "displacement window does not fit in shared memory for this image size");
  bioem_b200_context *h = new bioem_b200_context;
  h->cfg = *cfg;
  h->device = device;
  h->N = N;
  h->npos = npos;
  h->nw = nw;
  h->nwp = nw + (nw & 1);
  h->generic = is_generic(N);
  h->map4 = h->generic ? map4_generic(N) : map4_for(N);
  h->time_kernels = getenv("BIOEM_B200_KERNEL_TIMING") != nullptr && atoi(getenv("BIOEM_B200_KERNEL_TIMING")) != 0;
  const int rc = create_impl(h, cfg);
  if (rc != BIOEM_B200_OK)
  {
    const std::string msg = g_err; // destroy() must not lose the reason
    bioem_b200_destroy(h);
    return fail(rc, msg);
  }
  *out = h;
  return BIOEM_B200_OK;
}

int bioem_b200_destroy(bioem_b200_handle h)
{
  if (!h)
    return BIOEM_B200_OK;
  cudaSetDevice(h->device);
  if (h->stream)
    cudaStreamSynchronize(h->stream);
  nccl_release(h);
  free_batch(h);
  for (auto &ev : h->lik_events)
  {
    cudaEventDestroy(ev.first);
    cudaEventDestroy(ev.second);
  }
  for (auto &ev : h->event_pool)
    cudaEventDestroy(ev);
  dfree(h, h->d_skipped);
  dfree(h, h->d_gather);
  dfree(h, h->d_xyzr);
  dfree(h, h->d_dens);
  dfree(h, h->d_angles);
  dfree(h, h->d_ctf);
  dfree(h, h->d_kreal);
  dfree(h, h->d_prior);
  dfree(h, h->d_group);
  dfree(h, h->d_perm);
  dfree(h, h->d_refs);
  dfree(h, h->d_sumRef);
  dfree(h, h->d_sumsqRef);
  dfree(h, h->d_tw_inv);
  dfree(h, h->d_tw_fwd);
  dfree(h, h->d_wtab);
  dfree(h, h->d_wl);
  dfree(h, h->d_state);
  dfree(h, h->d_angtab);
  dfree(h, h->d_out);
  if (h->stream)
  {
    cudaStreamSynchronize(h->stream);
    cudaStreamDestroy(h->stream);
  }
  cudaGetLastError();
  delete h;
  return BIOEM_B200_OK;
}

int bioem_b200_upload_model(bioem_b200_handle h, const bioem_b200_model_point *pts, int A, float NormDen)
{
  if (!h || !pts || A <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_model: bad argument");
  CU(cudaSetDevice(h->device));
  std::vector<float4> xyzr(A);
  std::vector<float> dens(A);
  for (int i = 0; i < A; i++)
  {
    xyzr[i] = make_float4(pts[i].pos[0], pts[i].pos[1], pts[i].pos[2], pts[i].radius);
    dens[i] = pts[i].density;
  }
  h->A = 0; // stays 0 (run() refuses) unless everything below succeeds
  h->state_ready = false; // new inputs: the next run() starts from a fresh per-image state
  RC(dev_realloc(h, h->d_xyzr, (size_t) A));
  RC(dev_realloc(h, h->d_dens, (size_t) A));
  CU(cudaMemcpyAsync(h->d_xyzr, xyzr.data(), sizeof(float4) * A, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpyAsync(h->d_dens, dens.data(), sizeof(float) * A, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->A = A;
  h->NormDen = NormDen;
  return BIOEM_B200_OK;
}

int bioem_b200_upload_orientations(bioem_b200_handle h, const float *angles4, int O)
{
  if (!h || !angles4 || O <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_orientations: bad argument");
  CU(cudaSetDevice(h->device));
  const int Oold = h->O;
  h->O = 0;
  h->state_ready = false;
  if (O != Oold)
  {
    dfree(h, h->d_angtab);
    h->d_angtab = nullptr;
    dfree(h, h->d_skipped);
    h->d_skipped = nullptr;
    free_batch(h); // the batch size is clamped to the number of orientations
  }
  RC(dev_realloc(h, h->d_angles, (size_t) O));
  CU(cudaMemcpyAsync(h->d_angles, angles4, sizeof(float4) * O, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->h_angles.assign(reinterpret_cast<const float4 *>(angles4), reinterpret_cast<const float4 *>(angles4) + O);
  h->O = O;
  return BIOEM_B200_OK;
}

// upload_ctf and upload_ctf_groups (G groups of C / G rows)
static int upload_ctf_table(bioem_b200_context *h, const float *refCTF, const float *CtfParam4, int C, int G,
                            const float *cent, bool grouped)
{
  CU(cudaSetDevice(h->device));
  const int N = h->N;
  const size_t stdsz = (size_t) N * (N / 2 + 1);
  DevTmp tmp(h);
  RC(tmp.alloc(sizeof(float2) * stdsz * C));
  CU(cudaMemcpyAsync(tmp.p, refCTF, sizeof(float2) * stdsz * C, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->state_ready = false;
  const int Cold = h->C;
  h->C = 0;
  RC(dev_realloc(h, h->d_ctf, h->map4 * C));
  CU(do_pack(N, tmp.as<float2>(), h->d_ctf, C, h->stream));
  h->launches++;
  // CTFs computed in Fourier space are real (param.cpp:1540-1570): the fused kernel can then run in its
  // cached-product mode, for which the real parts are laid out in column-pass order
  bool real = true;
  for (size_t i = 0; i < stdsz * C && real; i++)
    real = refCTF[2 * i + 1] == 0.f;
  h->ctf_is_real = false;
  if (real && !h->generic)
  {
    size_t kr4 = 0;
    int ctas = 0;
    zgeo_for(N, 0, &kr4, &ctas);
    h->kr4 = kr4;
    RC(dev_realloc(h, h->d_kreal, kr4 * C));
    CU(do_kreal(N, h->d_ctf, h->d_kreal, C, h->stream));
    h->launches++;
    h->ctf_is_real = true;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->C = Cold;
  return set_ctf_priors(h, CtfParam4, C, G, cent, grouped);
}

int bioem_b200_upload_ctf(bioem_b200_handle h, const float *refCTF, const float *CtfParam4, int C)
{
  if (!h || !refCTF || !CtfParam4 || C <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf: bad argument");
  return upload_ctf_table(h, refCTF, CtfParam4, C, 1, nullptr, false);
}

int bioem_b200_upload_ctf_groups(bioem_b200_handle h, const float *refCTF, const float *CtfParam4, const float *Priordefcent,
                                 int G, int C)
{
  if (!h || !refCTF || !CtfParam4)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_groups: null handle or table");
  if (G < 1 || C < 1 || (long long) G * C > INT_MAX / 2)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_groups: G = " + std::to_string(G) + ", C = " + std::to_string(C) +
                                            ": need G >= 1 and C >= 1");
  if (h->generic)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_groups: NUMBER_PIXELS " + std::to_string(h->N) +
                                            " runs on the direct-DFT path, which takes no grouped CTF table");
  if (h->cfg.tousepsf)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_groups: USE_PSF kernels are complex; grouped tables must be real");
  const size_t n = (size_t) h->N * (h->N / 2 + 1) * G * C;
  for (size_t i = 0; i < n; i++)
    if (refCTF[2 * i + 1] != 0.f)
      return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_groups: row " + std::to_string(i / (n / ((size_t) G * C))) +
                                              " has a non-zero imaginary part; grouped tables must be real");
  return upload_ctf_table(h, refCTF, CtfParam4, G * C, G, Priordefcent, true);
}

int bioem_b200_upload_ctf_real(bioem_b200_handle h, const float *kernels, const float *CtfParam4, int C)
{
  if (!h || !kernels || !CtfParam4 || C <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_ctf_real: bad argument");
  CU(cudaSetDevice(h->device));
  const int N = h->N;
  const size_t n2 = (size_t) N * N;
  DevTmp img(h), scr(h);
  RC(img.alloc(sizeof(float) * n2 * C));
  RC(scr.alloc(sizeof(float2) * (size_t) N * (N / 2 + 1) * C));
  CU(cudaMemcpyAsync(img.p, kernels, sizeof(float) * n2 * C, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->state_ready = false;
  const int Cold = h->C;
  h->C = 0;
  h->ctf_is_real = false; // spectra of real-space kernels: complex in general
  RC(dev_realloc(h, h->d_ctf, h->map4 * C));
  CU(do_fft2d(N, img.as<float>(), nullptr, 0, 0.f, h->d_tw_fwd, scr.as<float2>(), h->d_ctf, C, h->stream));
  h->launches += 2;
  CU(cudaStreamSynchronize(h->stream));
  h->C = Cold;
  return set_ctf_priors(h, CtfParam4, C);
}

// Particle buffers for M images.  h->M stays 0 (run() refuses) until the upload that called this has
// succeeded and set it; a new particle stack always invalidates the running per-image state.
static int begin_particles(bioem_b200_context *h, int M, size_t *cap)
{
  h->state_ready = false;
  h->groups_set = false; // a new stack needs its own group list
  const bool same = (size_t) M == *cap && h->d_refs && h->d_sumRef && h->d_sumsqRef && h->d_state && h->d_out;
  h->M = 0;
  if (!same)
  {
    *cap = 0;
    dfree(h, h->d_angtab);
    h->d_angtab = nullptr;
    free_batch(h);
    RC(dev_realloc(h, h->d_refs, h->map4 * (size_t) M));
    RC(dev_realloc(h, h->d_sumRef, (size_t) M));
    RC(dev_realloc(h, h->d_sumsqRef, (size_t) M));
    RC(dev_realloc(h, h->d_state, (size_t) M));
    RC(dev_realloc(h, h->d_out, (size_t) M));
    *cap = (size_t) M;
  }
  return BIOEM_B200_OK;
}

int bioem_b200_upload_particles(bioem_b200_handle h, const float *maps, int M)
{
  if (!h || !maps || M <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_particles: bad argument");
  CU(cudaSetDevice(h->device));
  RC(begin_particles(h, M, &h->particle_cap));
  const int N = h->N;
  const size_t n2 = (size_t) N * N;
  // chunked so that the real-space staging stays small next to 180 GB of HBM
  const int chunk = (int) std::max<size_t>(1, std::min<size_t>((size_t) M, ((size_t) 1 << 30) / (n2 * 4)));
  DevTmp img(h), scr(h);
  RC(img.alloc(sizeof(float) * n2 * chunk));
  RC(scr.alloc(sizeof(float2) * (size_t) N * (N / 2 + 1) * chunk));
  for (int m0 = 0; m0 < M; m0 += chunk)
  {
    const int mc = std::min(chunk, M - m0);
    CU(cudaMemcpyAsync(img.p, maps + (size_t) m0 * n2, sizeof(float) * n2 * mc, cudaMemcpyHostToDevice, h->stream));
    image_sums_kernel<<<(mc + 63) / 64, 64, 0, h->stream>>>(img.as<float>(), (int) n2, mc, h->d_sumRef + m0, h->d_sumsqRef + m0);
    CU(cudaGetLastError());
    CU(do_fft2d(N, img.as<float>(), nullptr, 0, 0.f, h->d_tw_fwd, scr.as<float2>(), h->d_refs + (size_t) m0 * h->map4, mc,
                h->stream));
    h->launches += 3;
    CU(cudaStreamSynchronize(h->stream));
  }
  h->M = M;
  return BIOEM_B200_OK;
}

int bioem_b200_upload_particles_mrc(bioem_b200_handle h, const float *raw, int M, int normalise)
{
  if (!h || !raw || M <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_particles_mrc: bad argument");
  CU(cudaSetDevice(h->device));
  RC(begin_particles(h, M, &h->particle_cap));
  const int N = h->N;
  const size_t n2 = (size_t) N * N;
  const int chunk = (int) std::max<size_t>(1, std::min<size_t>((size_t) M, ((size_t) 1 << 29) / (n2 * 4)));
  DevTmp t_raw(h), t_img(h), t_mean(h), t_dev(h), t_scr(h);
  RC(t_raw.alloc(sizeof(float) * n2 * chunk));
  RC(t_img.alloc(sizeof(float) * n2 * chunk));
  RC(t_mean.alloc(sizeof(float) * chunk));
  RC(t_dev.alloc(sizeof(float) * chunk));
  RC(t_scr.alloc(sizeof(float2) * (size_t) N * (N / 2 + 1) * chunk));
  float *d_raw = t_raw.as<float>(), *d_img = t_img.as<float>(), *d_mean = t_mean.as<float>(), *d_dev = t_dev.as<float>();
  for (int m0 = 0; m0 < M; m0 += chunk)
  {
    const int mc = std::min(chunk, M - m0);
    CU(cudaMemcpyAsync(d_raw, raw + (size_t) m0 * n2, sizeof(float) * n2 * mc, cudaMemcpyHostToDevice, h->stream));
    if (normalise)
      mrc_stats_kernel<<<(mc + 63) / 64, 64, 0, h->stream>>>(d_raw, (int) n2, mc, d_mean, d_dev);
    dim3 tg((N + 31) / 32, (N + 31) / 32, mc);
    mrc_transpose_kernel<<<tg, dim3(32, 8), 0, h->stream>>>(d_raw, d_mean, d_dev, N, normalise, d_img);
    image_sums_kernel<<<(mc + 63) / 64, 64, 0, h->stream>>>(d_img, (int) n2, mc, h->d_sumRef + m0, h->d_sumsqRef + m0);
    CU(cudaGetLastError());
    CU(do_fft2d(N, d_img, nullptr, 0, 0.f, h->d_tw_fwd, t_scr.as<float2>(), h->d_refs + (size_t) m0 * h->map4, mc, h->stream));
    h->launches += 5;
    CU(cudaStreamSynchronize(h->stream));
  }
  h->M = M;
  return BIOEM_B200_OK;
}

int bioem_b200_upload_particles_fft(bioem_b200_handle h, const float *fft, const float *sum, const float *sumsq, int M)
{
  if (!h || !fft || !sum || !sumsq || M <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "upload_particles_fft: bad argument");
  CU(cudaSetDevice(h->device));
  RC(begin_particles(h, M, &h->particle_cap));
  const int N = h->N;
  const size_t stdsz = (size_t) N * (N / 2 + 1);
  const int chunk = (int) std::max<size_t>(1, std::min<size_t>((size_t) M, ((size_t) 1 << 30) / (stdsz * 8)));
  DevTmp tmp(h);
  RC(tmp.alloc(sizeof(float2) * stdsz * chunk));
  for (int m0 = 0; m0 < M; m0 += chunk)
  {
    const int mc = std::min(chunk, M - m0);
    CU(cudaMemcpyAsync(tmp.p, fft + (size_t) m0 * stdsz * 2, sizeof(float2) * stdsz * mc, cudaMemcpyHostToDevice, h->stream));
    CU(do_pack(N, tmp.as<float2>(), h->d_refs + (size_t) m0 * h->map4, mc, h->stream));
    h->launches++;
    CU(cudaStreamSynchronize(h->stream));
  }
  CU(cudaMemcpyAsync(h->d_sumRef, sum, sizeof(float) * M, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpyAsync(h->d_sumsqRef, sumsq, sizeof(float) * M, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->M = M;
  return BIOEM_B200_OK;
}

int bioem_b200_set_particle_groups(bioem_b200_handle h, const int *group, int M)
{
  if (!h || !group)
    return fail(BIOEM_B200_ERR_INVALID, "set_particle_groups: null handle or list");
  if (h->M <= 0 || !h->grouped || h->C <= 0)
    return fail(BIOEM_B200_ERR_STATE, "set_particle_groups: upload the particles and a grouped CTF table first");
  if (M != h->M)
    return fail(BIOEM_B200_ERR_INVALID, "set_particle_groups: " + std::to_string(M) + " entries for " + std::to_string(h->M) +
                                            " particles");
  int gmax = -1;
  for (int m = 0; m < M; m++)
  {
    if (group[m] < 0 || group[m] >= h->G)
      return fail(BIOEM_B200_ERR_INVALID, "set_particle_groups: particle " + std::to_string(m) + ": group " +
                                              std::to_string(group[m]) + " out of range [0, " + std::to_string(h->G) + ")");
    gmax = std::max(gmax, group[m]);
  }
  CU(cudaSetDevice(h->device));
  h->state_ready = false;
  h->groups_set = false;
  // CTAs take the particles group by group: the resident ones share one or two groups' tables in L2
  std::vector<int> perm((size_t) M);
  for (int m = 0; m < M; m++)
    perm[m] = m;
  std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return group[a] < group[b]; });
  RC(dev_realloc(h, h->d_group, (size_t) M));
  RC(dev_realloc(h, h->d_perm, (size_t) M));
  CU(cudaMemcpyAsync(h->d_group, group, sizeof(int) * M, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_perm, perm.data(), sizeof(int) * M, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->group_max = gmax;
  h->groups_set = true;
  return BIOEM_B200_OK;
}

static int ensure_batch(bioem_b200_context *h)
{
  if (h->OB > 0)
    return BIOEM_B200_OK;
  // a grouped table runs in cached-product mode only (its kernels are real and the fused kernel's grouped variant is a
  // cached-product one): the environment cannot switch that mode off for it
  if (h->grouped && getenv("BIOEM_B200_CACHED_PRODUCT") && atoi(getenv("BIOEM_B200_CACHED_PRODUCT")) == 0)
    return fail(BIOEM_B200_ERR_INVALID, "run: a grouped CTF table needs the cached-product mode; "
                                        "BIOEM_B200_CACHED_PRODUCT=0 is not supported with it");
  const int N = h->N;
  const size_t mapbytes = h->map4 * sizeof(float4);
  // Orientations per batch: the conv spectra of a batch live in HBM (1 GB budget); what has to stay
  // in L2 is only the group of orientations the resident CTAs are working on (CTAs are numbered
  // image-fastest, so all images pass over one group before the next), i.e. a few MB.  Measured on
  // cfg2: 15 orientations per launch 18.93, 60: 19.21, 150: 19.26 M likelihoods/s (fewer launch tails).
  size_t budget = (size_t) 1 << 30;
  // experiment knobs; a value that does not parse to a positive number is ignored
  auto env_pos = [](const char *name) -> long {
    const char *v = getenv(name);
    if (!v)
      return 0;
    char *end = nullptr;
    const long x = strtol(v, &end, 10);
    return (end != v && x > 0) ? x : 0;
  };
  if (env_pos("BIOEM_B200_CONV_MB"))
    budget = (size_t) env_pos("BIOEM_B200_CONV_MB") << 20;
  long ob = (long) (budget / (mapbytes * (size_t) h->C));
  // a grouped table keeps no conv spectra: per orientation a batch holds its projection (image, r2c scratch, packed
  // spectrum), its G x C conv parameters and at most one partial per particle
  if (h->grouped)
    ob = (long) (budget / ((size_t) N * N * sizeof(float) + (size_t) N * (N / 2 + 1) * sizeof(float2) + mapbytes +
                           (size_t) h->C * sizeof(ConvParam) + (size_t) h->M * sizeof(Running)));
  ob = std::max<long>(1, std::min<long>(ob, h->O));
  if (env_pos("BIOEM_B200_OB"))
    ob = std::max<long>(1, std::min<long>(env_pos("BIOEM_B200_OB"), h->O));
  if (h->generic)
  {
    // direct-DFT path: the correlation windows of a batch go through HBM (same budget), one grid row per conv spectrum
    const size_t per_o = (size_t) h->C * h->M * h->nw * h->nw * sizeof(float);
    ob = std::max<long>(1, std::min<long>(ob, (long) (budget / std::max<size_t>(per_o, 1))));
    ob = std::max<long>(1, std::min<long>(ob, 65535 / std::max(1, h->C)));
  }
  h->OB = (int) ob;
  // orientations per CTA: amortise the CTA prologue (and the one likelihood per CTA whose first radix pass
  // cannot be run ahead) over >= 64 likelihoods, keep >= 4 waves (cfg2: 1 -> 2 orientations, +0.5 %)
  // (above N = 224, one CTA per SM, more than one orientation per CTA at 32 CTFs costs 3-5 %)
  const int per_cta = h->N <= 224 ? 64 : 16;
  int og = std::max(1, (per_cta + h->Cg - 1) / h->Cg);
  const long long cta_slots = h->N <= 128 ? 592 : h->N <= 224 ? 296 : 148; // resident CTAs of the fused kernel per GPU
  while (og > 1 && (long long) h->M * ((h->OB + og - 1) / og) < 4LL * cta_slots)
    og--;
  if (env_pos("BIOEM_B200_OG"))
    og = (int) env_pos("BIOEM_B200_OG");
  h->OG = og;
  // Bands of image rows per projection CTA.  Every warp of a band walks the model points that touch the band IN
  // ORDER (a serial chain), so what hides its latency is the number of resident warps: aim at >= 4 x 148 CTAs per
  // launch, within 24 KB of band per CTA.  Large batches (cfg 2: 165 orientations) reach that with 9 bands of 26
  // rows and 8 warps; small batches of a big model (cfg 4: 8 orientations of 110,592 voxels) get 90 bands of 4 rows
  // with one row per warp -- 3.7 ms per orientation with the 22 bands of 17 rows this used to launch.
  size_t band_budget = 24 * 1024;
  if (env_pos("BIOEM_B200_BAND_KB"))
    band_budget = (size_t) env_pos("BIOEM_B200_BAND_KB") * 1024;
  const int by_budget = (int) (((size_t) N * N * 4 + band_budget - 1) / band_budget);
  const int by_ctas = (int) std::min<long>((4 * 148 + h->OB - 1) / h->OB, N);
  h->nbands = std::max(1, std::max(by_budget, by_ctas));
  h->band_rows = (N + h->nbands - 1) / h->nbands;
  if (h->band_rows < 8)
  { // one row per warp, a power of two of warps (the kernel splits its point tiles evenly over the warps)
    int r = 1;
    while (2 * r <= h->band_rows)
      r *= 2;
    h->band_rows = r;
  }
  h->nbands = (N + h->band_rows - 1) / h->band_rows;
  h->proj_threads = 32 * std::min(8, h->band_rows);
  const int OB = h->OB;
  h->OB = 0; // a failed allocation below leaves "no batch buffers" behind, not a half-built set
  RC(dev_realloc(h, h->d_proj, (size_t) N * N * OB));
  RC(dev_realloc(h, h->d_tempden, (size_t) h->nbands * OB));
  RC(dev_realloc(h, h->d_scratch, (size_t) N * (N / 2 + 1) * OB));
  RC(dev_realloc(h, h->d_projfft, h->map4 * OB));
  // Cached-product mode (real CTF tables): per orientation the fused kernel forms projection * conj(particle) once
  // (about 0.12 likelihoods' worth of work) and saves about 5 % per likelihood -- worth it from 4 CTFs on.  The
  // convolved spectra are then never formed: no OB x C conv maps in HBM (cfg 2: 1 GB), one scratch map per resident CTA.
  bool zmode = h->ctf_is_real && h->d_kreal && h->C >= 4;
  if (const char *v = getenv("BIOEM_B200_CACHED_PRODUCT"))
    zmode = h->ctf_is_real && h->d_kreal && atoi(v) != 0;
  if (h->grouped)
    zmode = true;
  if (h->generic)
  {
    zmode = false;
    RC(dev_realloc(h, h->d_values, (size_t) OB * h->C * h->M * h->nw * h->nw));
  }
  if (zmode)
  {
    int dev_sms = 0, ctas = 0;
    size_t kr4 = 0;
    CU(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, h->device));
    zgeo_for(N, smem_for(N, h->cfg.maxDisplaceCenter, h->nwp), &kr4, &ctas);
    const int nslots = dev_sms * ctas;
    RC(dev_realloc(h, h->d_zbuf, h->map4 * (size_t) nslots));
    RC(dev_realloc(h, h->d_zflags, (size_t) nslots));
    CU(cudaMemsetAsync(h->d_zflags, 0, sizeof(int) * (size_t) nslots, h->stream));
    h->nslots = nslots;
  }
  // (in that mode only the inspection entry point debug_convolved wants convolved spectra: one orientation's worth)
  // (a grouped table: one conv spectrum, debug_convolved forms the one it is asked for)
  RC(dev_realloc(h, h->d_conv, h->map4 * (size_t) (zmode ? 1 : OB) * (h->grouped ? 1 : h->C)));
  RC(dev_realloc(h, h->d_cpar, (size_t) OB * h->C));
  h->partials_cap = (size_t) h->M * ((OB + h->OG - 1) / h->OG);
  RC(dev_realloc(h, h->d_partials, h->partials_cap));
  h->OB = OB;
  h->zmode = zmode;
  return BIOEM_B200_OK;
}

int bioem_b200_reset(bioem_b200_handle h)
{
  if (!h || h->M <= 0)
    return fail(BIOEM_B200_ERR_STATE, "reset: upload particles first");
  CU(cudaSetDevice(h->device));
  init_state_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_state, h->M);
  CU(cudaGetLastError());
  h->launches++;
  if (h->cfg.writeAngles)
  {
    if (h->O <= 0)
      return fail(BIOEM_B200_ERR_STATE, "reset: upload orientations first");
    const size_t n = (size_t) h->O * h->M;
    if (!h->d_angtab)
      RC(dev_realloc(h, h->d_angtab, n));
    init_angles_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, h->stream>>>(h->d_angtab, n);
    CU(cudaGetLastError());
    h->launches++;
  }
  if (h->O > 0)
  {
    if (!h->d_skipped)
      RC(dev_realloc(h, h->d_skipped, (size_t) h->O));
    CU(cudaMemsetAsync(h->d_skipped, 0, sizeof(int) * (size_t) h->O, h->stream));
  }
  h->launches = 0;
  h->likelihoods = 0;
  h->lik_launches = 0;
  h->argmax_exact = true;
  h->state_ready = true;
  return BIOEM_B200_OK;
}

// stages 1 + 2 for orientations [o0, o0+OBcur) into the batch buffers
// (conv_dst: where the convolved spectra go when want_conv is set, instead of the batch buffer -- render_maps in
// cached-product mode, whose batch buffer holds one orientation's worth)
static int run_front(bioem_b200_context *h, int o0, int OBcur, const float4 *angles = nullptr, const int4 *sel = nullptr,
                     int nsel = 0, bool want_conv = false, float4 *conv_dst = nullptr)
{
  const int N = h->N;
  ProjParams pp;
  pp.xyzr = h->d_xyzr;
  pp.dens = h->d_dens;
  pp.angles = angles ? angles : h->d_angles; // (a private list: the exact arg-max pass)
  pp.proj = h->d_proj;
  pp.tempden = h->d_tempden;
  pp.skipped = angles ? nullptr : h->d_skipped; // indexed by the absolute orientation number
  pp.A = h->A;
  pp.N = N;
  pp.band_rows = h->band_rows;
  pp.nbands = h->nbands;
  pp.o_base = o0;
  pp.doquater = h->cfg.doquater;
  pp.shiftX = h->cfg.shiftX;
  pp.shiftY = h->cfg.shiftY;
  pp.pixelSize = h->cfg.pixelSize;
  dim3 pg(OBcur, h->nbands);
  // the attribute belongs to the function, not to this handle: other handles (other image sizes)
  // may have changed it since, so it is set at every launch
  CU(cudaFuncSetAttribute(project_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ((size_t) h->band_rows * N * 4)));
  project_kernel<<<pg, h->proj_threads, (size_t) h->band_rows * N * 4, h->stream>>>(pp);
  CU(cudaGetLastError());
  CU(do_fft2d(N, h->d_proj, h->d_tempden, h->nbands, h->NormDen, h->d_tw_fwd, h->d_scratch, h->d_projfft, OBcur, h->stream));
  float4 *conv = (h->zmode && !want_conv) ? nullptr : h->d_conv; // (want_conv in cached-product mode: OBcur == 1)
  if (want_conv && conv_dst)
    conv = conv_dst;
  if (h->grouped && !conv && !sel)
    CU(do_sums(N, h->d_projfft, h->d_ctf, h->d_prior, h->d_cpar, h->C, OBcur, h->cfg.Ntotpi, h->stream));
  else
    CU(do_conv(N, h->d_projfft, h->d_ctf, h->d_prior, conv, h->d_cpar, h->C, OBcur, h->cfg.Ntotpi, h->stream, sel, nsel));
  h->launches += 4;
  return BIOEM_B200_OK;
}

static void fill_lik_params(bioem_b200_context *h, LikParams &lp, int o0, int OBcur)
{
  const int N = h->N;
  lp.convs = h->d_conv;
  lp.refs = h->d_refs;
  lp.cpar = h->d_cpar;
  lp.sumRef = h->d_sumRef;
  lp.sumsqRef = h->d_sumsqRef;
  lp.tw_inv = h->d_tw_inv;
  lp.wtab = h->d_wtab;
  lp.partials = h->d_partials;
  lp.angles = h->cfg.writeAngles ? h->d_angtab : nullptr;
  lp.dbg_values = nullptr;
  lp.pairs = nullptr;
  lp.projs = h->d_projfft;
  lp.kreal = h->d_kreal;
  lp.zbuf = h->d_zbuf;
  lp.zflags = h->d_zflags;
  lp.nslots = h->nslots;
  lp.kr4 = (int) h->kr4;
  lp.zmode = h->zmode ? 1 : 0;
  lp.M = h->M;
  lp.C = h->Cg; // rows per particle; the grouped variant's particles take theirs out of lp.GC
  lp.GC = h->C;
  lp.group = h->grouped ? h->d_group : nullptr;
  lp.perm = h->grouped ? h->d_perm : nullptr;
  lp.OBcur = OBcur;
  lp.OG = h->OG;
  lp.o_base = o0;
  lp.nw = h->nw;
  lp.nwp = h->nwp;
  lp.Ntotpi = h->cfg.Ntotpi;
  lp.invNN = 1.0f / (float) (N * N);
  lp.acoef_d = (double) (3.f - h->cfg.Ntotpi) * 0.5;
  lp.ex2coef = (float) (lp.acoef_d * 1.4426950408889634074);
}

// stages 3-5 of one batch on the direct-DFT path: correlation windows into d_values, then calc_logpro + calProb per
// particle in (orientation, CTF) order straight into the running state (the record carries its displacement: there
// is no separate exact arg-max pass on this path)
static int gen_corr_launch(bioem_b200_context *h, const float4 *refs, int M, int nspec, float *values)
{
  const int N = h->N;
  const size_t smem = gen_corr_smem(N, h->nw);
  CU(cudaFuncSetAttribute(gen_corr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
  gen_corr_kernel<<<dim3(M, nspec), 256, smem, h->stream>>>(reinterpret_cast<const float2 *>(h->d_conv),
                                                            reinterpret_cast<const float2 *>(refs), h->d_tw_inv, h->d_wl, N,
                                                            2 * h->map4, h->nw, M, 1.0f / (float) (N * N), values);
  CU(cudaGetLastError());
  return BIOEM_B200_OK;
}
static int run_generic_batch(bioem_b200_context *h, int o0, int OBcur)
{
  RC(gen_corr_launch(h, h->d_refs, h->M, OBcur * h->C, h->d_values));
  gen_fold_kernel<<<h->M, 128, 0, h->stream>>>(h->d_values, h->d_cpar, h->d_sumRef, h->d_sumsqRef, OBcur, h->C, h->M, h->nw, o0,
                                               h->cfg.Ntotpi, (double) (3.f - h->cfg.Ntotpi) * 0.5, h->d_state,
                                               h->cfg.writeAngles ? h->d_angtab : nullptr);
  CU(cudaGetLastError());
  h->launches += 2;
  h->likelihoods += (long long) OBcur * h->C * h->M;
  return BIOEM_B200_OK;
}

// run() for orientations [oBegin, oEnd); capture != nullptr (inspection): every correlation value lCC/N^2 of the range
// is copied out as well, capture[o - oBegin][c][m][nw*nw], in the window order of debug_correlation
static int run_range(bioem_b200_context *h, int oBegin, int oEnd, float *capture)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "run: null handle");
  if (h->A <= 0 || h->O <= 0 || h->C <= 0 || h->M <= 0)
    return fail(BIOEM_B200_ERR_STATE, "run: model, orientations, CTF table and particles must be uploaded first");
  if (h->grouped && !h->groups_set)
    return fail(BIOEM_B200_ERR_STATE, "run: a grouped CTF table needs the particles' groups (set_particle_groups)");
  if (oBegin < 0 || oEnd > h->O || oBegin > oEnd)
    return fail(BIOEM_B200_ERR_INVALID, "run: orientation range out of bounds");
  CU(cudaSetDevice(h->device));
  if (!h->state_ready)
  {
    int rc = bioem_b200_reset(h);
    if (rc)
      return rc;
  }
  int rc = ensure_batch(h);
  if (rc)
    return rc;
  for (int o0 = oBegin; o0 < oEnd; o0 += h->OB)
  {
    const int OBcur = std::min(h->OB, oEnd - o0);
    rc = run_front(h, o0, OBcur);
    if (rc)
      return rc;
    // capture: the batch's windows land in a temp (fused kernel) or in d_values (direct-DFT path), prefilled with
    // 0xFF bytes -- a NaN -- so that an entry the kernel does not write shows up
    const size_t ncap = capture ? (size_t) OBcur * h->Cg * h->M * h->nw * h->nw : 0;
    DevTmp t_cap(h);
    float *d_cap = nullptr;
    if (capture)
    {
      if (!h->generic)
        RC(t_cap.alloc(sizeof(float) * ncap));
      d_cap = h->generic ? h->d_values : t_cap.as<float>();
      CU(cudaMemsetAsync(d_cap, 0xFF, sizeof(float) * ncap, h->stream));
    }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (h->time_kernels)
    {
      for (cudaEvent_t *e : {&e0, &e1})
      {
        if (!h->event_pool.empty())
        {
          *e = h->event_pool.back();
          h->event_pool.pop_back();
        }
        else
          CU(cudaEventCreate(e));
      }
      CU(cudaEventRecord(e0, h->stream));
    }
    LikParams lp;
    fill_lik_params(h, lp, o0, OBcur);
    if (capture && !h->generic)
      lp.dbg_values = d_cap;
    const int NG = (OBcur + h->OG - 1) / h->OG;
    if (h->generic)
    {
      rc = run_generic_batch(h, o0, OBcur);
      if (rc)
        return rc;
    }
    else
      CU(do_lik(h->N, lp, h->M * NG, h->cfg.maxDisplaceCenter, h->stream));
    if (h->time_kernels)
    {
      CU(cudaEventRecord(e1, h->stream));
      h->lik_events.emplace_back(e0, e1);
    }
    h->lik_launches += 1;
    if (capture)
    {
      CU(cudaMemcpyAsync(capture + (size_t) (o0 - oBegin) * h->Cg * h->M * h->nw * h->nw, d_cap, sizeof(float) * ncap,
                         cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
    }
    if (h->generic)
      continue;
    merge_partials_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_partials, NG, h->M, h->d_state);
    CU(cudaGetLastError());
    h->launches += 2;
    h->likelihoods += (long long) OBcur * h->Cg * h->M;
    h->argmax_exact = false;
  }
  return BIOEM_B200_OK;
}

int bioem_b200_run(bioem_b200_handle h, int oBegin, int oEnd) { return run_range(h, oBegin, oEnd, nullptr); }

// Exact first-of-ties displacement for the arg-max record of every particle (see exact_argmax_kernel): the
// winning (orientation, CTF) of each particle is evaluated once more by the fused kernel with its correlation
// window written out, then the reference's rule is applied to all of its displacements.  One extra likelihood
// per particle on top of nOrient x nCtf: cost below 0.1 % of a run.
static int refine_argmax(bioem_b200_context *h)
{
  if (h->argmax_exact || h->generic) // (direct-DFT path: every record already carries its exact displacement)
    return BIOEM_B200_OK;
  // (the fused kernel does not track displacements at all, so this pass is what fills them in)
  if (h->A <= 0 || h->O <= 0 || h->C <= 0 || h->M <= 0 || (int) h->h_angles.size() != h->O)
    return fail(BIOEM_B200_ERR_STATE, "download: the arg-max displacement is evaluated on this handle and needs its model, "
                                      "orientations, CTF table and particles (upload them before importing partials)");
  RC(ensure_batch(h));
  const int M = h->M;
  std::vector<Running> st((size_t) M);
  CU(cudaMemcpyAsync(st.data(), h->d_state, sizeof(Running) * (size_t) M, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  // particles ordered by winning orientation; distinct orientations are projected once
  std::vector<int> order;
  order.reserve(M);
  for (int m = 0; m < M; m++)
    if (st[m].Const > kMinProb && st[m].orient >= 0 && st[m].orient < h->O && st[m].conv >= 0 && st[m].conv < h->C)
      order.push_back(m);
  std::sort(order.begin(), order.end(), [&](int a, int b) {
    return st[a].orient != st[b].orient ? st[a].orient < st[b].orient : a < b;
  });
  const size_t nv = (size_t) h->nw * h->nw;
  DevTmp t_cnt(h);
  RC(t_cnt.alloc(sizeof(int) * 3));
  CU(cudaMemsetAsync(t_cnt.p, 0, sizeof(int) * 3, h->stream));
  size_t pos = 0;
  while (pos < order.size())
  {
    // one batch: up to OB distinct orientations
    std::vector<float4> ang;
    std::vector<RefineItem> items;
    int last = -1;
    while (pos < order.size())
    {
      const int m = order[pos];
      // the batch buffers hold OB projections and OB*C conv spectra (one conv slot per item here)
      if ((st[m].orient != last && (int) ang.size() == h->OB) || items.size() == (size_t) h->OB * h->C)
        break;
      if (st[m].orient != last)
      {
        ang.push_back(h->h_angles[st[m].orient]);
        last = st[m].orient;
      }
      RefineItem it;
      it.m = m;
      it.slot = (int) ang.size() - 1;
      it.conv = st[m].conv;
      it.pad = 0;
      items.push_back(it);
      pos++;
    }
    DevTmp t_ang(h), t_items(h), t_val(h), t_part(h);
    RC(t_ang.alloc(sizeof(float4) * ang.size()));
    RC(t_items.alloc(sizeof(RefineItem) * items.size()));
    RC(t_val.alloc(sizeof(float) * nv * items.size()));
    RC(t_part.alloc(sizeof(Running) * items.size()));
    CU(cudaMemcpyAsync(t_ang.p, ang.data(), sizeof(float4) * ang.size(), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(t_items.p, items.data(), sizeof(RefineItem) * items.size(), cudaMemcpyHostToDevice, h->stream));
    static_assert(sizeof(RefineItem) == sizeof(int4), "work item layout");
    RC(run_front(h, 0, (int) ang.size(), t_ang.as<float4>(), t_items.as<int4>(), (int) items.size()));
    LikParams lp;
    fill_lik_params(h, lp, 0, (int) items.size()); // one "orientation" of one CTF per item
    lp.C = 1;
    lp.OG = 1;
    lp.group = lp.perm = nullptr; // (the items name rows of the whole table)
    lp.pairs = t_items.as<int4>();
    lp.partials = t_part.as<Running>();
    lp.angles = nullptr;
    lp.dbg_values = t_val.as<float>();
    CU(do_lik(h->N, lp, (int) items.size(), h->cfg.maxDisplaceCenter, h->stream));
    exact_argmax_kernel<<<(unsigned) items.size(), 128, 0, h->stream>>>(t_items.as<RefineItem>(), t_val.as<float>(), h->d_cpar,
                                                                        h->d_sumRef, h->d_sumsqRef, h->C, h->nw, h->cfg.Ntotpi,
                                                                        lp.invNN, lp.acoef_d, h->d_state, t_cnt.as<int>());
    CU(cudaGetLastError());
    h->launches += 6;
    CU(cudaStreamSynchronize(h->stream)); // the host vectors of this batch go out of scope
  }
  CU(cudaMemcpyAsync(h->refine_counts, t_cnt.p, sizeof(int) * 3, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->argmax_exact = true;
  return BIOEM_B200_OK;
}

int bioem_b200_synchronize(bioem_b200_handle h)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

int bioem_b200_download(bioem_b200_handle h, bioem_b200_prob_map *maps_out, bioem_b200_prob_angle *angles_out)
{
  if (!h || !maps_out)
    return fail(BIOEM_B200_ERR_INVALID, "download: bad argument");
  if (!h->state_ready)
    return fail(BIOEM_B200_ERR_STATE, "download: nothing has been run");
  CU(cudaSetDevice(h->device));
  static_assert(sizeof(ProbMapOut) == sizeof(bioem_b200_prob_map) && sizeof(ProbMapOut) == 40, "result layout");
  static_assert(sizeof(ProbAngleOut) == sizeof(bioem_b200_prob_angle) && sizeof(ProbAngleOut) == 16, "result layout");
  RC(refine_argmax(h));
  finalize_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_state, h->d_sumRef, h->M, h->nw, h->npos,
                                                            h->cfg.maxDisplaceCenter, h->cfg.GridSpaceCenter, h->cfg.Ntotpi,
                                                            h->d_out);
  CU(cudaGetLastError());
  h->launches++;
  CU(cudaMemcpyAsync(maps_out, h->d_out, sizeof(ProbMapOut) * h->M, cudaMemcpyDeviceToHost, h->stream));
  if (angles_out && h->cfg.writeAngles && h->d_angtab)
    CU(cudaMemcpyAsync(angles_out, h->d_angtab, sizeof(ProbAngleOut) * (size_t) h->O * h->M, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

// Calculated images of arbitrary records (bioem_b200.h).  Records are sorted by orientation and taken in batches of
// at most OB distinct orientations and OB * C images, as the exact arg-max pass does: every distinct orientation is
// projected once into the batch buffers (a private orientation list, no out-of-frame counting), each image's conv
// spectrum is formed by the selection path of the conv kernel (a slot per image; on the direct-DFT path every CTF
// of the batch's orientations), then transformed back and copied out.  Nothing of the running state is touched.
int bioem_b200_render_maps(bioem_b200_handle h, const bioem_b200_prob_map *records, int n, float *maps_out)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "render_maps: null handle");
  if (n < 0)
    return fail(BIOEM_B200_ERR_INVALID, "render_maps: negative record count " + std::to_string(n));
  if (n > 0 && (!records || !maps_out))
    return fail(BIOEM_B200_ERR_INVALID, "render_maps: null records or output");
  if (h->A <= 0 || h->O <= 0 || h->C <= 0 || (int) h->h_angles.size() != h->O)
    return fail(BIOEM_B200_ERR_STATE, "render_maps: model, orientations and CTF table must be uploaded first");
  const int N = h->N;
  for (int i = 0; i < n; i++)
  {
    const bioem_b200_prob_map &r = records[i];
    if (r.max_prob_orient < 0 || r.max_prob_orient >= h->O)
      return fail(BIOEM_B200_ERR_INVALID, "render_maps: record " + std::to_string(i) + ": orientation " +
                                              std::to_string(r.max_prob_orient) + " out of range [0, " + std::to_string(h->O) + ")");
    if (r.max_prob_conv < 0 || r.max_prob_conv >= h->C)
      return fail(BIOEM_B200_ERR_INVALID, "render_maps: record " + std::to_string(i) + ": CTF " + std::to_string(r.max_prob_conv) +
                                              " out of range [0, " + std::to_string(h->C) + ")");
    if (r.max_prob_cent_x <= -N || r.max_prob_cent_x >= N || r.max_prob_cent_y <= -N || r.max_prob_cent_y >= N)
      return fail(BIOEM_B200_ERR_INVALID, "render_maps: record " + std::to_string(i) + ": displacement (" +
                                              std::to_string(r.max_prob_cent_x) + ", " + std::to_string(r.max_prob_cent_y) +
                                              ") not inside (-" + std::to_string(N) + ", " + std::to_string(N) + ")");
  }
  if (n == 0)
    return BIOEM_B200_OK;
  CU(cudaSetDevice(h->device));
  RC(ensure_batch(h));
  // (the front end counts its launches; stats() describes run() and stays as it was)
  struct KeepLaunches
  {
    bioem_b200_context *h;
    long long v;
    ~KeepLaunches() { h->launches = v; }
  } keep{h, h->launches};
  std::vector<int> order((size_t) n);
  for (int i = 0; i < n; i++)
    order[i] = i;
  std::stable_sort(order.begin(), order.end(),
                   [&](int a, int b) { return records[a].max_prob_orient < records[b].max_prob_orient; });
  // images per batch: OB * C conv slots, and the 65535 grid rows of the kernels
  const int cap = (int) std::min<long long>({(long long) h->OB * h->C, (long long) n, 65535LL});
  const size_t n2 = (size_t) N * N;
  DevTmp t_out(h), t_scr(h), t_items(h), t_sel(h), t_ang(h), t_conv(h);
  RC(t_out.alloc(sizeof(float) * n2 * cap));
  RC(t_scr.alloc(sizeof(float2) * (size_t) N * (N / 2 + 1) * cap));
  RC(t_items.alloc(sizeof(RenderItem) * cap));
  RC(t_sel.alloc(sizeof(int4) * cap));
  RC(t_ang.alloc(sizeof(float4) * h->OB));
  // the fused path's conv spectra: the batch buffer holds OB * C of them, except in cached-product mode (one
  // orientation's worth)
  float4 *convs = h->d_conv;
  if (!h->generic && h->zmode)
  {
    RC(t_conv.alloc(sizeof(float4) * h->map4 * cap));
    convs = t_conv.as<float4>();
  }
  size_t pos = 0;
  while (pos < order.size())
  {
    std::vector<float4> ang;
    std::vector<int4> sel;
    std::vector<RenderItem> items;
    const size_t first = pos;
    int last = -1;
    while (pos < order.size())
    {
      const bioem_b200_prob_map &r = records[order[pos]];
      if ((r.max_prob_orient != last && (int) ang.size() == h->OB) || (int) items.size() == cap)
        break;
      if (r.max_prob_orient != last)
      {
        ang.push_back(h->h_angles[r.max_prob_orient]);
        last = r.max_prob_orient;
      }
      const int ob = (int) ang.size() - 1;
      RenderItem it;
      it.slot = h->generic ? ob * h->C + r.max_prob_conv : (int) items.size();
      it.sx = (r.max_prob_cent_x + N) % N;
      it.sy = (r.max_prob_cent_y + N) % N;
      it.norm = r.max_prob_norm;
      it.mu = r.max_prob_mu;
      sel.push_back(make_int4(order[pos], ob, r.max_prob_conv, 0));
      items.push_back(it);
      pos++;
    }
    const int ni = (int) items.size();
    // output slots in ascending record order: consecutive records land next to each other (all of them, when the
    // whole call fits one batch) and go back to the caller in one copy per run
    std::vector<int> recs(order.begin() + first, order.begin() + pos);
    std::sort(recs.begin(), recs.end());
    for (int b = 0; b < ni; b++)
      items[b].out = (int) (std::lower_bound(recs.begin(), recs.end(), order[first + b]) - recs.begin());
    CU(cudaMemcpyAsync(t_ang.p, ang.data(), sizeof(float4) * ang.size(), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(t_items.p, items.data(), sizeof(RenderItem) * ni, cudaMemcpyHostToDevice, h->stream));
    if (h->generic) // (no selection path here: every CTF of the batch's orientations, slot ob * C + c)
      RC(run_front(h, 0, (int) ang.size(), t_ang.as<float4>()));
    else
    {
      CU(cudaMemcpyAsync(t_sel.p, sel.data(), sizeof(int4) * ni, cudaMemcpyHostToDevice, h->stream));
      RC(run_front(h, 0, (int) ang.size(), t_ang.as<float4>(), t_sel.as<int4>(), ni, true, convs));
    }
    CU(do_render(N, convs, t_items.as<RenderItem>(), h->d_tw_inv, t_scr.as<float2>(), t_out.as<float>(), ni, h->stream));
    for (int b = 0; b < ni;)
    {
      int e = b + 1;
      while (e < ni && recs[e] == recs[e - 1] + 1)
        e++;
      CU(cudaMemcpyAsync(maps_out + (size_t) recs[b] * n2, t_out.as<float>() + (size_t) b * n2, sizeof(float) * n2 * (e - b),
                         cudaMemcpyDeviceToHost, h->stream));
      b = e;
    }
    CU(cudaStreamSynchronize(h->stream)); // the host vectors of this batch go out of scope
  }
  return BIOEM_B200_OK;
}

int bioem_b200_download_top_angles(bioem_b200_handle h, int oBegin, int oEnd, int K, bioem_b200_top_angle *out)
{
  if (!h || !out || K <= 0 || oBegin < 0 || oEnd > (h ? h->O : 0) || oBegin > oEnd)
    return fail(BIOEM_B200_ERR_INVALID, "download_top_angles: bad argument");
  if (!h->cfg.writeAngles || !h->d_angtab)
    return fail(BIOEM_B200_ERR_STATE, "download_top_angles: the handle was created with writeAngles == 0");
  if (!h->state_ready)
    return fail(BIOEM_B200_ERR_STATE, "download_top_angles: nothing has been run");
  static_assert(sizeof(TopAngleOut) == sizeof(bioem_b200_top_angle) && sizeof(TopAngleOut) == 24, "result layout");
  CU(cudaSetDevice(h->device));
  const size_t n = (size_t) h->M * K;
  DevTmp key(h), top(h);
  RC(key.alloc(n * sizeof(double)));
  RC(top.alloc(n * sizeof(TopAngleOut)));
  top_angles_kernel<<<(h->M + 63) / 64, 64, 0, h->stream>>>(h->d_angtab, h->M, oBegin, oEnd, K, key.as<double>(),
                                                           top.as<TopAngleOut>());
  CU(cudaGetLastError());
  h->launches++;
  CU(cudaMemcpyAsync(out, top.p, n * sizeof(TopAngleOut), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

size_t bioem_b200_partial_bytes(bioem_b200_handle h) { return h ? sizeof(Running) * (size_t) h->M : 0; }

int bioem_b200_export_partial(bioem_b200_handle h, void *device_dst)
{
  if (!h || !device_dst || !h->state_ready)
    return fail(BIOEM_B200_ERR_STATE, "export_partial: nothing to export");
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(device_dst, h->d_state, sizeof(Running) * h->M, cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

int bioem_b200_import_partials(bioem_b200_handle h, const void *device_gathered, int nRanks)
{
  if (!h || !device_gathered || nRanks <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "import_partials: bad argument");
  CU(cudaSetDevice(h->device));
  init_state_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_state, h->M);
  merge_partials_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>((const Running *) device_gathered, nRanks, h->M, h->d_state);
  CU(cudaGetLastError());
  h->launches += 2;
  h->state_ready = true;
  h->argmax_exact = false;
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

// ---------------------------------------------------------------- multi-GPU merge inside the library
// Let kernels on device `reader` (the current device) dereference this library's buffers on device `owner`.  The
// buffers come from the owner's stream-ordered memory pool (cudaMallocAsync), whose allocations are NOT covered by
// cudaDeviceEnablePeerAccess: the pool itself has to grant the reader access (cudaMemPoolSetAccess).
static bool enable_peer_read(int reader, int owner)
{
  if (reader == owner)
    return true;
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, reader, owner) != cudaSuccess || !can)
  {
    cudaGetLastError();
    return false;
  }
  const cudaError_t e = cudaDeviceEnablePeerAccess(owner, 0);
  if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
  {
    cudaGetLastError();
    return false;
  }
  cudaGetLastError();
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, owner) != cudaSuccess)
  {
    cudaGetLastError();
    return false;
  }
  cudaMemAccessDesc desc;
  memset(&desc, 0, sizeof(desc));
  desc.location.type = cudaMemLocationTypeDevice;
  desc.location.id = reader;
  desc.flags = cudaMemAccessFlagsProtReadWrite;
  if (cudaMemPoolSetAccess(pool, &desc, 1) != cudaSuccess)
  {
    cudaGetLastError();
    return false;
  }
  return true;
}

int bioem_b200_merge_peers(bioem_b200_handle *hs, int n)
{
  if (!hs || n <= 0 || n > 16)
    return fail(BIOEM_B200_ERR_INVALID, "merge_peers: 1..16 handles expected");
  for (int r = 0; r < n; r++)
    if (!hs[r] || !hs[r]->state_ready || hs[r]->M != hs[0]->M)
      return fail(BIOEM_B200_ERR_STATE, "merge_peers: every handle must have run over the same particles");
  bioem_b200_context *d = hs[0];
  // all blocks must be complete before GPU 0 reads them
  for (int r = 1; r < n; r++)
  {
    CU(cudaSetDevice(hs[r]->device));
    CU(cudaStreamSynchronize(hs[r]->stream));
  }
  CU(cudaSetDevice(d->device));
  PeerParts parts;
  parts.n = n;
  std::vector<DevTmp *> staged;
  int rc = BIOEM_B200_OK;
  for (int r = 0; r < n && rc == BIOEM_B200_OK; r++)
  {
    parts.p[r] = hs[r]->d_state;
    if (hs[r]->device == d->device)
      continue;
    const bool can = enable_peer_read(d->device, hs[r]->device);
    if (!can)
    {
      // no peer mapping (PCIe box without P2P): stage the block with a peer copy instead
      DevTmp *t = new DevTmp(d);
      staged.push_back(t);
      rc = t->alloc(sizeof(Running) * (size_t) d->M);
      if (rc == BIOEM_B200_OK &&
          cudaMemcpyPeerAsync(t->p, d->device, hs[r]->d_state, hs[r]->device, sizeof(Running) * (size_t) d->M, d->stream) !=
              cudaSuccess)
        rc = fail(BIOEM_B200_ERR_CUDA, "merge_peers: cudaMemcpyPeerAsync failed");
      parts.p[r] = t->as<Running>();
    }
  }
  if (rc == BIOEM_B200_OK)
  {
    DevTmp merged(d);
    rc = merged.alloc(sizeof(Running) * (size_t) d->M);
    if (rc == BIOEM_B200_OK)
    {
      merge_peers_kernel<<<(d->M + 127) / 128, 128, 0, d->stream>>>(parts, d->M, merged.as<Running>());
      if (cudaGetLastError() != cudaSuccess ||
          cudaMemcpyAsync(d->d_state, merged.p, sizeof(Running) * (size_t) d->M, cudaMemcpyDeviceToDevice, d->stream) != cudaSuccess ||
          cudaStreamSynchronize(d->stream) != cudaSuccess)
        rc = fail(BIOEM_B200_ERR_CUDA, std::string("merge_peers: ") + cudaGetErrorString(cudaGetLastError()));
      d->launches += 1;
      d->argmax_exact = false;
    }
  }
  for (DevTmp *t : staged)
    delete t;
  return rc;
}

int bioem_b200_merge_top_angles_peers(bioem_b200_handle *hs, const int *oBegin, const int *oEnd, int n, int K,
                                      bioem_b200_top_angle *out)
{
  if (!hs || !oBegin || !oEnd || !out || n <= 0 || n > 16 || K <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "merge_top_angles_peers: bad argument");
  for (int r = 0; r < n; r++)
    if (!hs[r] || !hs[r]->state_ready || !hs[r]->cfg.writeAngles || !hs[r]->d_angtab || hs[r]->M != hs[0]->M ||
        oBegin[r] < 0 || oEnd[r] > hs[r]->O || oBegin[r] > oEnd[r] || (r > 0 && oBegin[r] < oEnd[r - 1]))
      return fail(BIOEM_B200_ERR_STATE, "merge_top_angles_peers: handles must hold ascending orientation blocks with writeAngles");
  bioem_b200_context *d = hs[0];
  const size_t rows = (size_t) d->M * K;
  // every GPU selects the K best orientations of its block where its angle table lies
  std::vector<DevTmp *> bufs;
  PeerLists lists;
  lists.n = n;
  int rc = BIOEM_B200_OK;
  for (int r = 0; r < n && rc == BIOEM_B200_OK; r++)
  {
    bioem_b200_context *h = hs[r];
    if (cudaSetDevice(h->device) != cudaSuccess)
      rc = fail(BIOEM_B200_ERR_CUDA, "merge_top_angles_peers: cudaSetDevice failed");
    DevTmp *key = new DevTmp(h), *top = new DevTmp(h);
    bufs.push_back(key);
    bufs.push_back(top);
    if (rc == BIOEM_B200_OK)
      rc = key->alloc(rows * sizeof(double));
    if (rc == BIOEM_B200_OK)
      rc = top->alloc(rows * sizeof(TopAngleOut));
    if (rc != BIOEM_B200_OK)
      break;
    top_angles_kernel<<<(h->M + 63) / 64, 64, 0, h->stream>>>(h->d_angtab, h->M, oBegin[r], oEnd[r], K, key->as<double>(),
                                                             top->as<TopAngleOut>());
    h->launches++;
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(h->stream) != cudaSuccess)
      rc = fail(BIOEM_B200_ERR_CUDA, "merge_top_angles_peers: selection kernel failed");
    lists.p[r] = top->as<TopAngleOut>();
  }
  if (rc == BIOEM_B200_OK && cudaSetDevice(d->device) != cudaSuccess)
    rc = fail(BIOEM_B200_ERR_CUDA, "merge_top_angles_peers: cudaSetDevice failed");
  for (int r = 1; r < n && rc == BIOEM_B200_OK; r++)
  {
    if (hs[r]->device == d->device)
      continue;
    const bool can = enable_peer_read(d->device, hs[r]->device);
    if (!can)
    {
      DevTmp *t = new DevTmp(d);
      bufs.push_back(t);
      rc = t->alloc(rows * sizeof(TopAngleOut));
      if (rc == BIOEM_B200_OK && cudaMemcpyPeerAsync(t->p, d->device, lists.p[r], hs[r]->device, rows * sizeof(TopAngleOut),
                                                     d->stream) != cudaSuccess)
        rc = fail(BIOEM_B200_ERR_CUDA, "merge_top_angles_peers: cudaMemcpyPeerAsync failed");
      lists.p[r] = t->as<TopAngleOut>();
    }
  }
  if (rc == BIOEM_B200_OK)
  {
    DevTmp key(d), top(d);
    rc = key.alloc(rows * sizeof(double));
    if (rc == BIOEM_B200_OK)
      rc = top.alloc(rows * sizeof(TopAngleOut));
    if (rc == BIOEM_B200_OK)
    {
      merge_top_lists_kernel<<<(d->M + 63) / 64, 64, 0, d->stream>>>(lists, d->M, K, key.as<double>(), top.as<TopAngleOut>());
      d->launches++;
      if (cudaGetLastError() != cudaSuccess ||
          cudaMemcpyAsync(out, top.p, rows * sizeof(TopAngleOut), cudaMemcpyDeviceToHost, d->stream) != cudaSuccess ||
          cudaStreamSynchronize(d->stream) != cudaSuccess)
        rc = fail(BIOEM_B200_ERR_CUDA, std::string("merge_top_angles_peers: ") + cudaGetErrorString(cudaGetLastError()));
    }
  }
  for (DevTmp *t : bufs)
  {
    cudaSetDevice(t->h->device);
    delete t;
  }
  cudaSetDevice(d->device);
  return rc;
}

int bioem_b200_nccl_unique_id(void *id128)
{
  if (!id128)
    return fail(BIOEM_B200_ERR_INVALID, "nccl_unique_id: null argument");
  NcclApi *a = nccl_api();
  if (!a)
    return fail(BIOEM_B200_ERR_STATE, "NCCL (libnccl.so.2) cannot be loaded");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  NC(a->GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return BIOEM_B200_OK;
}

int bioem_b200_nccl_init(bioem_b200_handle h, int nRanks, int rank, const void *id128)
{
  if (!h || !id128 || nRanks <= 0 || rank < 0 || rank >= nRanks)
    return fail(BIOEM_B200_ERR_INVALID, "nccl_init: bad argument");
  NcclApi *a = nccl_api();
  if (!a)
    return fail(BIOEM_B200_ERR_STATE, "NCCL (libnccl.so.2) cannot be loaded");
  CU(cudaSetDevice(h->device));
  nccl_release(h);
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  NC(a->CommInitRank(&comm, nRanks, id, rank));
  h->nccl_comm = comm;
  h->nccl_owned = true;
  h->nccl_ranks = nRanks;
  h->nccl_rank = rank;
  return BIOEM_B200_OK;
}

int bioem_b200_nccl_attach(bioem_b200_handle h, void *ncclComm)
{
  if (!h || !ncclComm)
    return fail(BIOEM_B200_ERR_INVALID, "nccl_attach: bad argument");
  NcclApi *a = nccl_api();
  if (!a)
    return fail(BIOEM_B200_ERR_STATE, "NCCL (libnccl.so.2) cannot be loaded");
  nccl_release(h);
  int n = 0, r = 0;
  NC(a->CommCount((ncclComm_t) ncclComm, &n));
  NC(a->CommUserRank((ncclComm_t) ncclComm, &r));
  h->nccl_comm = ncclComm;
  h->nccl_owned = false;
  h->nccl_ranks = n;
  h->nccl_rank = r;
  return BIOEM_B200_OK;
}

void *bioem_b200_nccl_comm(bioem_b200_handle h) { return h ? h->nccl_comm : nullptr; }

int bioem_b200_merge_nccl(bioem_b200_handle h)
{
  if (!h || !h->nccl_comm)
    return fail(BIOEM_B200_ERR_STATE, "merge_nccl: no communicator (bioem_b200_nccl_init / _attach first)");
  if (!h->state_ready)
    return fail(BIOEM_B200_ERR_STATE, "merge_nccl: nothing has been run");
  CU(cudaSetDevice(h->device));
  const size_t need = (size_t) h->M * h->nccl_ranks;
  if (h->gather_cap < need)
  {
    h->gather_cap = 0;
    RC(dev_realloc(h, h->d_gather, need));
    h->gather_cap = need;
  }
  // one all-gather of M x 48 bytes per rank, straight out of the running state, on the handle's own
  // stream; the fold follows in stream order (no host synchronisation in between)
  NC(nccl_api()->AllGather(h->d_state, h->d_gather, sizeof(Running) * (size_t) h->M, ncclInt8, (ncclComm_t) h->nccl_comm,
                           h->stream));
  init_state_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_state, h->M);
  merge_partials_kernel<<<(h->M + 127) / 128, 128, 0, h->stream>>>(h->d_gather, h->nccl_ranks, h->M, h->d_state);
  CU(cudaGetLastError());
  h->launches += 2;
  h->argmax_exact = false;
  return BIOEM_B200_OK;
}

int bioem_b200_top_angles_nccl(bioem_b200_handle h, int oBegin, int oEnd, int K, bioem_b200_top_angle *out)
{
  if (!h || !out || K <= 0 || oBegin < 0 || oEnd > h->O || oBegin > oEnd)
    return fail(BIOEM_B200_ERR_INVALID, "top_angles_nccl: bad argument");
  if (!h->nccl_comm)
    return fail(BIOEM_B200_ERR_STATE, "top_angles_nccl: no communicator (bioem_b200_nccl_init / _attach first)");
  if (!h->cfg.writeAngles || !h->d_angtab || !h->state_ready)
    return fail(BIOEM_B200_ERR_STATE, "top_angles_nccl: writeAngles == 0 or nothing has been run");
  CU(cudaSetDevice(h->device));
  const size_t rows = (size_t) h->M * K;
  const int R = h->nccl_ranks;
  if (R > 16)
    return fail(BIOEM_B200_ERR_INVALID, "top_angles_nccl: more than 16 ranks");
  DevTmp key(h), mine(h), all(h), top(h);
  RC(key.alloc(rows * sizeof(double)));
  RC(mine.alloc(rows * sizeof(TopAngleOut)));
  RC(all.alloc(rows * sizeof(TopAngleOut) * R));
  RC(top.alloc(rows * sizeof(TopAngleOut)));
  top_angles_kernel<<<(h->M + 63) / 64, 64, 0, h->stream>>>(h->d_angtab, h->M, oBegin, oEnd, K, key.as<double>(),
                                                           mine.as<TopAngleOut>());
  CU(cudaGetLastError());
  NC(nccl_api()->AllGather(mine.p, all.p, rows * sizeof(TopAngleOut), ncclInt8, (ncclComm_t) h->nccl_comm, h->stream));
  PeerLists lists;
  lists.n = R;
  for (int r = 0; r < R; r++)
    lists.p[r] = all.as<TopAngleOut>() + (size_t) r * rows;
  merge_top_lists_kernel<<<(h->M + 63) / 64, 64, 0, h->stream>>>(lists, h->M, K, key.as<double>(), top.as<TopAngleOut>());
  CU(cudaGetLastError());
  h->launches += 2;
  CU(cudaMemcpyAsync(out, top.p, rows * sizeof(TopAngleOut), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

void *bioem_b200_stream(bioem_b200_handle h) { return h ? (void *) h->stream : nullptr; }
void *bioem_b200_device_angles(bioem_b200_handle h) { return h ? (void *) h->d_angtab : nullptr; }

int bioem_b200_stats(bioem_b200_handle h, long long *launches, long long *likelihoods)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  if (launches)
    *launches = h->launches;
  if (likelihoods)
    *likelihoods = h->likelihoods;
  return BIOEM_B200_OK;
}

int bioem_b200_set_kernel_timing(bioem_b200_handle h, int on)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  h->time_kernels = on != 0;
  return BIOEM_B200_OK;
}

int bioem_b200_kernel_time(bioem_b200_handle h, double *ms, long long *n)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  double t = 0.0;
  for (auto &ev : h->lik_events)
  {
    float f = 0.f;
    CU(cudaEventElapsedTime(&f, ev.first, ev.second));
    t += f;
  }
  if (ms)
    *ms = t;
  if (n)
    *n = (long long) h->lik_events.size();
  for (auto &ev : h->lik_events)
  {
    h->event_pool.push_back(ev.first);
    h->event_pool.push_back(ev.second);
  }
  h->lik_events.clear();
  return BIOEM_B200_OK;
}

int bioem_b200_exact_argmax_info(bioem_b200_handle h, int *evaluated, int *corrected, int *disagreed)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  if (evaluated)
    *evaluated = h->refine_counts[0];
  if (corrected)
    *corrected = h->refine_counts[1];
  if (disagreed)
    *disagreed = h->refine_counts[2];
  return BIOEM_B200_OK;
}

int bioem_b200_out_of_frame(bioem_b200_handle h, int *perOrient, long long *total)
{
  if (!h)
    return fail(BIOEM_B200_ERR_INVALID, "null handle");
  if (!h->state_ready || !h->d_skipped)
    return fail(BIOEM_B200_ERR_STATE, "out_of_frame: nothing has been run");
  CU(cudaSetDevice(h->device));
  std::vector<int> tmp((size_t) h->O);
  CU(cudaMemcpyAsync(tmp.data(), h->d_skipped, sizeof(int) * (size_t) h->O, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  long long t = 0;
  for (int o = 0; o < h->O; o++)
    t += tmp[o];
  if (perOrient)
    memcpy(perOrient, tmp.data(), sizeof(int) * (size_t) h->O);
  if (total)
    *total = t;
  return BIOEM_B200_OK;
}

int bioem_b200_cached_product(bioem_b200_handle h)
{
  if (!h || h->OB <= 0)
    return -1;
  return h->zmode ? 1 : 0;
}

// ------------------------------------------------------------------ inspection
int bioem_b200_debug_projection(bioem_b200_handle h, int o, float *out)
{
  if (!h || !out || o < 0 || o >= h->O || h->A <= 0 || h->C <= 0 || h->M <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "debug_projection: bad argument / inputs missing");
  CU(cudaSetDevice(h->device));
  int rc = ensure_batch(h);
  if (rc)
    return rc;
  rc = run_front(h, o, 1);
  if (rc)
    return rc;
  const size_t n2 = (size_t) h->N * h->N;
  std::vector<double> td(h->nbands);
  CU(cudaMemcpyAsync(out, h->d_proj, sizeof(float) * n2, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(td.data(), h->d_tempden, sizeof(double) * h->nbands, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  double t = 0.0;
  for (double v : td)
    t += v;
  const float ratio = h->NormDen / (float) t;
  for (size_t i = 0; i < n2; i++)
    out[i] *= ratio;
  return BIOEM_B200_OK;
}

int bioem_b200_debug_convolved(bioem_b200_handle h, int o, int c, float *conv_out, float *sumC, float *sumsqC)
{
  if (!h || o < 0 || o >= h->O || c < 0 || c >= h->C || h->A <= 0 || h->M <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "debug_convolved: bad argument / inputs missing");
  CU(cudaSetDevice(h->device));
  int rc = ensure_batch(h);
  if (rc)
    return rc;
  // (a grouped table: only row c is convolved, through the selection path, into slot 0)
  DevTmp t_sel(h);
  if (h->grouped)
  {
    const int4 one = make_int4(0, 0, c, 0);
    RC(t_sel.alloc(sizeof(int4)));
    CU(cudaMemcpyAsync(t_sel.p, &one, sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    rc = run_front(h, o, 1, nullptr, t_sel.as<int4>(), 1, true);
    c = 0;
  }
  else
    rc = run_front(h, o, 1, nullptr, nullptr, 0, true);
  if (rc)
    return rc;
  const size_t stdsz = (size_t) h->N * (h->N / 2 + 1);
  if (conv_out)
  {
    DevTmp tmp(h);
    RC(tmp.alloc(sizeof(float2) * stdsz));
    CU(do_unpack(h->N, h->d_conv + (size_t) c * h->map4, tmp.as<float2>(), 1, h->stream));
    CU(cudaMemcpyAsync(conv_out, tmp.p, sizeof(float2) * stdsz, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  ConvParam cp;
  CU(cudaMemcpyAsync(&cp, h->d_cpar + c, sizeof(cp), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (sumC)
    *sumC = cp.sumC;
  if (sumsqC)
    *sumsqC = cp.sumsqC;
  return BIOEM_B200_OK;
}

int bioem_b200_debug_correlation(bioem_b200_handle h, int o, int c, int m, float *values, int *nvalues)
{
  if (!h || !values || o < 0 || o >= h->O || c < 0 || c >= h->C || m < 0 || m >= h->M || h->A <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "debug_correlation: bad argument / inputs missing");
  CU(cudaSetDevice(h->device));
  int rc = ensure_batch(h);
  if (rc)
    return rc;
  rc = run_front(h, o, 1);
  if (rc)
    return rc;
  const size_t nv = (size_t) h->nw * h->nw;
  if (h->generic)
  {
    DevTmp t_val(h);
    RC(t_val.alloc(sizeof(float) * nv * h->C));
    RC(gen_corr_launch(h, h->d_refs + (size_t) m * h->map4, 1, h->C, t_val.as<float>()));
    CU(cudaMemcpyAsync(values, t_val.as<float>() + (size_t) c * nv, sizeof(float) * nv, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (nvalues)
      *nvalues = (int) nv;
    return BIOEM_B200_OK;
  }
  DevTmp t_dbg(h), t_part(h);
  RC(t_dbg.alloc(sizeof(float) * nv * h->C));
  RC(t_part.alloc(sizeof(Running)));
  float *d_dbg = t_dbg.as<float>();
  Running *d_part = t_part.as<Running>();
  LikParams lp;
  fill_lik_params(h, lp, o, 1);
  lp.refs = h->d_refs + (size_t) m * h->map4;
  lp.sumRef = h->d_sumRef + m;
  lp.sumsqRef = h->d_sumsqRef + m;
  lp.partials = d_part;
  lp.angles = nullptr;
  lp.dbg_values = d_dbg;
  lp.M = 1;
  lp.OG = 1;
  lp.C = h->C; // every row of the table (a grouped one too)
  lp.group = lp.perm = nullptr;
  CU(do_lik(h->N, lp, 1, h->cfg.maxDisplaceCenter, h->stream));
  CU(cudaMemcpyAsync(values, d_dbg + (size_t) c * nv, sizeof(float) * nv, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (nvalues)
    *nvalues = (int) nv;
  return BIOEM_B200_OK;
}

int bioem_b200_debug_run_values(bioem_b200_handle h, int oBegin, int oEnd, float *values_out)
{
  if (!values_out)
    return fail(BIOEM_B200_ERR_INVALID, "debug_run_values: null output");
  return run_range(h, oBegin, oEnd, values_out);
}

int bioem_b200_debug_particle(bioem_b200_handle h, int m, float *fft_out, float *sum, float *sumsq)
{
  if (!h || m < 0 || m >= h->M)
    return fail(BIOEM_B200_ERR_INVALID, "debug_particle: bad argument");
  CU(cudaSetDevice(h->device));
  const size_t stdsz = (size_t) h->N * (h->N / 2 + 1);
  if (fft_out)
  {
    DevTmp tmp(h);
    RC(tmp.alloc(sizeof(float2) * stdsz));
    CU(do_unpack(h->N, h->d_refs + (size_t) m * h->map4, tmp.as<float2>(), 1, h->stream));
    CU(cudaMemcpyAsync(fft_out, tmp.p, sizeof(float2) * stdsz, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  if (sum)
    CU(cudaMemcpyAsync(sum, h->d_sumRef + m, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (sumsq)
    CU(cudaMemcpyAsync(sumsq, h->d_sumsqRef + m, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return BIOEM_B200_OK;
}

// host-side merge of per-rank results (same rule as merge_partials_kernel: strict '<'
// in rank order keeps the lowest rank on ties)
int bioem_b200_merge_host(const bioem_b200_prob_map *parts, int nRanks, int nMaps, bioem_b200_prob_map *out)
{
  if (!parts || !out || nRanks <= 0 || nMaps <= 0)
    return fail(BIOEM_B200_ERR_INVALID, "merge_host: bad argument");
  for (int m = 0; m < nMaps; m++)
  {
    bioem_b200_prob_map s = parts[m];
    for (int r = 1; r < nRanks; r++)
    {
      const bioem_b200_prob_map &p = parts[(size_t) r * nMaps + m];
      if (s.Constoadd < p.Constoadd)
      {
        const double T = s.Total * exp(s.Constoadd - p.Constoadd) + p.Total;
        s = p;
        s.Total = T;
      }
      else
        s.Total += p.Total * exp(p.Constoadd - s.Constoadd);
    }
    out[m] = s;
  }
  return BIOEM_B200_OK;
}

} // extern "C"
