/* bioem_b200 — C ABI of the B200-native BioEM likelihood path.
 *
 * This is the drop-in boundary for the reference's per-orientation likelihood
 * pipeline.  In the reference the seam is the C++ virtual interface of class bioem
 * (reference include/bioem.h:52-59,76-79: compareRefMaps / deviceInit / deviceStartRun
 * / deviceFinishRun / malloc_device_host) behind the factory bioem_cuda_create()
 * (reference include/bioem_cuda.h:20).  Because this library also moves projection
 * and CTF convolution onto the GPU, the seam sits one level higher: the host hands
 * over the inputs once and then asks for a RANGE OF ORIENTATIONS to be evaluated
 * against all particle images; results come back in the reference's own result
 * structs (bioem_Probability_map / bioem_Probability_angle).
 *
 * Conventions: plain C types only; every function returns 0 on success and a
 * non-zero code on failure, with a message available from bioem_b200_last_error()
 * (the reference itself prints and exit(1)s, defs.h:18-26 — the host binary keeps
 * doing that on a non-zero return).  The library copies all inputs at upload time;
 * the caller keeps ownership of every pointer it passes.  A handle is bound to one
 * CUDA device and must be driven by one host thread at a time; handles are
 * independent.  There is no CPU fallback: without a usable CUDA device every
 * device entry point fails.
 */
#ifndef BIOEM_B200_H
#define BIOEM_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIOEM_B200_OK 0
#define BIOEM_B200_ERR_INVALID 1 /* bad argument / unsupported size   */
#define BIOEM_B200_ERR_CUDA 2    /* CUDA runtime failure              */
#define BIOEM_B200_ERR_STATE 3   /* call order violated               */

typedef struct bioem_b200_context *bioem_b200_handle;

/* Replaces bioem_param_device (reference include/param.h:26-47) plus the four host
 * parameters createProjection reads (pixelSize, shiftX, shiftY, doquater;
 * reference bioem.cpp:1627,1715-1750). */
typedef struct bioem_b200_config
{
  int NumberPixels;      /* N; see bioem_b200_supported_size() for the edges with a fused FFT kernel */
  int maxDisplaceCenter; /* DISPLACE_CENTER first value  */
  int GridSpaceCenter;   /* DISPLACE_CENTER second value (need not divide the first: the window is the one
                            the reference's Algo 1 enumerates, bioem_algorithm.h:156-197) */
  int writeAngles;       /* WRITE_PROB_ANGLES (0 = off)  */
  int tousepsf;          /* USE_PSF                       */
  int doquater;          /* orientations are quaternions  */
  int shiftX, shiftY;    /* SHIFT_X / SHIFT_Y             */
  float pixelSize;
  float Ntotpi; /* (float)(N*N), reference param.cpp:1612 */
  float volu;   /* reference param.cpp:1600-1607 (only used by the caller's output stage) */
  float sigmaPriorbctf, sigmaPriordefo, Priordefcent, sigmaPrioramp, Priorampcent;
} bioem_b200_config;

/* == bioem_Probability_map (reference include/map.h:116-129), 40 bytes */
typedef struct bioem_b200_prob_map
{
  double Total;
  double Constoadd;
  int max_prob_cent_x, max_prob_cent_y, max_prob_orient, max_prob_conv;
  float max_prob_norm, max_prob_mu;
} bioem_b200_prob_map;

/* == bioem_Probability_angle (reference include/map.h:131-135), 16 bytes */
typedef struct bioem_b200_prob_angle
{
  double forAngles;
  double ConstAngle;
} bioem_b200_prob_angle;

/* One row of the per-particle list of most probable orientations (WRITE_PROB_ANGLES):
 * what the reference's heap of (log(forAngles) + ConstAngle, orientation) pairs keeps
 * (bioem.cpp:1254-1290), 24 bytes.  orient = -1: fewer orientations than rows. */
typedef struct bioem_b200_top_angle
{
  int orient;
  int pad;
  double forAngles;
  double ConstAngle;
} bioem_b200_top_angle;

/* == bioem_model::bioem_model_point (reference include/model.h:179-185), 24 bytes */
typedef struct bioem_b200_model_point
{
  float pos[3];
  float quat4; /* padding in the reference's myfloat3_t */
  float radius;
  float density;
} bioem_b200_model_point;

const char *bioem_b200_last_error(void);
int bioem_b200_version(void);
/* number of visible CUDA devices (0 when there is none; never an error) */
int bioem_b200_device_count(void);
/* 1 if N is an image edge the fused FFT kernel is instantiated for (every even edge 16..512 with prime factors 2/3/5/7
 * except 490).  Any other edge from 2 to 4096 -- odd ones included, which the reference accepts (param.cpp:140-152,
 * Parseval weights bioem.cpp:1893-1918) -- is accepted by create() as well and runs on the direct-DFT path: same
 * stages and results, plain O(N^2)-per-line transforms, many times slower. */
int bioem_b200_supported_size(int NumberPixels);

/* replaces bioem_cuda_create() + deviceInit() (reference bioem_cuda.cu:818-911) */
int bioem_b200_create(const bioem_b200_config *cfg, int device, bioem_b200_handle *out);
int bioem_b200_destroy(bioem_b200_handle h);

/* Model.points / Model.NormDen (reference model.h, bioem.cpp:1677-1810) */
int bioem_b200_upload_model(bioem_b200_handle h, const bioem_b200_model_point *points, int nPoints,
                            float NormDen);
/* param.angles: nOrient x myfloat3_t {pos[3], quat4} (reference param.h, defs.h:105-110) */
int bioem_b200_upload_orientations(bioem_b200_handle h, const float *angles4, int nOrient);
/* param.refCTF (nCtf x N x (N/2+1) interleaved complex, reference param.cpp:1359) and
 * param.CtfParam (nCtf x myfloat3_t {amp, phase, env, -}) */
int bioem_b200_upload_ctf(bioem_b200_handle h, const float *refCTF, const float *CtfParam4, int nCtf);
/* USE_PSF: the nCtf kernels given as real-space point-spread functions (nCtf x N x N); the library
 * takes their forward r2c transform, which the reference does on the host (param.cpp:1466-1535). */
int bioem_b200_upload_ctf_real(bioem_b200_handle h, const float *kernels, const float *CtfParam4, int nCtf);
/* Per-micrograph CTF groups: G tables of C rows each, group-major (G*C rows in the layouts of upload_ctf), and
 * Priordefcent[G], each group's defocus-prior centre in phase units (NULL: the config's Priordefcent for all).  Row
 * g*C + c's prior is that of upload_ctf with group g's centre.  After set_particle_groups, particle m integrates over
 * the C rows of its own group only, and every record names a row of the whole table (max_prob_conv = g*C + c), so
 * render_maps, download and the multi-GPU merges need no knowledge of groups.  A grouped run gives what G separate
 * ungrouped runs (group g's table, group g's particles) give: the same records and angle rows; Total bit for bit at
 * the same batch geometry (BIOEM_B200_OB / BIOEM_B200_OG), else up to the order of the partial merges.  The table
 * must be real (CTFs computed in Fourier space: cached-product mode, which a grouped table always runs in).  Refused
 * (BIOEM_B200_ERR_INVALID): a non-zero imaginary part, USE_PSF, G < 1, C < 1, and an edge without a fused kernel
 * (bioem_b200_supported_size(N) == 0); run() refuses BIOEM_B200_CACHED_PRODUCT=0 with it.  debug_run_values captures
 * [o][c][m] with c < C (each particle's own rows).  upload_ctf / upload_ctf_real replace a grouped table by an
 * ungrouped one and drop the particle groups; a new grouped table keeps them while they name groups it has. */
int bioem_b200_upload_ctf_groups(bioem_b200_handle h, const float *refCTF, const float *CtfParam4, const float *Priordefcent,
                                 int G, int C);
/* group[nMaps]: the CTF group of every particle, in [0, G).  nMaps must be the uploaded particle count; needs the
 * particles and a grouped table on the handle (else BIOEM_B200_ERR_STATE).  Invalidates the running state like an
 * upload; upload_particles* drop the list.  run() with a grouped table and no list returns BIOEM_B200_ERR_STATE. */
int bioem_b200_set_particle_groups(bioem_b200_handle h, const int *group, int nMaps);
/* RefMap.maps (nMaps x N x N, as read, BEFORE RefMap.precalculate): the library
 * computes sum_RefMap / sumsquare_RefMap / RefMapsFFT itself (replaces reference
 * map.cpp:557-630). */
int bioem_b200_upload_particles(bioem_b200_handle h, const float *maps, int nMaps);
/* the images of an MRC mode-2 stack exactly as they lie in the file (nMaps x nr x nc floats, column
 * index fastest): the library does what the reference's reader does on the host -- transposition
 * and, if normalise != 0 (no NO_MAP_NORM), zero mean / unit deviation with float accumulators in
 * file order (map.cpp:811-845) -- then the precalculation above. */
int bioem_b200_upload_particles_mrc(bioem_b200_handle h, const float *raw, int nMaps, int normalise);
/* alternative: the caller already ran RefMap.precalculate (RefMapsFFT nMaps x N x
 * (N/2+1) complex, sum_RefMap, sumsquare_RefMap) */
int bioem_b200_upload_particles_fft(bioem_b200_handle h, const float *RefMapsFFT, const float *sum_RefMap,
                                    const float *sumsquare_RefMap, int nMaps);

/* Every upload_* call invalidates the running per-image state: the next run() starts from a freshly
 * initialised state (as if reset() had been called), so results of different inputs never mix.  An
 * upload that fails leaves the handle without that input (run() then refuses with ERR_STATE). */

/* replaces the initialisation loop of bioem::run (reference bioem.cpp:681-699) */
int bioem_b200_reset(bioem_b200_handle h);
/* replaces the main loop of bioem::run (reference bioem.cpp:763-891) for orientations
 * [oBegin, oEnd): projection, convolution with every CTF, comparison with every
 * particle.  Asynchronous; results accumulate on the device across calls. */
int bioem_b200_run(bioem_b200_handle h, int oBegin, int oEnd);
int bioem_b200_synchronize(bioem_b200_handle h);
/* replaces deviceFinishRun's copy-back (reference bioem_cuda.cu:1017-1021):
 * maps_out[nMaps]; angles_out[nOrient*nMaps] in the reference's layout
 * angle*nMaps+map (map.h:147-150), may be NULL when writeAngles == 0. */
int bioem_b200_download(bioem_b200_handle h, bioem_b200_prob_map *maps_out, bioem_b200_prob_angle *angles_out);
/* download() first makes the displacement of every particle's arg-max record exact with respect to the
 * reference's rule "first maximum of the float-narrowed logpro in enumeration order" (bioem_algorithm.h:84-96,
 * quirks Q6/Q10): the winning (orientation, CTF) of each particle is evaluated once more and all of its
 * displacements are compared.  Counts of the last such pass: records re-evaluated, displacement indices that
 * changed, re-evaluations that did not reproduce the record's logpro (left untouched; never expected). */
int bioem_b200_exact_argmax_info(bioem_b200_handle h, int *evaluated, int *corrected, int *disagreed);
/* replaces the host heap of the WRITE_PROB_ANGLES writer (reference bioem.cpp:1254-1290):
 * the K most probable orientations of every particle among the orientations
 * [oBegin, oEnd), selected on the device; out[map*K + i], most probable first, in the order
 * the reference's heap is emptied (descending (logp, orientation); a full list only takes a
 * strictly greater logp).  Moves K*24 bytes per particle instead of nOrient*16. */
int bioem_b200_download_top_angles(bioem_b200_handle h, int oBegin, int oEnd, int K, bioem_b200_top_angle *out);

/* Multi-GPU (replaces the MPI reduction, reference bioem.cpp:909-1044).  Each GPU
 * runs a contiguous block of orientations; the per-image partial results are
 * exported as an opaque device blob of bioem_b200_partial_bytes(h) bytes, gathered
 * from all ranks by the caller (one all-gather, e.g. ncclAllGather), and imported in
 * rank order.  Ties between ranks resolve to the LOWEST rank (= lowest orientation
 * index, like a 1-process run). */
size_t bioem_b200_partial_bytes(bioem_b200_handle h);
int bioem_b200_export_partial(bioem_b200_handle h, void *device_dst);
int bioem_b200_import_partials(bioem_b200_handle h, const void *device_gathered, int nRanks);
/* same merge on host buffers */
int bioem_b200_merge_host(const bioem_b200_prob_map *parts, int nRanks, int nMaps, bioem_b200_prob_map *out);

/* The merge inside the library (replaces MPI_Allreduce / MPI_Reduce / MPI_Send of reference
 * bioem.cpp:909-977; lowest rank wins ties, see above).
 *
 * One process, one handle per GPU of the box (the bioEM_b200 binary): handles[0]'s GPU reads the other
 * GPUs' per-image states over NVLink peer memory inside the merge kernel (gather and fold are one
 * kernel; a peer copy is used where two GPUs have no peer mapping) and ends up holding the merged state;
 * download it from handles[0].  handles[] in ascending orientation-block order, n <= 16. */
int bioem_b200_merge_peers(bioem_b200_handle *handles, int n);
/* WRITE_PROB_ANGLES with several handles (replaces the angle reduction, reference bioem.cpp:979-1040, and the
 * writer's heap :1254-1290): every GPU selects the K most probable orientations of its block
 * [oBegin[r], oEnd[r]) per particle, handles[0]'s GPU merges the lists over peer memory; out[map*K + i]
 * as bioem_b200_download_top_angles. */
int bioem_b200_merge_top_angles_peers(bioem_b200_handle *handles, const int *oBegin, const int *oEnd, int n, int K,
                                      bioem_b200_top_angle *out);
/* One process per GPU (torchrun / MPI launchers): NCCL, bound at run time (libnccl.so.2).
 * Either let the library build the communicator -- rank 0 calls bioem_b200_nccl_unique_id(id) (128
 * bytes), the launcher's own plumbing broadcasts id, every rank calls bioem_b200_nccl_init -- or hand
 * over an existing ncclComm_t with bioem_b200_nccl_attach (not destroyed by the library). */
int bioem_b200_nccl_unique_id(void *id128);
int bioem_b200_nccl_init(bioem_b200_handle h, int nRanks, int rank, const void *id128);
int bioem_b200_nccl_attach(bioem_b200_handle h, void *ncclComm);
/* the handle's communicator (an ncclComm_t; NULL if none): lets further handles of the same process and device
 * share it through bioem_b200_nccl_attach instead of building their own (it stays owned by this handle) */
void *bioem_b200_nccl_comm(bioem_b200_handle h);
/* one ncclAllGather of the per-image partials (48 bytes per image and rank) on the handle's stream,
 * followed in stream order by the fold in rank order: every rank ends up with the merged state.
 * Collective: every rank of the communicator must call it.  Asynchronous like run(). */
int bioem_b200_merge_nccl(bioem_b200_handle h);
/* WRITE_PROB_ANGLES across ranks: device selection of this rank's block [oBegin, oEnd), one all-gather
 * of K x 24 bytes per image and rank, device merge; every rank receives out[map*K + i]. Collective. */
int bioem_b200_top_angles_nccl(bioem_b200_handle h, int oBegin, int oEnd, int K, bioem_b200_top_angle *out);
/* the stream all work of this handle is enqueued on (a cudaStream_t) */
void *bioem_b200_stream(bioem_b200_handle h);
/* device pointer to the [nOrient][nMaps] angle table (NULL when writeAngles == 0) */
void *bioem_b200_device_angles(bioem_b200_handle h);

/* statistics of the last run() calls since reset(): kernels launched, likelihoods */
int bioem_b200_stats(bioem_b200_handle h, long long *kernel_launches, long long *likelihoods);
/* Optional CUDA-event timing of the fused likelihood kernel (roofline accounting of bench.py / the
 * profiling tools).  Off by default: run() then records no events.  bioem_b200_kernel_time synchronises
 * the stream and returns the duration [ms] and number of the launches recorded since its previous call
 * (or since timing was switched on); it is not affected by reset(). */
int bioem_b200_set_kernel_timing(bioem_b200_handle h, int on);
int bioem_b200_kernel_time(bioem_b200_handle h, double *likelihood_ms, long long *likelihood_launches);
/* Model points that fell outside the image frame and were skipped (reference bioem.cpp:1724-1734,
 * 1756-1780 prints "point out of image size" once per projection): per orientation since reset()
 * (perOrient[nOrient], may be NULL) and in total. */
int bioem_b200_out_of_frame(bioem_b200_handle h, int *perOrient, long long *total);

/* Mode of the fused kernel for the inputs now on the handle: 1 = cached-product mode (every CTF kernel is real,
 * i.e. computed in Fourier space as param.cpp:1540-1570 does, and there are at least 4 of them: the product
 * projection * conj(particle) is formed once per orientation and multiplied by the real kernels), 0 = complex
 * convolved spectra (USE_PSF, few CTFs), -1 = not decided yet (decided by the first run() after the uploads).
 * The results of the two modes differ by FP32 rounding only (multiplication order).
 * BIOEM_B200_CACHED_PRODUCT=0/1 in the environment overrides the choice for real kernels. */
int bioem_b200_cached_product(bioem_b200_handle h);

/* The calculated image each record names: maps_out[i][N][N], in the layout of the images given to
 * upload_particles (RefMap.maps), so that particle - map is the residual.  Reads max_prob_orient, max_prob_conv,
 * max_prob_cent_x/y (as download() returns them), max_prob_norm and max_prob_mu:
 *     maps_out[i][x][y] = norm * R0[(x - cent_x) mod N][(y - cent_y) mod N] + mu
 * where R0 is the convolved projection c2r(P_o K_c) / N^2 (sum R0 = sumC; sum R0^2 is sumsquareC less the part of
 * the CTF table's non-Hermitian self-conjugate columns that no real image carries), so that render_maps(download())
 * gives every particle's best-fit map.  Needs model, orientations and CTF table, not
 * particles or a run.  Synchronous.  Leaves the running state untouched (download(), the angle table,
 * exact_argmax_info, out_of_frame and stats are what they would have been without the call).  Refuses an
 * orientation or CTF index out of range, |cent| >= N, n < 0 and null pointers when n > 0 (BIOEM_B200_ERR_INVALID);
 * missing uploads give BIOEM_B200_ERR_STATE. */
int bioem_b200_render_maps(bioem_b200_handle h, const bioem_b200_prob_map *records, int n, float *maps_out);

/* ---- inspection entry points (tests): intermediate products of one orientation ---- */
/* real-space projection (N*N, already scaled by NormDen/tempden) */
int bioem_b200_debug_projection(bioem_b200_handle h, int iOrient, float *proj_out);
/* convolved map in the reference's N x (N/2+1) interleaved complex layout + sumC, sumsquareC */
int bioem_b200_debug_convolved(bioem_b200_handle h, int iOrient, int iConv, float *conv_out, float *sumC,
                               float *sumsquareC);
/* correlation values lCC/N^2 over the displacement window of (iOrient, iConv, iMap),
 * in doRefMapFFT enumeration order (reference bioem_algorithm.h:156-197) */
int bioem_b200_debug_correlation(bioem_b200_handle h, int iOrient, int iConv, int iMap, float *values_out,
                                 int *nValues);
/* run(h, oBegin, oEnd) -- same batching, kernel mode and launch grid, the running state accumulates as there, so
 * download() afterwards is valid -- and every correlation value lCC/N^2 it computes, written to
 * values_out[(o - oBegin) * nCtf * nMaps + c * nMaps + m][nValues] in the order of debug_correlation.  Synchronous. */
int bioem_b200_debug_run_values(bioem_b200_handle h, int oBegin, int oEnd, float *values_out);
/* particle spectrum in the reference layout + its sums */
int bioem_b200_debug_particle(bioem_b200_handle h, int iMap, float *fft_out, float *sum, float *sumsq);

/* ---- host-side input preparation (pure CPU; mirrors the reference's one-off setup) ---- */
/* param.cpp:601-607 */
void bioem_b200_host_defocus_to_phase(float startDefocus, float endDefocus, float elecwavel, float *startPhase,
                                      float *endPhase, float *Priordefcent, float *sigmaPriordefo);
/* param.cpp:1336-1620 CalculateRefCTF (CTF mode and PSF mode); returns nCtf.  refCTF / CtfParam4 may
 * be NULL to query the count and the grid steps (grids[3] = amp, phase, envelope step). */
int bioem_b200_host_ctf_table(int N, float pixelSize, int usepsf, float startAmp, float endAmp, int nAmp,
                              float startPhase, float endPhase, int nPhase, float startEnv, float endEnv,
                              int nEnv, float *refCTF, float *CtfParam4, float *grids);
/* param.cpp:1336-1536 with USE_PSF: real-space point-spread functions (nCtf x N x N, unit sum) for
 * bioem_b200_upload_ctf_real; returns nCtf (kernels / CtfParam4 may be NULL to query), -3 if the
 * widest envelope does not fit the kernel length */
int bioem_b200_host_psf_kernels(int N, float pixelSize, float startAmp, float endAmp, int nAmp, float startPhase,
                                float endPhase, int nPhase, float startEnv, float endEnv, int nEnv, float *kernels,
                                float *CtfParam4, float *grids);
/* param.cpp:1600-1607 */
float bioem_b200_host_volu(float voluang, int GridSpaceCenter, float pixelSize, int maxDisplaceCenter,
                           int nAmp, float gridEnvelop, float gridCTF_phase, float sigmaPriorbctf,
                           float sigmaPriordefo, float sigmaPrioramp);
/* model.cpp:604-672 (centre of density) and NormDen; points modified in place; returns NormDen */
float bioem_b200_host_model_prepare(bioem_b200_model_point *points, int nPoints, int center);
/* map.cpp:830-845: the MRC reader's per-image normalisation (in place, N*N) */
void bioem_b200_host_normalise_map(float *img, int N);
/* bioem.cpp:1144-1149: final log posterior of one image */
double bioem_b200_host_final_logprob(const bioem_b200_config *cfg, double Total, double Constoadd);

#ifdef __cplusplus
}
#endif
#endif
