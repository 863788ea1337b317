// bioEM_b200 — host front end of the B200 likelihood path.
//
// Keeps the reference's command line (bioem.cpp:193-224), input parameter file
// (param.cpp:121-627), orientation sources (param.cpp:988-1334), model / particle file formats
// (model.cpp, map.cpp, include/mrc.h) and text outputs (bioem.cpp:1046-1374); everything between
// reading the inputs and writing the outputs goes through the C ABI of libbioem_b200.so.
#pragma once
#include "../../../include/bioem_b200.h"
#include <string>
#include <vector>

namespace bhost
{

[[noreturn]] void fail(const char *fmt, ...); // the reference's myError: message, exit(1) (defs.h:18-26)
void warn(const char *fmt, ...);

struct Options // reference bioem.cpp:193-224
{
  std::string modelfile, particlesfile, inputfile, orientfile, outfile = "Output_Probabilities";
  bool readPDB = false, readModelMRC = false, readMRC = false, readMultMRC = false;
  bool dumpMaps = false, loadMapDump = false, dumpModel = false, loadModelDump = false;
  bool printCoordRead = false;
  int gpus = 0; // extension: number of GPUs of this box to use (0 = all visible)
  std::string bestmapsfile; // extension: --WriteBestMaps, every particle's best-fit calculated map (MRC stack)
  std::string defocusfile;  // extension: --DefocusPerParticle, one defocus [micro-m] per particle (CTF groups)
};

struct Params // reference bioem_param after readParameters + CalculateGridsParam + CalculateRefCTF
{
  int N = 0;
  float pixelSize = 0.f;
  int maxDisplaceCenter = 0, GridSpaceCenter = 0;
  int writeAngles = 0;
  bool usepsf = false, doquater = false, nocentermass = false, notnormmap = false, ignorePDB = false;
  bool yespriorAngles = false, writeCTF = false, notuniformangles = false;
  float elecwavel = 0.019866f;
  float priorMod = 1.f;
  int shiftX = 0, shiftY = 0;
  float sigmaPriorbctf = 100.f, sigmaPriordefo = 2.0f, Priordefcent = 3.0f, sigmaPrioramp = 0.5f, Priorampcent = 0.f;
  int angleGridPointsAlpha = 0, angleGridPointsBeta = 0, GridPointsQuatern = -1;
  float startAmp = 0, endAmp = 0, startPhase = 0, endPhase = 0, startEnv = 0, endEnv = 0;
  float startDef = 0, endDef = 0; // CTF_DEFOCUS [micro-m]
  int nAmp = 0, nPhase = 0, nEnv = 0;
  // derived
  std::vector<float> angles;   // nOrient x {pos[3], quat4}
  std::vector<float> angprior; // nOrient (PRIOR_ANGLES)
  float voluang = 0.f;
  std::vector<float> psfKernels; // USE_PSF: nCtf x N x N real-space kernels (refCTF stays empty)
  std::vector<float> refCTF;   // nCtf x N x (N/2+1) x 2
  std::vector<float> CtfParam; // nCtf x 4 {amp, phase, env, -} (CTF groups: nGroups x nCtf rows, group-major)
  int nCtf = 0;                // CTF rows every particle integrates over
  int nGroups = 0;             // --DefocusPerParticle: number of CTF groups (0 = one table for all particles)
  std::vector<int> group;      // nMaps: CTF group of every particle
  std::vector<float> groupDefcent; // nGroups: defocus-prior centre of every group [phase]
  float volu = 0.f;
  int nOrient() const { return (int) (angles.size() / 4); }
};

void parse_options(int argc, char **argv, Options &o);
void read_parameters(const std::string &file, Params &p);                  // param.cpp:64-627
void make_orientations(const std::string &orientfile, Params &p);          // param.cpp:988-1334
void make_ctf_table(Params &p);                                            // param.cpp:1336-1620 via the C ABI
// --DefocusPerParticle: one CTF table per distinct defocus of the file (groups in order of first appearance), each with
// CTF_DEFOCUS's width and count centred on that value and PRIOR_DEFOCUS_CENTER = that value; replaces the table
void make_ctf_groups(const std::string &file, int nMaps, Params &p);
void read_model(const Options &o, const Params &p, std::vector<bioem_b200_model_point> &pts, float &NormDen);
// maps: nMaps x N x N.  For MRC stacks (rawMRC = true) the images are left exactly as they lie in the
// file; the library transposes / normalises them on the device (bioem_b200_upload_particles_mrc).
void read_particles(const Options &o, const Params &p, std::vector<float> &maps, int &nMaps, bool &rawMRC);
// what the reference's MRC reader does to a raw stack, on the host (for --DumpMaps and the test hook)
void mrc_host_ingest(const Params &p, std::vector<float> &maps, int nMaps);
// maps: n x N x N (the layout of the particles handed to the library) -> MRC mode-2 stack that read_particles with
// --ReadMRC and NO_MAP_NORM reads back to the same arrays
void write_mrc_stack(const std::string &file, const float *maps, int N, int n);
// cand: WRITE_PROB_ANGLES candidates, nMaps x nCand rows in ascending orientation order (orient -1 = unused): the
// per-GPU lists of most probable orientations selected on the device (bioem_b200_download_top_angles)
void write_outputs(const Options &o, const Params &p, const bioem_b200_config &cfg,
                   const std::vector<bioem_b200_prob_map> &pm, const std::vector<bioem_b200_top_angle> &cand, int nCand,
                   int nMaps);

} // namespace bhost
