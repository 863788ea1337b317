// Command line, parameter file, orientation sources, model and particle readers of bioEM_b200.
// Behaviour (keywords, defaults, error conditions, file layouts) follows the reference files cited
// at each function; the code is this project's own.
#include "bioem_host.hpp"
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

namespace bhost
{

void fail(const char *fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "Error - ");
  vfprintf(stderr, fmt, ap);
  fprintf(stderr, "\n");
  va_end(ap);
  exit(1);
}
void warn(const char *fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "Warning - ");
  vfprintf(stderr, fmt, ap);
  fprintf(stderr, "\n");
  va_end(ap);
}

// --------------------------------------------------------------------------- command line
static void usage()
{
  printf("\nCommand line inputs:\n"
         "  --Modelfile arg        (Mandatory) Name of model file\n"
         "  --Particlesfile arg    (Mandatory) Name of particle-image file\n"
         "  --Inputfile arg        (Mandatory) Name of input parameter file\n"
         "  --ReadOrientation arg  (Optional) Read file name containing orientations\n"
         "  --ReadPDB              (Optional) If reading model file in PDB format\n"
         "  --ReadModelMRC         (Optional) If reading model file in MRC format\n"
         "  --ReadMRC              (Optional) If reading particle file in MRC format\n"
         "  --ReadMultipleMRC      (Optional) If reading multiple MRCs\n"
         "  --DumpMaps             (Optional) Dump maps after they were read from particle-image file\n"
         "  --LoadMapDump          (Optional) Read maps from dump option\n"
         "  --DumpModel            (Optional) Dump model after it was read from model file\n"
         "  --LoadModelDump        (Optional) Read model from dump option\n"
         "  --PrintCOORDREAD       (Optional) Print model coordinates\n"
         "  --OutputFile arg       (Optional) For changing the outputfile name\n"
         "  --Gpus arg             (Extension) number of GPUs of this box to use (default: all)\n"
         "  --WriteBestMaps arg    (Extension) write every particle's best-fit calculated map (orientation, CTF,\n"
         "                         displacement, normalisation and offset of its Maximizing Param line) to this\n"
         "                         file, one MRC mode-2 stack that --ReadMRC with NO_MAP_NORM reads back as the\n"
         "                         rendered images.  Not the reference's --PrintBestCalMap: its parameter keywords,\n"
         "                         BESTMAP text format and noise option are not reproduced\n"
         "  --DefocusPerParticle arg (Extension) file with one defocus [micro-m] per particle, in particle order:\n"
         "                         particles with equal values form one CTF group, whose defocus grid has\n"
         "                         CTF_DEFOCUS's width and count centred on the value, and whose PRIOR_DEFOCUS_CENTER\n"
         "                         is the value; every particle integrates over its own group's CTFs only\n"
         "  --help                 (Optional) Produce help message\n\n");
}

// reference bioem.cpp:170-380
void parse_options(int argc, char **argv, Options &o)
{
  if (argc < 2)
  {
    printf("Error - Need to specify all mandatory options\n");
    usage();
    exit(1);
  }
  for (int i = 1; i < argc; i++)
  {
    std::string a = argv[i];
    if (a.rfind("--", 0) != 0)
    {
      printf("Error - Non-option ARGV-elements: %s\n", a.c_str());
      usage();
      exit(1);
    }
    a = a.substr(2);
    std::string val;
    bool has_val = false;
    const size_t eq = a.find('=');
    if (eq != std::string::npos)
    {
      val = a.substr(eq + 1);
      a = a.substr(0, eq);
      has_val = true;
    }
    auto need = [&]() -> std::string {
      if (has_val)
        return val;
      if (i + 1 >= argc)
        fail("option --%s requires an argument", a.c_str());
      return argv[++i];
    };
    if (a == "Modelfile")
      o.modelfile = need();
    else if (a == "Particlesfile")
      o.particlesfile = need();
    else if (a == "Inputfile")
      o.inputfile = need();
    else if (a == "ReadOrientation")
      o.orientfile = need();
    else if (a == "OutputFile")
      o.outfile = need();
    else if (a == "Gpus")
      o.gpus = atoi(need().c_str());
    else if (a == "WriteBestMaps")
      o.bestmapsfile = need();
    else if (a == "DefocusPerParticle")
      o.defocusfile = need();
    else if (a == "ReadPDB")
      o.readPDB = true;
    else if (a == "ReadModelMRC")
      o.readModelMRC = true;
    else if (a == "ReadMRC")
      o.readMRC = true;
    else if (a == "ReadMultipleMRC")
      o.readMultMRC = true;
    else if (a == "DumpMaps")
      o.dumpMaps = true;
    else if (a == "LoadMapDump")
      o.loadMapDump = true;
    else if (a == "DumpModel")
      o.dumpModel = true;
    else if (a == "LoadModelDump")
      o.loadModelDump = true;
    else if (a == "PrintCOORDREAD")
      o.printCoordRead = true;
    else if (a == "help")
    {
      usage();
      exit(0);
    }
    else if (a == "PrintBestCalMap")
      fail("--PrintBestCalMap is not part of the likelihood path and is not provided by bioEM_b200");
    else
    {
      printf("Error - unknown option --%s\n", a.c_str());
      usage();
      exit(1);
    }
  }
  if (o.modelfile.empty() || o.particlesfile.empty() || o.inputfile.empty())
  {
    printf("Error - Need to specify all mandatory options\n");
    usage();
    exit(1);
  }
  if (o.readMultMRC && !o.readMRC)
    fail("For multiple MRCs command --ReadMRC is necessary too");
}

// --------------------------------------------------------------------------- parameter file
// reference param.cpp:64-627: one keyword per line, tokens separated by single spaces, '#' in
// column 0 starts a comment.
void read_parameters(const std::string &file, Params &p)
{
  std::ifstream in(file.c_str());
  if (!in.good())
    fail("Opening file: %s", file.c_str());
  bool yPix = false, yNum = false, yAl = false, yBe = false, yMDC = false, yB = false, yDef = false, yAmp = false;
  bool yPenv = false, yPpha = false, yQgrid = false;
  float startB = 0, endB = 0, startDef = 0, endDef = 0;
  std::string line;
  printf("\n +++++++++++++++++++++++++++++++++++++++++ \n\n   READING BioEM PARAMETERS             \n\n"
         " +++++++++++++++++++++++++++++++++++++++++ \n");
  while (std::getline(in, line))
  {
    if (line.size() > 511)
      line.resize(511);
    if (line.empty() || line[0] == '#')
      continue;
    std::vector<std::string> tok;
    {
      // strtok(line, " "): runs of blanks separate tokens
      size_t pos = 0;
      while (pos < line.size())
      {
        while (pos < line.size() && line[pos] == ' ')
          pos++;
        size_t e = pos;
        while (e < line.size() && line[e] != ' ')
          e++;
        if (e > pos)
          tok.push_back(line.substr(pos, e - pos));
        pos = e;
      }
    }
    if (tok.empty())
      continue;
    const std::string &k = tok[0];
    auto f = [&](size_t i) -> float {
      if (i >= tok.size())
        fail("keyword %s: missing value", k.c_str());
      return (float) atof(tok[i].c_str());
    };
    auto n = [&](size_t i) -> int {
      if (i >= tok.size())
        fail("keyword %s: missing value", k.c_str());
      return atoi(tok[i].c_str());
    };
    auto grid3 = [&](float &a, float &b, int &cnt, const char *what) {
      a = f(1);
      if (a < 0)
        fail("Negative start %s", what);
      b = f(2);
      if (b < 0)
        fail("Negative end %s", what);
      cnt = n(3);
      if (cnt < 0)
        fail("Negative number of grid points %s", what);
      if (a > b)
        fail("Grid ill defined end > start");
    };
    if (k == "PIXEL_SIZE")
    {
      p.pixelSize = f(1);
      if (p.pixelSize < 0)
        fail("Negative pixel size");
      std::cout << "Pixel Size " << p.pixelSize << "\n";
      yPix = true;
    }
    else if (k == "NUMBER_PIXELS")
    {
      p.N = n(1);
      if (p.N < 0)
        fail("Negative Number of Pixels");
      std::cout << "Number of Pixels " << p.N << "\n";
      yNum = true;
    }
    else if (k == "GRIDPOINTS_ALPHA")
    {
      p.angleGridPointsAlpha = n(1);
      if (p.angleGridPointsAlpha < 0)
        fail("Negative GRIDPOINTS_ALPHA");
      std::cout << "Grid points alpha " << p.angleGridPointsAlpha << "\n";
      yAl = true;
    }
    else if (k == "GRIDPOINTS_BETA")
    {
      p.angleGridPointsBeta = n(1);
      if (p.angleGridPointsBeta < 0)
        fail("Negative GRIDPOINTS_BETA");
      std::cout << "Grid points in Cosine ( beta ) " << p.angleGridPointsBeta << "\n";
      yBe = true;
    }
    else if (k == "USE_QUATERNIONS")
    {
      std::cout << "Orientations with Quaternions. \n";
      p.doquater = true;
    }
    else if (k == "GRIDPOINTS_QUATERNION")
    {
      if (p.notuniformangles)
        fail("Inconsistent input: grid or list with quaternions?");
      p.GridPointsQuatern = n(1);
      yQgrid = true;
      p.doquater = true;
    }
    else if (k == "CTF_B_ENV")
    {
      grid3(startB, endB, p.nEnv, "B Env.");
      std::cout << "Grid CTF B-ENV: " << startB << " " << endB << " " << p.nEnv << "\n";
      yB = true;
    }
    else if (k == "CTF_DEFOCUS")
    {
      grid3(startDef, endDef, p.nPhase, "defocus");
      std::cout << "Grid CTF Defocus: " << startDef << " " << endDef << " " << p.nPhase << "\n";
      if (endDef > 8.)
        fail("Defocus beyond 8micro-m range is not allowed");
      yDef = true;
    }
    else if (k == "CTF_AMPLITUDE" || k == "PSF_AMPLITUDE")
    {
      grid3(p.startAmp, p.endAmp, p.nAmp, "amplitude");
      std::cout << "Grid Amplitude: " << p.startAmp << " " << p.endAmp << " " << p.nAmp << "\n";
      yAmp = true;
    }
    else if (k == "ELECTRON_WAVELENGTH")
    {
      p.elecwavel = f(1);
      if (p.elecwavel < 0.0150)
        fail("Wrong electron wave length %lf. Has to be in Angstrom (A)", (double) p.elecwavel);
    }
    else if (k == "USE_PSF")
    {
      p.usepsf = true;
      std::cout << "Important: Using Point Spread Function. Thus, all parameters are in Real Space. \n";
    }
    else if (k == "PSF_ENVELOPE")
    {
      grid3(p.startEnv, p.endEnv, p.nEnv, "PSF Env.");
      std::cout << "Grid PSF Envelope: " << p.startEnv << " " << p.endEnv << " " << p.nEnv << "\n";
      yPenv = true;
    }
    else if (k == "PSF_PHASE")
    {
      grid3(p.startPhase, p.endPhase, p.nPhase, "PSF phase");
      std::cout << "Grid PSF phase: " << p.startPhase << " " << p.endPhase << " " << p.nPhase << "\n";
      yPpha = true;
    }
    else if (k == "DISPLACE_CENTER")
    {
      p.maxDisplaceCenter = n(1);
      if (p.maxDisplaceCenter < 0)
        fail("Negative MAX_D_CENTER");
      std::cout << "Maximum displacement Center " << p.maxDisplaceCenter << "\n";
      p.GridSpaceCenter = n(2);
      if (p.GridSpaceCenter < 0)
        fail("Negative PIXEL_GRID_CENTER");
      std::cout << "Grid space displacement center " << p.GridSpaceCenter << "\n";
      yMDC = true;
    }
    else if (k == "WRITE_PROB_ANGLES")
    {
      p.writeAngles = n(1);
      if (p.writeAngles < 0)
        fail("Negative WRITE_PROB_ANGLES");
      std::cout << "Writing " << p.writeAngles << " Probabilies of each angle \n";
    }
    else if (k == "IGNORE_PDB")
      p.ignorePDB = true;
    else if (k == "NO_PROJECT_RADIUS")
    {
      // accepted and ignored: the reference sets a flag that nothing reads (param.cpp:425-430)
    }
    else if (k == "WRITE_CTF_PARAM")
      p.writeCTF = true;
    else if (k == "NO_CENTEROFMASS")
      p.nocentermass = true;
    else if (k == "PRINT_ROTATED_MODELS")
      warn("PRINT_ROTATED_MODELS is a debugging aid of the reference and is ignored");
    else if (k == "NO_MAP_NORM")
      p.notnormmap = true;
    else if (k == "PRIOR_MODEL")
      p.priorMod = f(1);
    else if (k == "PRIOR_ANGLES")
      p.yespriorAngles = true;
    else if (k == "SHIFT_X")
      p.shiftX = n(1);
    else if (k == "SHIFT_Y")
      p.shiftY = n(1);
    else if (k == "SIGMA_PRIOR_B_CTF")
      p.sigmaPriorbctf = f(1);
    else if (k == "SIGMA_PRIOR_DEFOCUS")
      p.sigmaPriordefo = f(1);
    else if (k == "PRIOR_DEFOCUS_CENTER")
      p.Priordefcent = f(1);
    else if (k == "SIGMA_PRIOR_AMP_CTF")
      p.sigmaPrioramp = f(1);
    else if (k == "PRIOR_AMP_CTF_CENTER")
      p.Priorampcent = f(1);
    // unknown keywords are skipped silently, like the reference
  }
  std::cout << "To verify input of Priors:\nSigma Prior B-Env: " << p.sigmaPriorbctf << "\nSigma Prior Defocus: " << p.sigmaPriordefo
            << "\nCenter Prior Defocus: " << p.Priordefcent << "\n";
  if (!yPix)
    fail("Input missing: please provide PIXEL_SIZE");
  if (!yNum)
    fail("Input missing: please provide NUMBER_PIXELS");
  if (!p.notuniformangles)
  {
    if (!p.doquater)
    {
      if (!yAl)
        fail("Input missing: please provide GRIDPOINTS_ALPHA");
      if (!yBe)
        fail("Input missing: please provide GRIDPOINTS_BETA");
    }
    else if (!yQgrid)
      fail("Input missing: please provide GRIDPOINTS_QUATERNION");
  }
  if (!yMDC)
    fail("Input missing: please provide grid displacement CENTER");
  if (p.usepsf)
  {
    if (!yPpha)
      fail("Input missing: please provide grid PSF PHASE");
    if (!yPenv)
      fail("Input missing: please provide grid PSF ENVELOPE");
    if (!yAmp)
      fail("Input missing: please provide grid PSF AMPLITUD");
  }
  else
  {
    if (!yB)
      fail("Input missing: please provide grid CTF B Env.");
    if (!yDef)
      fail("Input missing: please provide grid CTF defocus");
    if (!yAmp)
      fail("Input missing: please provide grid CTF amplitude");
    p.startDef = startDef;
    p.endDef = endDef;
    // defocus [micro-m] -> phase, prior centre and width scaled alike (param.cpp:601-607)
    bioem_b200_host_defocus_to_phase(startDef, endDef, p.elecwavel, &p.startPhase, &p.endPhase, &p.Priordefcent,
                                     &p.sigmaPriordefo);
    p.startEnv = startB;
    p.endEnv = endB;
  }
  if (p.writeCTF && !p.usepsf)
    fail("Writing CTF is only valid when integrating over the PSF");
  // (a spacing that does not divide the maximum displacement is fine: the library enumerates the window of
  // the reference's Algo 1, bioem_algorithm.h:156-197; the reference itself divides by the spacing,
  // param.cpp:1614, so 0 is not a usable value there either)
  if (p.GridSpaceCenter < 1)
    fail("DISPLACE_CENTER: the grid spacing must be at least 1");
}

// --------------------------------------------------------------------------- orientations
// fixed 12-character columns (param.cpp:1051-1133,1213-1327): column k is the text at [12k, 12k+12)
static bool fixed_col(const std::string &line, int k, float *out)
{
  char buf[13] = {0};
  if ((size_t) (12 * k) < line.size())
    strncpy(buf, line.c_str() + 12 * k, 12);
  return sscanf(buf, "%f", out) == 1;
}

void make_orientations(const std::string &orientfile, Params &p)
{
  p.angles.clear();
  p.angprior.clear();
  if (!p.notuniformangles)
  {
    if (p.yespriorAngles)
      fail("This option is not valid with prior for orientations. Please provide separate file with "
           "orientations and priors");
    if (!p.doquater)
    {
      // uniform grid in (alpha, cos beta, gamma), param.cpp:1009-1048
      std::cout << "Calculating Grids in Euler Angles\n";
      const float grid_alpha = 2.f * M_PI / (float) p.angleGridPointsAlpha;
      const float cos_grid_beta = 2.f / (float) p.angleGridPointsBeta;
      for (int ia = 0; ia < p.angleGridPointsAlpha; ia++)
        for (int ib = 0; ib < p.angleGridPointsBeta; ib++)
          for (int ig = 0; ig < p.angleGridPointsAlpha; ig++)
          {
            p.angles.push_back((float) ia * grid_alpha - M_PI + grid_alpha * 0.5f);
            p.angles.push_back(acos((float) ib * cos_grid_beta - 1 + cos_grid_beta * 0.5f));
            p.angles.push_back((float) ig * grid_alpha - M_PI + grid_alpha * 0.5f);
            p.angles.push_back(0.f);
          }
      p.voluang = grid_alpha * grid_alpha * cos_grid_beta / (2.f * M_PI) / (2.f * M_PI) / 2.f * p.priorMod;
    }
    else
    {
      // quaternion grid: cell centres of a cube inside the unit ball, both signs of q4 (param.cpp:1141-1210)
      std::cout << "Calculating Grids in Quaterions\n ";
      if (p.GridPointsQuatern < 0)
        fail("Missing gridpoints quaternions. After QUATERNIONS (int). (int)=Number of gridpoins per dimension");
      const int G = p.GridPointsQuatern + 1;
      const float d = 2.f / (float) G;
      for (int a = 0; a < G; a++)
      {
        const float q1 = (float) a * d - 1.f + 0.5 * d;
        for (int b = 0; b < G; b++)
        {
          const float q2 = (float) b * d - 1.f + 0.5 * d;
          for (int c = 0; c < G; c++)
          {
            const float q3 = (float) c * d - 1.f + 0.5 * d;
            if (q1 * q1 + q2 * q2 + q3 * q3 <= 1.f)
            {
              const float q4 = sqrt(1.f - q1 * q1 - q2 * q2 - q3 * q3);
              const float row[8] = {q1, q2, q3, q4, q1, q2, q3, -q4};
              p.angles.insert(p.angles.end(), row, row + 8);
            }
          }
        }
      }
      p.voluang = d * d * d * p.priorMod;
    }
  }
  else
  {
    std::ifstream in(orientfile.c_str());
    if (!in.good())
      fail(p.doquater ? "Quaterion list file %s" : "Euler angle file failed to open file %s", orientfile.c_str());
    std::string line;
    std::getline(in, line);
    int count = 0;
    {
      char buf[13] = {0};
      strncpy(buf, line.c_str(), 12);
      if (sscanf(buf, "%d", &count) != 1)
        fail("orientation list %s: cannot read the number of orientations", orientfile.c_str());
    }
    if (count < 1)
      fail(p.doquater ? "Invalid number of quaternions %d" : "Euler angles not defined in input file", count);
    std::cout << (p.doquater ? "Number of quaternions " : "Number of Euler angles ") << count << "\n";
    const int ncol = p.doquater ? 4 : 3;
    int nrow = 0;
    while (std::getline(in, line))
    {
      float v[5] = {0, 0, 0, 0, 0};
      for (int k = 0; k < ncol; k++)
        if (!fixed_col(line, k, &v[k]))
          fail("orientation list %s: row %d, column %d is not a number", orientfile.c_str(), nrow, k);
      if (p.doquater)
        for (int k = 0; k < 4; k++)
          if (v[k] < -1 || v[k] > 1)
            fail("Reading quaterions from list. Value out of range %lf row %d", (double) v[k], nrow);
      if (p.yespriorAngles)
      {
        float pp = 0.f;
        if (!fixed_col(line, ncol, &pp))
          fail("orientation list %s: row %d has no prior column", orientfile.c_str(), nrow);
        if (pp < 0.0000001)
          std::cout << "Sure your input is correct? Very small prior.\n";
        p.angprior.push_back(pp);
      }
      p.angles.push_back(v[0]);
      p.angles.push_back(v[1]);
      p.angles.push_back(v[2]);
      p.angles.push_back(p.doquater ? v[3] : 0.f);
      nrow++;
      if (count < nrow)
        fail("More orientations than expected in header %d instead of %d", nrow, count);
    }
    if (count > nrow)
      fail("Less orientations than expected in header %d instead of %d", nrow, count);
    p.voluang = 1. / (float) count * p.priorMod;
  }
  if (p.doquater)
    std::cout << "Analysis with Quaternions. Total number of quaternions " << p.nOrient() << "\n";
}

// param.cpp:1336-1620 (table + volu), through the library's host entry points
void make_ctf_table(Params &p)
{
  float grids[3];
  if (p.startAmp < 0 || p.endAmp > 1)
    fail("PSF amplitude should be between 0 and 1. start: %lf end: %lf", (double) p.startAmp, (double) p.endAmp);
  if (p.usepsf)
  {
    // kernels in real space; the library takes their r2c transform on the device (param.cpp:1466-1535)
    p.nCtf = bioem_b200_host_psf_kernels(p.N, p.pixelSize, p.startAmp, p.endAmp, p.nAmp, p.startPhase, p.endPhase, p.nPhase,
                                         p.startEnv, p.endEnv, p.nEnv, nullptr, nullptr, grids);
    if (p.nCtf <= 0)
      fail("PSF grid is empty");
    p.psfKernels.assign((size_t) p.nCtf * p.N * p.N, 0.f);
    p.CtfParam.assign((size_t) p.nCtf * 4, 0.f);
    const int got = bioem_b200_host_psf_kernels(p.N, p.pixelSize, p.startAmp, p.endAmp, p.nAmp, p.startPhase, p.endPhase,
                                                p.nPhase, p.startEnv, p.endEnv, p.nEnv, p.psfKernels.data(), p.CtfParam.data(),
                                                grids);
    if (got == -3)
      fail("MAX standard deviation of envelope is larger than allowed KERNEL length");
    if (got != p.nCtf)
      fail("PSF table: %d kernels built, %d expected", got, p.nCtf);
  }
  else
  {
    p.nCtf = bioem_b200_host_ctf_table(p.N, p.pixelSize, 0, p.startAmp, p.endAmp, p.nAmp, p.startPhase, p.endPhase, p.nPhase,
                                       p.startEnv, p.endEnv, p.nEnv, nullptr, nullptr, grids);
    if (p.nCtf <= 0)
      fail("CTF grid is empty");
    const size_t F = (size_t) p.N * (p.N / 2 + 1);
    p.refCTF.assign((size_t) p.nCtf * F * 2, 0.f);
    p.CtfParam.assign((size_t) p.nCtf * 4, 0.f);
    const int got = bioem_b200_host_ctf_table(p.N, p.pixelSize, 0, p.startAmp, p.endAmp, p.nAmp, p.startPhase, p.endPhase,
                                              p.nPhase, p.startEnv, p.endEnv, p.nEnv, p.refCTF.data(), p.CtfParam.data(), grids);
    if (got != p.nCtf)
      fail("CTF table: %d kernels built, %d expected", got, p.nCtf);
  }
  p.volu = bioem_b200_host_volu(p.voluang, p.GridSpaceCenter, p.pixelSize, p.maxDisplaceCenter, p.nAmp, grids[2], grids[1],
                                p.sigmaPriorbctf, p.sigmaPriordefo, p.sigmaPrioramp);
}

void make_ctf_groups(const std::string &file, int nMaps, Params &p)
{
  if (p.usepsf)
    fail("--DefocusPerParticle: USE_PSF kernels are complex; CTF groups need CTF_DEFOCUS tables");
  std::ifstream in(file.c_str());
  if (!in.good())
    fail("--DefocusPerParticle: cannot open %s", file.c_str());
  std::vector<float> vals;
  std::string tok;
  while (in >> tok)
  {
    char *end = nullptr;
    const float v = strtof(tok.c_str(), &end);
    if (end == tok.c_str() || *end != 0)
      fail("--DefocusPerParticle %s: entry %d (%s) is not a number", file.c_str(), (int) vals.size(), tok.c_str());
    vals.push_back(v);
  }
  if ((int) vals.size() != nMaps)
    fail("--DefocusPerParticle %s: %d values for %d particles", file.c_str(), (int) vals.size(), nMaps);
  std::vector<float> defs; // one per group, in order of first appearance
  p.group.assign(nMaps, 0);
  for (int m = 0; m < nMaps; m++)
  {
    const auto it = std::find(defs.begin(), defs.end(), vals[m]);
    p.group[m] = (int) (it - defs.begin());
    if (it == defs.end())
      defs.push_back(vals[m]);
  }
  const int G = (int) defs.size();
  const float half = 0.5f * (p.endDef - p.startDef);
  const size_t F = (size_t) p.N * (p.N / 2 + 1);
  std::vector<float> ref, par;
  p.groupDefcent.assign(G, 0.f);
  float volu0 = 0.f;
  int C = 0;
  for (int g = 0; g < G; g++)
  {
    const float d0 = defs[g] - half, d1 = defs[g] + half;
    // the reference's checks of CTF_DEFOCUS (param.cpp), per group
    if (d0 < 0)
      fail("--DefocusPerParticle: defocus %g: Negative start defocus (%g)", (double) defs[g], (double) d0);
    if (d1 > 8.)
      fail("--DefocusPerParticle: defocus %g: Defocus beyond 8micro-m range is not allowed (%g)", (double) defs[g],
           (double) d1);
    float ph0, ph1, cen = defs[g];
    bioem_b200_host_defocus_to_phase(d0, d1, p.elecwavel, &ph0, &ph1, &cen, nullptr);
    float grids[3];
    const int c = bioem_b200_host_ctf_table(p.N, p.pixelSize, 0, p.startAmp, p.endAmp, p.nAmp, ph0, ph1, p.nPhase, p.startEnv,
                                            p.endEnv, p.nEnv, nullptr, nullptr, grids);
    if (c <= 0 || (g > 0 && c != C))
      fail("--DefocusPerParticle: defocus %g: CTF grid of %d kernels", (double) defs[g], c);
    C = c;
    ref.resize((size_t) (g + 1) * C * F * 2);
    par.resize((size_t) (g + 1) * C * 4);
    bioem_b200_host_ctf_table(p.N, p.pixelSize, 0, p.startAmp, p.endAmp, p.nAmp, ph0, ph1, p.nPhase, p.startEnv, p.endEnv,
                              p.nEnv, &ref[(size_t) g * C * F * 2], &par[(size_t) g * C * 4], grids);
    // every group has the grid steps of CTF_DEFOCUS, so the same volu (up to the rounding of the phase step)
    const float volu = bioem_b200_host_volu(p.voluang, p.GridSpaceCenter, p.pixelSize, p.maxDisplaceCenter, p.nAmp, grids[2],
                                            grids[1], p.sigmaPriorbctf, p.sigmaPriordefo, p.sigmaPrioramp);
    if (g == 0)
      volu0 = volu;
    else if (!(fabsf(volu - volu0) <= 1e-5f * fabsf(volu0)))
      fail("--DefocusPerParticle: defocus %g: volume element %g differs from the first group's %g", (double) defs[g],
           (double) volu, (double) volu0);
    p.groupDefcent[g] = cen;
  }
  p.refCTF.swap(ref);
  p.CtfParam.swap(par);
  p.nCtf = C;
  p.nGroups = G;
  p.volu = volu0;
  std::cout << "CTF groups: " << G << " defocus values, " << C << " CTF kernels each\n";
}

// --------------------------------------------------------------------------- MRC helpers
// include/mrc.h:72-149: the byte order is guessed from how many header fields fall outside
// plausible ranges under each interpretation.
static unsigned bswap32(unsigned v) { return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24); }
struct MrcHeader
{
  int nc = 0, nr = 0, ns = 0, mode = 0, nsymbt = 0;
  bool swap = false;
};
static int mrc_range_violations(const unsigned *w, bool swap)
{
  auto I = [&](int i) { return (int) (swap ? bswap32(w[i]) : w[i]); };
  auto Fl = [&](int i) {
    unsigned u = swap ? bswap32(w[i]) : w[i];
    float f;
    memcpy(&f, &u, 4);
    return f;
  };
  int v = 0;
  for (int i = 0; i < 3; i++)
    v += (I(i) > 5000) + (I(i) < 0);
  for (int i = 4; i < 7; i++)
    v += (I(i) > 5000) + (I(i) < -5000);
  for (int i = 7; i < 10; i++)
    v += (I(i) > 5000) + (I(i) < 0);
  for (int i = 13; i < 16; i++)
    v += (Fl(i) > 360.0f) + (Fl(i) < -360.0f);
  return v;
}
static MrcHeader read_mrc_header(FILE *f, const char *name)
{
  unsigned w[256];
  if (fread(w, 4, 256, f) != 256)
    fail("Reading MRC header: %s", name);
  MrcHeader h;
  const int v0 = mrc_range_violations(w, false), v1 = mrc_range_violations(w, true);
  h.swap = !(v0 < v1);
  const int v = h.swap ? v1 : v0;
  if (v > 0)
    warn("%i header field range violations detected in file %s", v, name);
  auto I = [&](int i) { return (int) (h.swap ? bswap32(w[i]) : w[i]); };
  h.nc = I(0);
  h.nr = I(1);
  h.ns = I(2);
  h.mode = I(3);
  h.nsymbt = I(23);
  return h;
}
static void read_mrc_floats(FILE *f, float *dst, size_t n, bool swap, const char *name)
{
  if (fread(dst, 4, n, f) != n)
    fail("Converting Data: %s", name);
  if (swap)
    for (size_t i = 0; i < n; i++)
    {
      unsigned u;
      memcpy(&u, &dst[i], 4);
      u = bswap32(u);
      memcpy(&dst[i], &u, 4);
    }
}

// --WriteBestMaps: maps[i][x][y] as one mode-2 stack, stored as the reader expects it (read_particles with --ReadMRC
// stores file[j*N + i] at maps[i*N + j], so the file holds each image transposed)
void write_mrc_stack(const std::string &file, const float *maps, int N, int n)
{
  int w[256];
  memset(w, 0, sizeof(w));
  w[0] = N; // nc, nr, ns
  w[1] = N;
  w[2] = n;
  w[3] = 2; // mode: 32-bit float
  w[7] = N; // mx, my, mz
  w[8] = N;
  w[9] = 1;
  const float cell[6] = {(float) N, (float) N, 1.f, 90.f, 90.f, 90.f};
  memcpy(&w[10], cell, sizeof(cell));
  w[16] = 1; // mapc, mapr, maps
  w[17] = 2;
  w[18] = 3;
  const size_t n2 = (size_t) N * N;
  float mn = n ? maps[0] : 0.f, mx = mn;
  double sum = 0.0;
  for (size_t k = 0; k < n2 * n; k++)
  {
    mn = std::min(mn, maps[k]);
    mx = std::max(mx, maps[k]);
    sum += maps[k];
  }
  const float st[3] = {mn, mx, n ? (float) (sum / (double) (n2 * n)) : 0.f};
  memcpy(&w[19], st, sizeof(st));
  memcpy(&w[52], "MAP ", 4);
  w[53] = 0x00004444; // little-endian machine stamp
  FILE *f = fopen(file.c_str(), "wb");
  if (!f)
    fail("Opening file: %s", file.c_str());
  bool ok = fwrite(w, 4, 256, f) == 256;
  std::vector<float> t(n2);
  for (int m = 0; m < n && ok; m++)
  {
    const float *img = maps + (size_t) m * n2;
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++)
        t[(size_t) j * N + i] = img[(size_t) i * N + j];
    ok = fwrite(t.data(), sizeof(float), n2, f) == n2;
  }
  if (fclose(f) != 0 || !ok)
    fail("Writing file: %s", file.c_str());
}

// --------------------------------------------------------------------------- model
// residue tables of the reference's C-alpha model (model.cpp:738-844): radius [A], electrons
static const struct
{
  const char *name;
  float radius, electrons;
} kResidues[] = {{"CYS", 2.75f, 64.f}, {"PHE", 3.2f, 88.f},  {"LEU", 3.1f, 72.f},  {"TRP", 3.4f, 108.f}, {"VAL", 2.95f, 64.f},
                 {"ILE", 3.1f, 72.f},  {"MET", 3.1f, 80.f},  {"HIS", 3.05f, 82.f}, {"TYR", 3.25f, 96.f}, {"ALA", 2.5f, 48.f},
                 {"GLY", 2.25f, 40.f}, {"PRO", 2.8f, 62.f},  {"ASN", 2.85f, 66.f}, {"THR", 2.8f, 64.f},  {"SER", 2.6f, 56.f},
                 {"ARG", 3.3f, 93.f},  {"GLN", 3.0f, 78.f},  {"ASP", 2.8f, 59.f},  {"LYS", 3.2f, 79.f},  {"GLU", 2.95f, 53.f}};

static bool has_ext(const std::string &s, const char *ext)
{
  const size_t found = s.find(ext), end = s.find_last_not_of(" \t");
  return found != std::string::npos && found <= end;
}

// --PrintCOORDREAD: the (centred) model as the reference lists it (model.cpp:712-740)
static void print_coordread(const std::vector<bioem_b200_model_point> &pts)
{
  std::cout << "Note - Look at file COORDREAD to confirm that the Model coordinates are correct\n";
  std::ofstream out("COORDREAD");
  out << "Text --- Number ---- x ---- y ---- z ---- radius ---- number of electron\n";
  for (size_t n = 0; n < pts.size(); n++)
    out << "RESIDUE " << n << " " << pts[n].pos[0] << " " << pts[n].pos[1] << " " << pts[n].pos[2] << " " << pts[n].radius
        << " " << pts[n].density << "\n";
}

void read_model(const Options &o, const Params &p, std::vector<bioem_b200_model_point> &pts, float &NormDen)
{
  pts.clear();
  if (o.loadModelDump)
  {
    // model.dump: float NormDen, int nPoints, nPoints x 24-byte points (model.cpp:41-82)
    FILE *f = fopen("model.dump", "rb");
    if (!f)
      fail("Opening file: model.dump");
    int n = 0;
    if (fread(&NormDen, sizeof(float), 1, f) != 1 || fread(&n, sizeof(int), 1, f) != 1 || n <= 0)
      fail("Reading model dump");
    pts.resize(n);
    if (fread(pts.data(), sizeof(bioem_b200_model_point), n, f) != (size_t) n)
      fail("Reading model dump");
    fclose(f);
    std::cout << "Protein structure read from model dump\n";
    // like the reference, a dump holds the model as read: it is centred after loading, with the
    // NormDen stored in the dump (model.cpp:676-707, 604-672)
    if (!p.nocentermass)
    {
      float cm[3] = {0.f, 0.f, 0.f};
      for (const auto &pt : pts)
        for (int k = 0; k < 3; k++)
          cm[k] += pt.pos[k] * pt.density;
      for (int k = 0; k < 3; k++)
        cm[k] /= NormDen;
      for (auto &pt : pts)
        for (int k = 0; k < 3; k++)
          pt.pos[k] -= cm[k];
    }
    std::cout << "Total Number of Voxels " << pts.size() << "\nTotal Number of Electrons " << NormDen << "\n+++++++++++++++++++++++++++++++++++++++++ \n";
    if (o.printCoordRead)
      print_coordread(pts);
    return;
  }
  const char *name = o.modelfile.c_str();
  if (o.readPDB)
  {
    // ATOM records whose atom name (columns 13-16) is CA; residue name columns 18-20,
    // coordinates columns 31-54 (model.cpp:85-329)
    if (!has_ext(o.modelfile, ".pdb"))
      warn("PDB extension NOT detected in file name: %s. Are you sure you want to read a PDB?", name);
    std::ifstream in(name);
    if (!in.good())
      fail("Opening file: %s", name);
    std::string line;
    while (std::getline(in, line))
    {
      if (line.size() < 54)
        continue;
      char type[7] = {0}, atom[5] = {0}, res[4] = {0};
      sscanf(line.substr(0, 6).c_str(), "%6s", type);
      sscanf(line.substr(12, 4).c_str(), "%4s", atom);
      if (strcmp(type, "ATOM") != 0 || strcmp(atom, "CA") != 0)
        continue;
      sscanf(line.substr(17, 3).c_str(), "%3s", res);
      double x = 0, y = 0, z = 0;
      if (sscanf(line.substr(30, 24).c_str(), "%lf %lf %lf", &x, &y, &z) != 3)
        fail("PDB %s: cannot read the coordinates of '%s'", name, line.c_str());
      bioem_b200_model_point pt;
      pt.pos[0] = (float) x;
      pt.pos[1] = (float) y;
      pt.pos[2] = (float) z;
      pt.quat4 = 0.f;
      pt.radius = pt.density = 0.f;
      bool known = false;
      for (const auto &r : kResidues)
        if (strcmp(res, r.name) == 0)
        {
          pt.radius = r.radius;
          pt.density = r.electrons;
          known = true;
        }
      if (!known)
        fail("Residue Name %s not valid", res);
      pts.push_back(pt);
    }
    std::cout << "Protein structure read from PDB\n";
  }
  else if (o.readModelMRC)
  {
    // mode-2 volume: one point per voxel, radius 2 pixels, density = voxel (model.cpp:332-416)
    if (!has_ext(o.modelfile, ".mrc"))
      warn("MRC extension NOT detected in file name: %s. Are you sure you want to read an MRC?", name);
    FILE *f = fopen(name, "rb");
    if (!f)
      fail("Opening MRC: %s", name);
    const MrcHeader h = read_mrc_header(f, name);
    if (fseek(f, 1024 + h.nsymbt, SEEK_SET) != 0)
      fail("Converting Data: %s", name);
    const size_t total = (size_t) h.nc * h.nr * h.ns;
    std::vector<float> vox(total);
    read_mrc_floats(f, vox.data(), total, h.swap, name);
    fclose(f);
    pts.reserve(total);
    size_t idx = 0;
    // the reference walks (i, j, k) = 1..nx, 1..ny, 1..nz with k fastest over the file order
    for (int i = 1; i <= h.nc; i++)
      for (int j = 1; j <= h.nr; j++)
        for (int k = 1; k <= h.ns; k++)
        {
          bioem_b200_model_point pt;
          pt.pos[0] = (i - h.nc / 2.0) * p.pixelSize;
          pt.pos[1] = (j - h.nr / 2.0) * p.pixelSize;
          pt.pos[2] = (k - h.ns / 2.0) * p.pixelSize;
          pt.quat4 = 0.f;
          pt.radius = 2.0 * p.pixelSize;
          pt.density = vox[idx++];
          pts.push_back(pt);
        }
    std::cout << "Protein structure read from MRC\n";
  }
  else
  {
    // text: x y z radius density per line (model.cpp:419-601)
    std::cout << "Note: Reading model in simple text format\n----  x   y   z  radius  density ------- \n";
    if (has_ext(o.modelfile, ".pdb"))
    {
      warn("PDB detected in file name: %s. Are you sure you do not need --ReadPDB? If so then you must include the "
           "keyword IGNORE_PDB in inputfile",
           name);
      if (!p.ignorePDB)
        fail("PDB is not ignored");
    }
    std::ifstream in(name);
    if (!in.good())
      fail("Opening file: %s", name);
    std::string line;
    while (std::getline(in, line))
    {
      double v[5];
      if (sscanf(line.c_str(), "%lf %lf %lf %lf %lf", &v[0], &v[1], &v[2], &v[3], &v[4]) != 5)
        continue;
      if (v[3] < 0)
        fail("Radius must be positive");
      bioem_b200_model_point pt;
      pt.pos[0] = (float) v[0];
      pt.pos[1] = (float) v[1];
      pt.pos[2] = (float) v[2];
      pt.quat4 = 0.f;
      pt.radius = (float) v[3];
      pt.density = (float) v[4];
      pts.push_back(pt);
    }
    std::cout << "Protein structure read from Standard File\n";
  }
  if (pts.empty())
    fail("No model points read from %s", name);
  // NormDen; --DumpModel writes the model as read, before the centring (model.cpp:695-698); then the centre of
  // density unless NO_CENTEROFMASS (model.cpp:229-234,604-672,704-707)
  NormDen = bioem_b200_host_model_prepare(pts.data(), (int) pts.size(), 0);
  if (o.dumpModel)
  {
    FILE *f = fopen("model.dump", "wb");
    if (!f)
      fail("Opening file: model.dump");
    const int n = (int) pts.size();
    fwrite(&NormDen, sizeof(float), 1, f);
    fwrite(&n, sizeof(int), 1, f);
    fwrite(pts.data(), sizeof(bioem_b200_model_point), n, f);
    fclose(f);
  }
  NormDen = bioem_b200_host_model_prepare(pts.data(), (int) pts.size(), p.nocentermass ? 0 : 1);
  std::cout << "Total Number of Voxels " << pts.size() << "\nTotal Number of Electrons " << NormDen << "\n+++++++++++++++++++++++++++++++++++++++++ \n";
  if (o.printCoordRead)
    print_coordread(pts);
}

// --------------------------------------------------------------------------- particles
static void append_mrc_stack(const std::string &file, const Params &p, std::vector<float> &maps, int &nMaps)
{
  // mode-2 stack; image stored transposed (maps[i*N + j] with the file running j-outer / i-inner),
  // then zero mean / unit deviation with float accumulators unless NO_MAP_NORM (map.cpp:663-853)
  const char *name = file.c_str();
  FILE *f = fopen(name, "rb");
  if (!f)
    fail("Opening MRC: %s", name);
  const MrcHeader h = read_mrc_header(f, name);
  printf("\n+++++++++++++++++++++++++++++++++++++++++++\nReading Information from MRC: %s \n", name);
  printf("Number Columns  = %8d \nNumber Rows     = %8d \nNumber Sections = %8d \n", h.nc, h.nr, h.ns);
  printf("MODE = %4d (only data type mode 2: 32-bit)\nNSYMBT = %4d (# bytes symmetry operators)\n", h.mode, h.nsymbt);
  if (h.nr != p.N || h.nc != p.N)
    fail("Inconsistent number of pixels in maps and inputfile ( %d, i %d, j %d)", p.N, h.nc, h.nr);
  if (h.mode != 2)
    fail("MRC mode: %d. Currently mode 2 is the only one allowed", h.mode);
  if (fseek(f, 1024 + h.nsymbt, SEEK_SET) != 0)
    fail("Converting Data: %s", name);
  const size_t n2 = (size_t) p.N * p.N;
  maps.resize((size_t) (nMaps + h.ns) * n2);
  read_mrc_floats(f, maps.data() + (size_t) nMaps * n2, n2 * h.ns, h.swap, name); // file order, untouched
  nMaps += h.ns;
  fclose(f);
}

// image stored transposed (maps[i*N + j] with the file running j-outer / i-inner), then zero mean /
// unit deviation with float accumulators in file order unless NO_MAP_NORM (map.cpp:811-845)
void mrc_host_ingest(const Params &p, std::vector<float> &maps, int nMaps)
{
  const size_t n2 = (size_t) p.N * p.N;
  std::vector<float> img(n2);
  for (int s = 0; s < nMaps; s++)
  {
    float *dst = maps.data() + (size_t) s * n2;
    std::copy(dst, dst + n2, img.begin());
    for (int j = 0; j < p.N; j++)
      for (int i = 0; i < p.N; i++)
        dst[(size_t) i * p.N + j] = img[(size_t) j * p.N + i];
    if (!p.notnormmap)
      bioem_b200_host_normalise_map(dst, p.N);
  }
}

void read_particles(const Options &o, const Params &p, std::vector<float> &maps, int &nMaps, bool &rawMRC)
{
  maps.clear();
  nMaps = 0;
  rawMRC = false;
  const size_t n2 = (size_t) p.N * p.N;
  if (o.loadMapDump)
  {
    // maps.dump: int nMaps, nMaps x N x N float (map.cpp:44-78)
    FILE *f = fopen("maps.dump", "rb");
    if (!f)
      fail("Opening file: maps.dump");
    if (fread(&nMaps, sizeof(int), 1, f) != 1 || nMaps <= 0)
      fail("Reading map dump");
    maps.resize((size_t) nMaps * n2);
    if (fread(maps.data(), sizeof(float), maps.size(), f) != maps.size())
      fail("Reading map dump");
    fclose(f);
    std::cout << "Particle Maps read from Map Dump\n";
  }
  else if (o.readMRC)
  {
    if (o.readMultMRC)
    {
      // a list of MRC file names, one per line, optionally closed by a line starting with XXX (map.cpp:85-135)
      std::cout << "Opening File with MRC list names: " << o.particlesfile << "\n";
      std::ifstream in(o.particlesfile.c_str());
      if (!in.good())
        fail("Failed to open file contaning MRC names: %s", o.particlesfile.c_str());
      std::string line;
      while (std::getline(in, line))
      {
        if (line.compare(0, 3, "XXX") == 0)
          continue;
        const size_t e = line.find_last_not_of(" \t\r");
        if (e == std::string::npos)
          continue;
        line = line.substr(0, e + 1);
        if (line.find("mrc") == std::string::npos)
          warn("MRC extension NOT detected in file name: %s. Are you sure you want to read an MRC?", line.c_str());
        append_mrc_stack(line, p, maps, nMaps);
      }
    }
    else
      append_mrc_stack(o.particlesfile, p, maps, nMaps);
    rawMRC = true;
    std::cout << "Particle Maps read from MRC\n";
  }
  else
  {
    // text: "PARTICLE ..." header line per image, then N*N lines "%8d%8d%16.8f" (i, j, value),
    // the last one (N-1, N-1) (map.cpp:268-414)
    std::ifstream in(o.particlesfile.c_str());
    if (!in.good())
      fail("Particle Maps Failed to open file %s", o.particlesfile.c_str());
    std::string line;
    bool first = true;
    float *cur = nullptr;
    int li = -1, lj = -1;
    auto close_particle = [&]() {
      if (cur && (li != p.N - 1 || lj != p.N - 1))
        fail("Inconsistent number of pixels in maps and inputfile ( %d, i %d, j %d)", p.N, li, lj);
    };
    while (std::getline(in, line))
    {
      if (line.compare(0, 8, "PARTICLE") == 0)
      {
        close_particle();
        maps.resize((size_t) (nMaps + 1) * n2, 0.f);
        cur = maps.data() + (size_t) nMaps * n2;
        nMaps++;
        li = lj = -1;
        first = false;
        continue;
      }
      if (first)
        fail("Missing correct standard map format: PARTICLE HEADER");
      if (line.size() < 32)
        continue;
      int i = 0, j = 0;
      float z = 0.f;
      char a[9] = {0}, b[9] = {0}, c[17] = {0};
      strncpy(a, line.c_str(), 8);
      strncpy(b, line.c_str() + 8, 8);
      strncpy(c, line.c_str() + 16, 16);
      if (sscanf(a, "%d", &i) != 1 || sscanf(b, "%d", &j) != 1 || sscanf(c, "%f", &z) != 1)
        fail("Particle file %s: malformed line '%s'", o.particlesfile.c_str(), line.c_str());
      cur = maps.data() + (size_t) (nMaps - 1) * n2; // resize may have moved the block
      if (i > -1 && i < p.N && j > -1 && j < p.N)
        cur[(size_t) i * p.N + j] = z;
      else
        fail("PARTICLE format: pixel (%d, %d) outside the %d x %d image", i, j, p.N, p.N);
      li = i;
      lj = j;
    }
    close_particle();
    std::cout << "Particle Maps read from Standard File\n";
  }
  if (nMaps <= 0)
    fail("No particle images read from %s", o.particlesfile.c_str());
  if (getenv("BIOEM_DEBUG_NMAPS")) // the reference's debugging knob (map.cpp:545-548)
  {
    const int cap = atoi(getenv("BIOEM_DEBUG_NMAPS"));
    if (cap > 0 && cap < nMaps)
    {
      nMaps = cap;
      maps.resize((size_t) nMaps * n2);
    }
  }
  if (o.dumpMaps)
  {
    if (rawMRC) // the dump holds the maps as the reference keeps them in memory
    {
      mrc_host_ingest(p, maps, nMaps);
      rawMRC = false;
    }
    FILE *f = fopen("maps.dump", "wb");
    if (!f)
      fail("Opening file: maps.dump");
    fwrite(&nMaps, sizeof(int), 1, f);
    fwrite(maps.data(), sizeof(float), maps.size(), f);
    fclose(f);
  }
  std::cout << "Total Number of particles: " << nMaps << "\n+++++++++++++++++++++++++++++++++++++++++++ \n";
}

} // namespace bhost
