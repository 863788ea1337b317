// bioEM_b200: the reference's bioEM command line on top of libbioem_b200.so.
//
//   bioEM_b200 --Modelfile m --Particlesfile p --Inputfile i [--ReadOrientation o] [--ReadPDB]
//              [--ReadModelMRC] [--ReadMRC] [--ReadMultipleMRC] [--DumpMaps] [--LoadMapDump]
//              [--DumpModel] [--LoadModelDump] [--PrintCOORDREAD] [--OutputFile f] [--Gpus n]
//              [--WriteBestMaps f] [--DefocusPerParticle f]
//
// Flow = the reference's main.cpp:34-140 / bioem::configure / bioem::run with the main loop
// (bioem.cpp:763-891) replaced by bioem_b200_run on every GPU of the box: the orientation grid is
// split in contiguous blocks (the reference's MPI split, bioem.cpp:748-753), one host thread
// drives one GPU, and the per-image partial results are merged in block order on the devices, over peer
// memory (bioem_b200_merge_peers: strict '<', so ties resolve to the lowest orientation like a 1-process run).
#include "bioem_host.hpp"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <queue>
#include <thread>

using namespace bhost;

#define B200(call)                                                                                          \
  do                                                                                                        \
  {                                                                                                         \
    if ((call) != BIOEM_B200_OK)                                                                            \
      fail("%s: %s", #call, bioem_b200_last_error());                                                       \
  } while (0)

namespace bhost
{

// reference bioem.cpp:1046-1374 (ofstream, fixed, precision OUTPUT_PRECISION = 4, defs.h:177)
void write_outputs(const Options &o, const Params &p, const bioem_b200_config &cfg,
                   const std::vector<bioem_b200_prob_map> &pm, const std::vector<bioem_b200_top_angle> &cand, int nCand,
                   int nMaps)
{
  const char *stars = "************************* HEADER:: NOTATION *******************************************\n";
  const double addc = 0.5 * log(M_PI) + (1 - cfg.Ntotpi * 0.5) * (log(2 * M_PI) + 1) + log(cfg.volu);
  std::ofstream ang;
  ang.precision(4);
  ang.setf(std::ios::fixed);
  if (cfg.writeAngles)
  {
    ang.open("ANG_PROB");
    ang << stars;
    if (!p.doquater)
      ang << " RefMap:  MapNumber ; alpha[rad] - beta[rad] - gamma[rad] - logP - cal log Probability + Constant: "
             "Numerical Const.+ log (volume) + prior ang\n";
    else
      ang << " RefMap:  MapNumber ; q1 - q2 -q3 - logP- cal log Probability + Constant: Numerical Const. + log "
             "(volume) + prior ang\n";
    ang << stars;
  }
  std::ofstream out;
  out.precision(4);
  out.setf(std::ios::fixed);
  out.open(o.outfile.c_str());
  if (!out.good())
    fail("Opening file: %s", o.outfile.c_str());
  out << stars;
  out << "Notation= RefMap:  MapNumber ; LogProb natural logarithm of posterior Probability ; Constant: Numerical "
         "Const. for adding Probabilities \n";
  if (!p.doquater)
    out << "Notation= RefMap:  MapNumber ; Maximizing Param: MaxLogProb - alpha[rad] - beta[rad] - gamma[rad] - "
        << (p.usepsf ? "PSF amp - PSF phase - PSF envelope" : "CTF amp - CTF defocus - CTF B-Env")
        << " - center x - center y - normalization - offsett \n";
  else if (p.usepsf)
    out << "Notation= RefMap:  MapNumber ; Maximizing Param: MaxLogProb - q1 - q2 - q3 - q4 -PSF amp - PSF phase - PSF "
           "envelope - center x - center y - normalization - offsett \n";
  else
    out << "Notation= RefMap:  MapNumber ; Maximizing Param: MaxLogProb - q1 - q2 - q3 - q4 - CTF amp - CTF defocus - CTF "
           "B-Env - center x - center y - normalization - offsett \n";
  if (p.writeCTF)
    out << " RefMap:  MapNumber ; CTFMaxParm: defocus - b-Env (B ref. Penzeck 2010)\n";
  if (p.yespriorAngles)
    out << "**** Remark: Using Prior Proability in Angles ****\n";
  out << stars << "\n";

  for (int m = 0; m < nMaps; m++)
  {
    const bioem_b200_prob_map &r = pm[m];
    if (r.Total > 1.e-38)
    {
      const double lp = log(r.Total) + r.Constoadd + addc;
      out << "RefMap: " << m << " LogProb:  " << lp << " Constant: " << r.Constoadd << "\n";
      out << "RefMap: " << m << " Maximizing Param: " << lp << " ";
    }
    else
    {
      out << "Warning - RefMap: " << m << "Numerical Integrated Probability without constant = 0.0;\n";
      out << "Warning - RefMap: " << m << "Check that constant is finite: " << r.Constoadd << "\n";
      out << "Warning - RefMap: i) check model, ii) check refmap , iii) check GPU on/off command inconsitency\n";
    }
    const float *a = &p.angles[(size_t) 4 * r.max_prob_orient];
    const float *c = &p.CtfParam[(size_t) 4 * r.max_prob_conv];
    out << a[0] << " [] " << a[1] << " [] " << a[2] << " [] ";
    if (p.doquater)
      out << a[3] << " [] ";
    out << c[0] << " [] ";
    if (!p.usepsf)
      out << c[1] / 2.f / M_PI / p.elecwavel * 0.0001 << " [micro-m] " << c[2] << " [A²] ";
    else
      out << c[1] << " [1/A²] " << c[2] << " [1/A²] ";
    out << r.max_prob_cent_x << " [pix] " << r.max_prob_cent_y << " [pix] " << r.max_prob_norm << " [] " << r.max_prob_mu
        << " [] \n";
    if (p.writeCTF && p.usepsf)
    {
      // PSF parameters of the maximum converted back to CTF defocus / B-envelope (bioem.cpp:1215-1232)
      const float denomi = c[1] * c[1] + c[2] * c[2];
      out << "RefMap: " << m << " CTFMaxParam: ";
      out << 2 * M_PI * c[1] / denomi / p.elecwavel * 0.0001 << " [micro-m] ";
      out << 4 * M_PI * M_PI * c[2] / denomi << " [A²] \n";
    }

    if (cfg.writeAngles)
    {
      // the K most probable orientations of this image, most probable first: the reference's min-heap of
      // size K (bioem.cpp:1254-1290), fed with the rows the GPUs kept, in ascending orientation order
      const unsigned K = (unsigned) cfg.writeAngles;
      typedef std::pair<double, int> PI; // (logp, index into this image's candidate rows)
      std::priority_queue<PI, std::vector<PI>, std::greater<PI>> q;
      const bioem_b200_top_angle *rows = &cand[(size_t) m * nCand];
      for (int i = 0; i < nCand; i++)
      {
        if (rows[i].orient < 0)
          continue;
        const double logp = log(rows[i].forAngles) + rows[i].ConstAngle + addc;
        if (q.size() < K)
          q.push(PI(logp, i));
        else if (q.top().first < logp)
        {
          q.pop();
          q.push(PI(logp, i));
        }
      }
      std::vector<PI> best(q.size());
      for (int i = (int) best.size() - 1; i >= 0; i--)
      {
        best[i] = q.top();
        q.pop();
      }
      for (const PI &b : best)
      {
        const bioem_b200_top_angle &pr = rows[b.second];
        const int io = pr.orient;
        double logp = b.first;
        if (p.yespriorAngles)
          logp += p.angprior[io];
        const float *an = &p.angles[(size_t) 4 * io];
        ang << " " << m << " " << an[0] << " " << an[1] << " " << an[2] << " ";
        if (p.doquater)
          ang << an[3] << " ";
        ang << logp << " Separated: " << log(pr.forAngles) << " " << pr.ConstAngle << " " << addc;
        if (p.yespriorAngles)
          ang << " " << p.angprior[io];
        ang << "\n";
      }
    }
  }
}

} // namespace bhost

int main(int argc, char **argv)
{
  const auto t0 = std::chrono::steady_clock::now();
  Options opt;
  Params par;
  std::cout << " ++++++++++++ FROM COMMAND LINE +++++++++++\n\n";
  parse_options(argc, argv, opt);
  par.notuniformangles = !opt.orientfile.empty();
  if (par.notuniformangles)
    std::cout << "Reading Orientation from File: " << opt.orientfile << "\n";

  printf("Configuring\n");
  read_parameters(opt.inputfile, par);
  std::vector<float> maps;
  int nMaps = 0;
  bool rawMRC = false;
  read_particles(opt, par, maps, nMaps, rawMRC);
  std::vector<bioem_b200_model_point> pts;
  float NormDen = 0.f;
  read_model(opt, par, pts, NormDen);
  make_orientations(opt.orientfile, par);
  make_ctf_table(par);
  if (!opt.defocusfile.empty())
  {
    if (getenv("BIOEM_DEBUG_BREAK") || getenv("BIOEM_B200_DUMP_INPUTS"))
      fail("--DefocusPerParticle: BIOEM_DEBUG_BREAK / BIOEM_B200_DUMP_INPUTS take one CTF table");
    make_ctf_groups(opt.defocusfile, nMaps, par);
  }

  int O = par.nOrient(), C = par.nCtf;
  if (getenv("BIOEM_DEBUG_BREAK")) // the reference's debugging knob (bioem.cpp:518-525)
  {
    const int cut = atoi(getenv("BIOEM_DEBUG_BREAK"));
    O = std::min(O, cut);
    C = std::min(C, cut);
    par.angles.resize((size_t) 4 * O);
  }

  if (const char *dump = getenv("BIOEM_B200_DUMP_INPUTS"))
  {
    // test hook: write what would be uploaded, then stop before any device work
    auto wr = [&](const char *name, const void *ptr, size_t bytes) {
      const std::string path = std::string(dump) + "/" + name;
      FILE *f = fopen(path.c_str(), "wb");
      if (!f || fwrite(ptr, 1, bytes, f) != bytes)
        fail("cannot write %s", path.c_str());
      fclose(f);
    };
    if (rawMRC)
      mrc_host_ingest(par, maps, nMaps);
    wr("points.bin", pts.data(), pts.size() * sizeof(pts[0]));
    wr("maps.bin", maps.data(), maps.size() * sizeof(float));
    wr("angles.bin", par.angles.data(), par.angles.size() * sizeof(float));
    wr("ctfparam.bin", par.CtfParam.data(), (size_t) C * 4 * sizeof(float));
    if (par.usepsf)
      wr("psfkernels.bin", par.psfKernels.data(), (size_t) C * par.N * par.N * sizeof(float));
    else
      wr("refctf.bin", par.refCTF.data(), (size_t) C * par.N * (par.N / 2 + 1) * 2 * sizeof(float));
    const std::string meta = std::string(dump) + "/meta.txt";
    FILE *f = fopen(meta.c_str(), "w");
    if (!f)
      fail("cannot write %s", meta.c_str());
    fprintf(f, "N %d\nM %d\nO %d\nC %d\nA %d\nNormDen %.9g\nvolu %.9g\nsigmaPriordefo %.9g\nPriordefcent %.9g\n", par.N,
            nMaps, O, C, (int) pts.size(), (double) NormDen, (double) par.volu, (double) par.sigmaPriordefo,
            (double) par.Priordefcent);
    fclose(f);
    printf("inputs dumped to %s\n", dump);
    return 0;
  }

  if (!bioem_b200_supported_size(par.N))
    printf("NUMBER_PIXELS %d has no fused FFT kernel (even edges 16..512 with prime factors 2/3/5/7 have): running on "
           "the direct-DFT path, same results, many times slower\n",
           par.N);
  int ndev = bioem_b200_device_count();
  if (ndev == 0)
    fail("no CUDA device: bioEM_b200 has no CPU path");
  const int nphys = ndev;
  // BIOEM_B200_OVERSUBSCRIBE=1: more orientation blocks (handles) than GPUs, block g on GPU g % nphys -- the
  // multi-GPU code path (blocks, device merge) on a box with fewer GPUs (tests)
  const bool oversub = getenv("BIOEM_B200_OVERSUBSCRIBE") && atoi(getenv("BIOEM_B200_OVERSUBSCRIBE")) != 0;
  int want = opt.gpus > 0 ? opt.gpus : ndev;
  if (getenv("BIOEM_B200_GPUS"))
    want = std::max(1, atoi(getenv("BIOEM_B200_GPUS")));
  ndev = oversub ? std::min(want, 16) : std::min(ndev, want);
  ndev = std::min(ndev, O); // the reference needs at least one orientation per rank (bioem.cpp:675-678)

  bioem_b200_config cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.NumberPixels = par.N;
  cfg.maxDisplaceCenter = par.maxDisplaceCenter;
  cfg.GridSpaceCenter = par.GridSpaceCenter;
  cfg.writeAngles = par.writeAngles;
  cfg.tousepsf = par.usepsf;
  cfg.doquater = par.doquater;
  cfg.shiftX = par.shiftX;
  cfg.shiftY = par.shiftY;
  cfg.pixelSize = par.pixelSize;
  cfg.Ntotpi = (float) (par.N * par.N);
  cfg.volu = par.volu;
  cfg.sigmaPriorbctf = par.sigmaPriorbctf;
  cfg.sigmaPriordefo = par.sigmaPriordefo;
  cfg.Priordefcent = par.Priordefcent;
  cfg.sigmaPrioramp = par.sigmaPrioramp;
  cfg.Priorampcent = par.Priorampcent;

  printf("\n+++++++++++++++++++++++++++++++++++++++++++\n");
  printf("Running %d orientation block%s on %d GPU%s: %d orientations x %d CTF kernels x %d particles, %d x %d pixels\n", ndev,
         ndev > 1 ? "s" : "", std::min(ndev, nphys), std::min(ndev, nphys) > 1 ? "s" : "", O, C, nMaps, par.N, par.N);
  const auto t1 = std::chrono::steady_clock::now();

  // One host thread drives each GPU through its block of orientations; the per-image results are then merged
  // ON THE DEVICES: GPU 0 reads the other GPUs' partial states over NVLink peer memory inside the merge kernel
  // (bioem_b200_merge_peers), and for WRITE_PROB_ANGLES every GPU keeps the K most probable orientations of its
  // block per particle, merged the same way (bioem_b200_merge_top_angles_peers).
  const int K = cfg.writeAngles;
  std::vector<bioem_b200_handle> handles(ndev, nullptr);
  std::vector<int> oB(ndev), oE(ndev);
  std::vector<std::string> errors(ndev);
  auto worker = [&](int g) {
    const int o0 = (int) ((long long) g * O / ndev), o1 = (int) ((long long) (g + 1) * O / ndev);
    oB[g] = o0;
    oE[g] = o1;
    bioem_b200_handle h = nullptr;
    auto chk = [&](int rc, const char *what) {
      if (rc != BIOEM_B200_OK && errors[g].empty())
        errors[g] = std::string(what) + ": " + bioem_b200_last_error();
      return rc == BIOEM_B200_OK;
    };
    chk(bioem_b200_create(&cfg, g % nphys, &h), "create") &&
        chk(bioem_b200_upload_model(h, pts.data(), (int) pts.size(), NormDen), "upload_model") &&
        chk(bioem_b200_upload_orientations(h, par.angles.data(), O), "upload_orientations") &&
        chk(par.nGroups ? bioem_b200_upload_ctf_groups(h, par.refCTF.data(), par.CtfParam.data(), par.groupDefcent.data(),
                                                       par.nGroups, C)
            : par.usepsf ? bioem_b200_upload_ctf_real(h, par.psfKernels.data(), par.CtfParam.data(), C)
                         : bioem_b200_upload_ctf(h, par.refCTF.data(), par.CtfParam.data(), C),
            "upload_ctf") &&
        chk(rawMRC ? bioem_b200_upload_particles_mrc(h, maps.data(), nMaps, par.notnormmap ? 0 : 1)
                   : bioem_b200_upload_particles(h, maps.data(), nMaps),
            "upload_particles") &&
        (!par.nGroups || chk(bioem_b200_set_particle_groups(h, par.group.data(), nMaps), "set_particle_groups")) &&
        chk(bioem_b200_reset(h), "reset") && chk(bioem_b200_run(h, o0, o1), "run") &&
        chk(bioem_b200_synchronize(h), "synchronize");
    handles[g] = h;
  };
  std::vector<std::thread> th;
  for (int g = 0; g < ndev; g++)
    th.emplace_back(worker, g);
  for (auto &t : th)
    t.join();
  for (int g = 0; g < ndev; g++)
    if (!errors[g].empty())
      fail("GPU %d: %s", g, errors[g].c_str());

  // the reference warns once per projection that loses model points (bioem.cpp:1724-1734,1756-1780)
  {
    std::vector<int> per(O);
    for (int g = 0; g < ndev; g++)
    {
      long long tot = 0;
      B200(bioem_b200_out_of_frame(handles[g], per.data(), &tot));
      for (int o = oB[g]; o < oE[g] && tot > 0; o++)
        if (per[o] > 0)
          printf("Warning - Projection %d (rank %d): point out of image size. Please check that the input model is "
                 "correct. (%d model points skipped)\n",
                 0, o, per[o]);
    }
  }

  std::vector<bioem_b200_prob_map> pm(nMaps);
  B200(bioem_b200_merge_peers(handles.data(), ndev));
  B200(bioem_b200_download(handles[0], pm.data(), nullptr));
  const int nCand = K;
  std::vector<bioem_b200_top_angle> cand((size_t) nMaps * nCand);
  if (K)
  {
    B200(bioem_b200_merge_top_angles_peers(handles.data(), oB.data(), oE.data(), ndev, K, cand.data()));
    // the writer feeds its heap in ascending orientation order
    for (int m = 0; m < nMaps; m++)
    {
      bioem_b200_top_angle *row = &cand[(size_t) m * nCand];
      std::stable_sort(row, row + nCand, [](const bioem_b200_top_angle &a, const bioem_b200_top_angle &b) {
        return (unsigned) a.orient < (unsigned) b.orient; // -1 (unused) last
      });
    }
  }
  // --WriteBestMaps: the merged records rendered on GPU 0 (its handle holds every input)
  std::vector<float> bestmaps;
  if (!opt.bestmapsfile.empty())
  {
    bestmaps.resize((size_t) nMaps * par.N * par.N);
    B200(bioem_b200_render_maps(handles[0], pm.data(), nMaps, bestmaps.data()));
  }
  for (int g = 0; g < ndev; g++)
    bioem_b200_destroy(handles[g]);
  const auto t2 = std::chrono::steady_clock::now();

  write_outputs(opt, par, cfg, pm, cand, nCand, nMaps);
  if (!opt.bestmapsfile.empty())
    write_mrc_stack(opt.bestmapsfile, bestmaps.data(), par.N, nMaps);
  const auto t3 = std::chrono::steady_clock::now();
  auto sec = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  printf("Likelihood path (upload .. merge): %f seconds, %.3e likelihoods/s\n", sec(t1, t2),
         (double) O * C * nMaps / sec(t1, t2));
  printf("The code ran for %f seconds (rank 0).\n", sec(t0, t3));
  return 0;
}
