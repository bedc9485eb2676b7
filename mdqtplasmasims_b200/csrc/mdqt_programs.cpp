// mdqt_programs.cpp -- the host loops of the reference's OTHER programs on top of the C ABI, selected with
// `mdqt_run --program <name> <job> [options]`, writing the reference's own files:
//
//   md       MonteCarloFollowedByMDAndTempAnisotropy.cpp main() (MD:1030-1167), stages 1 and 4-8: collisional MD, the
//            collisionless recording stage (tagged-particle moments, temperature, g(r), velocity store), the four power
//            autocorrelations, the instantaneous-anisotropy stage, re-equilibration, and the laser-force anisotropy stages.
//   fz408l   randomFrozenStartTag408Linear.cpp main() (FZ408L:981-1076): frozen random start, leap-frog time loop with the
//            408 nm pump window, spin measurement and the tagged velocity autocorrelation.
//   fz408q, fz422l   its siblings randomFrozenStartTag408Quad.cpp (circular resonant pump, v_x^2 autocorrelation) and
//            randomFrozenStartTag422Linear.cpp (5-level 422 nm scheme): the same main() with their defaults and differences.
//   ts       laserCoolNoPlasmaThreeState.cpp main() (TS:352-409): free ions in a J = 0 -> J = 1 molasses, energies.dat.
//   mc408l, mc422l   MonteCarloFollowedByQTTagging408Linear.cpp / ...422Linear.cpp main() (MC408L:1140-1254, MC422L:1100-1222), stages 1, 4-7: collisional MD, the pump stage
//            (62 x 7-level qstep() per MDStep), the projective spin measurement, the recording stage with the tagged ions' moments
//            and velocity distribution, the autocorrelations.
//
// The Metropolis Monte-Carlo pre-equilibration of the MD family (MD:207-382, stage 3 of its main) is one sequential
// accept/reject chain -- "replicas only" (SURVEY.md 8(e)) -- and is NOT run here: the MD program starts from the lattice of
// init() (MD:174-205) or from positions given with --positions, and the collisional stage equilibrates it.
// Host random numbers that the reference draws from std::mt19937 (initial Maxwellian, velocity-dependent tagging) use the
// same standard generator and distributions in the same order, seeded with --seed (the reference seeds from random_device);
// the Andersen collisions of the MD steps are Philox streams on the device.
#include "../../include/mdqt.h"
#include "../../include/mdqt_io.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <chrono>
#include <map>
#include <random>
#include <string>
#include <vector>

namespace {

void prog_die(const char* what) {
  fprintf(stderr, "mdqt_run: %s: %s\n", what, mdqt_last_error());
  exit(1);
}
#define CKP(call) do { if ((call) != 0) prog_die(#call); } while (0)

typedef std::map<std::string, std::string> OptMap;
bool parse_opts(int argc, char** argv, int first, OptMap& opt, bool* quiet) {
  for (int i = first; i < argc; i++) {
    std::string a = argv[i];
    if (a == "--quiet") { *quiet = true; continue; }
    if (a.rfind("--", 0) != 0 || !opt.count(a.substr(2)) || i + 1 >= argc) { fprintf(stderr, "mdqt_run: bad option %s\n", a.c_str()); return false; }
    opt[a.substr(2)] = argv[++i];
  }
  return true;
}
int as_unsigned_printed(double x) { return (int)(long long)x; }  // (unsigned) cast printed with %d, as in mdqt_io_dirname

FILE* open_in(const std::string& dir, const char* name, const char* mode) {
  FILE* f = fopen((dir + name).c_str(), mode);
  if (!f) { fprintf(stderr, "mdqt_run: cannot open %s%s\n", dir.c_str(), name); exit(1); }
  return f;
}

// recordPairPairCorr(k) (MD:584-652): the file
void write_gr(mdqt_handle* h, const std::string& dir, int k, double step, double rmax) {
  const int nb = (int)(rmax / step);
  std::vector<double> g(nb);
  CKP(mdqt_pair_correlation(h, step, rmax, nb, g.data(), NULL));
  char name[64];
  snprintf(name, sizeof(name), "pairPairCorrStepNum%d.dat", k);
  FILE* fa = open_in(dir, name, "w");
  for (int i = 0; i < nb; i++) fprintf(fa, "%lg\t%lg\n", i * step, g[i]);  // MD:649
  fclose(fa);
}

// recordTempForEachAxis(fileName, k) (MD:560-582) for every recorded step of a stage
void write_axis_temps(const std::string& dir, const char* name, const std::vector<double>& rec, int nsteps, int N, double timeStep) {
  FILE* fa = open_in(dir, name, "a");
  for (int k = 0; k < nsteps; k++) {
    const double* r = &rec[(size_t)k * 23];
    fprintf(fa, "%lg\t%lg\t%lg\t%lg\n", k * timeStep, r[0] / N, r[1] / N, r[2] / N);  // MD:578
  }
  fclose(fa);
}

// --stress 1 of the md program (no counterpart in the reference): the pressure tensor of every recorded step and the Green-Kubo
// shear-stress autocorrelation, full precision (%.17g) because they feed further integrals.
//   stressTensor.dat    k*timeStep, K_xx K_yy K_zz K_xy K_xz K_yz, W_xx W_yy W_zz W_xy W_xz W_yz (mdqt_stress_download)
//   stressAutoCorr.dat  tD*timeStep, C(tD), eta(tD) = trapezoid integral of C from 0 to tD / (V Tbar), V = L^3 and Tbar = the stage
//                       mean of (K_xx + K_yy + K_zz) / (3N), the quantity temperature.dat prints
void write_stress(mdqt_handle* h, const std::string& dir, int nsteps, int N, double L, double timeStep) {
  std::vector<double> st((size_t)12 * nsteps), acf(nsteps);
  CKP(mdqt_stress_download(h, st.data(), nsteps));
  CKP(mdqt_stress_autocorr(h, nsteps, acf.data()));
  FILE* fs = open_in(dir, "stressTensor.dat", "w");
  double tsum = 0.0;
  for (int k = 0; k < nsteps; k++) {
    fprintf(fs, "%.17g", k * timeStep);
    for (int q = 0; q < 12; q++) fprintf(fs, "\t%.17g", st[(size_t)q * nsteps + k]);
    fprintf(fs, "\n");
    tsum += (st[k] + st[(size_t)nsteps + k] + st[(size_t)2 * nsteps + k]) / (3.0 * N);
  }
  fclose(fs);
  const double Tbar = tsum / nsteps, V = L * L * L;
  FILE* fa = open_in(dir, "stressAutoCorr.dat", "w");
  double integral = 0.0;
  for (int tD = 0; tD < nsteps; tD++) {
    if (tD > 0) integral += 0.5 * (acf[tD - 1] + acf[tD]) * timeStep;
    fprintf(fa, "%.17g\t%.17g\t%.17g\n", tD * timeStep, acf[tD], integral / (V * Tbar));
  }
  fclose(fa);
}

// --heat 1 of the md program (no counterpart in the reference): the heat current of every recorded step and the Green-Kubo
// heat-current autocorrelation, full precision (%.17g) because they feed further integrals.
//   heatCurrent.dat    k*timeStep, J_kin (3), J_pot (3), J_vir (3), P (3), E_kin, E_pot, tr W (mdqt_heat_download)
//   heatAutoCorr.dat   tD*timeStep, C(tD), lambda(tD) = trapezoid integral of C from 0 to tD / (V Tbar^2), V = L^3 and Tbar = the
//                      stage mean of 2 E_kin / (3N), the quantity temperature.dat prints
void write_heat(mdqt_handle* h, const std::string& dir, int nsteps, int N, double L, double timeStep) {
  std::vector<double> hc((size_t)15 * nsteps), acf(nsteps);
  CKP(mdqt_heat_download(h, hc.data(), nsteps));
  CKP(mdqt_heat_autocorr(h, nsteps, acf.data()));
  FILE* fh = open_in(dir, "heatCurrent.dat", "w");
  double tsum = 0.0;
  for (int k = 0; k < nsteps; k++) {
    fprintf(fh, "%.17g", k * timeStep);
    for (int q = 0; q < 15; q++) fprintf(fh, "\t%.17g", hc[(size_t)q * nsteps + k]);
    fprintf(fh, "\n");
    tsum += 2.0 * hc[(size_t)12 * nsteps + k] / (3.0 * N);
  }
  fclose(fh);
  const double Tbar = tsum / nsteps, V = L * L * L;
  FILE* fa = open_in(dir, "heatAutoCorr.dat", "w");
  double integral = 0.0;
  for (int tD = 0; tD < nsteps; tD++) {
    if (tD > 0) integral += 0.5 * (acf[tD - 1] + acf[tD]) * timeStep;
    fprintf(fa, "%.17g\t%.17g\t%.17g\n", tD * timeStep, acf[tD], integral / (V * Tbar * Tbar));
  }
  fclose(fa);
}

// --modes NMAX of the md program (no counterpart in the reference): the collective modes of the axis wave vectors k = 2 pi n / L
// along x, y and z, n = 1..NMAX (mdqt_modes_autocorr), each averaged over the three axes, full precision (%.17g):
//   intermediateScattering.dat   tD*timeStep, F(k_n, tD) for n = 1..NMAX
//   currentCorrL.dat             tD*timeStep, C_L(k_n, tD) for n = 1..NMAX
//   currentCorrT.dat             tD*timeStep, C_T(k_n, tD) for n = 1..NMAX
//   staticStructureFactor.dat    n, k_n, S(k_n) = F(k_n, 0)
// The recorder's vector q = 3 (n - 1) + a is n along axis a.
void write_modes(mdqt_handle* h, const std::string& dir, int nsteps, int nmax, double L, double timeStep) {
  const size_t K = (size_t)3 * nmax;
  std::vector<double> ac[3];
  for (auto& a : ac) a.resize(K * nsteps);
  CKP(mdqt_modes_autocorr(h, nsteps, ac[0].data(), ac[1].data(), ac[2].data()));
  auto avg = [&](const std::vector<double>& a, int n, int tD) {
    const size_t q = (size_t)3 * (n - 1);
    return (a[q * nsteps + tD] + a[(q + 1) * nsteps + tD] + a[(q + 2) * nsteps + tD]) / 3.0;
  };
  static const char* names[3] = {"intermediateScattering.dat", "currentCorrL.dat", "currentCorrT.dat"};
  for (int c = 0; c < 3; c++) {
    FILE* f = open_in(dir, names[c], "w");
    for (int tD = 0; tD < nsteps; tD++) {
      fprintf(f, "%.17g", tD * timeStep);
      for (int n = 1; n <= nmax; n++) fprintf(f, "\t%.17g", avg(ac[c], n, tD));
      fprintf(f, "\n");
    }
    fclose(f);
  }
  FILE* fs = open_in(dir, "staticStructureFactor.dat", "w");
  for (int n = 1; n <= nmax; n++) fprintf(fs, "%d\t%.17g\t%.17g\n", n, 2 * M_PI * n / L, avg(ac[0], n, 0));
  fclose(fs);
}

}  // namespace

// ---- MonteCarloFollowedByMDAndTempAnisotropy.cpp -----------------------------------------------------------------------------
int mdqt_program_md(int argc, char** argv) {
  OptMap opt = {{"N", "4096"}, {"Gamma", "3"}, {"kappa", "0.5"}, {"density", "0.4"}, {"timeStep", "0.005"}, {"collisionFreq", "0.25"},
                {"preSteps", "200"}, {"recordSteps", "2500"}, {"instSteps", "2500"}, {"reequilSteps", "500"}, {"establishSteps", "-1"},
                {"relaxSteps", "2000"}, {"tempPercentDiff", "0.15"}, {"beta", "26000"}, {"establishTime", "10"}, {"oneAxis", "0"},
                {"pairPairStep", "0.05"}, {"seed", ""}, {"saveDirectory", "data/"}, {"device", "0"}, {"program", "md"}, {"stress", "0"}, {"heat", "0"},
                {"modes", "0"}};
  bool quiet = false;
  if (argc < 2 || argv[1][0] == '-') {
    fprintf(stderr, "usage: mdqt_run --program md <job> [--N n] [--Gamma x] [--kappa x] ... [--stress 0|1] [--heat 0|1] [--modes NMAX]\n"
                    "       --stress 1: also record the pressure tensor at every step of the recording stage (stressTensor.dat) and its\n"
                    "                   Green-Kubo shear-stress autocorrelation with the running viscosity integral (stressAutoCorr.dat)\n"
                    "       --heat 1:   also record the heat current at every step of the recording stage (heatCurrent.dat) and its\n"
                    "                   Green-Kubo autocorrelation with the running thermal-conductivity integral (heatAutoCorr.dat)\n"
                    "       --modes NMAX: also record the density and current Fourier modes of k = 2 pi n / L along x, y and z,\n"
                    "                   n = 1..NMAX (at most 341), at every step of the recording stage; write the intermediate scattering\n"
                    "                   function and the longitudinal and transverse current correlations, axis-averaged\n"
                    "                   (intermediateScattering.dat, currentCorrL.dat, currentCorrT.dat), and S(k) (staticStructureFactor.dat)\n");
    return 2;
  }
  const unsigned job = (unsigned)atof(argv[1]);  // MD:1035
  if (!parse_opts(argc, argv, 2, opt, &quiet)) return 2;
  const int N = atoi(opt["N"].c_str());
  const double Gamma = atof(opt["Gamma"].c_str()), kappa = atof(opt["kappa"].c_str()), n = atof(opt["density"].c_str());
  const double timeStep = atof(opt["timeStep"].c_str()), collFreq = atof(opt["collisionFreq"].c_str());
  const int preSteps = atoi(opt["preSteps"].c_str()), recSteps = atoi(opt["recordSteps"].c_str()), instSteps = atoi(opt["instSteps"].c_str());
  const int reeqSteps = atoi(opt["reequilSteps"].c_str()), relaxSteps = atoi(opt["relaxSteps"].c_str());
  const double tempPercentDiff = atof(opt["tempPercentDiff"].c_str()), beta = atof(opt["beta"].c_str());
  int estSteps = atoi(opt["establishSteps"].c_str());
  if (estSteps < 0) estSteps = (int)round(.8 * atof(opt["establishTime"].c_str()) * sqrt(n) / timeStep);  // MD:101
  const int oneAxis = atoi(opt["oneAxis"].c_str());
  const double pairPairStep = atof(opt["pairPairStep"].c_str());
  const unsigned seed = opt["seed"].empty() ? (unsigned)time(NULL) + job : (unsigned)atol(opt["seed"].c_str());
  const bool stress = atoi(opt["stress"].c_str()) != 0;
  const bool heat = atoi(opt["heat"].c_str()) != 0;
  const int modes = atoi(opt["modes"].c_str());
  if (modes < 0 || 3 * modes > 1024) { fprintf(stderr, "mdqt_run: modes must be in [0, 341]\n"); return 2; }
  if (recSteps > 5000) { fprintf(stderr, "mdqt_run: recordSteps must be <= 5000\n"); return 2; }

  // directory tree (MD:1037-1058)
  std::string dir = opt["saveDirectory"];
  mkdir(dir.c_str(), 0777);
  char namebuf[256];
  snprintf(namebuf, sizeof(namebuf), "Gamma%dKappa%dNumIons%d", as_unsigned_printed(Gamma * 100), as_unsigned_printed(kappa * 100), N);
  dir += namebuf;
  mkdir(dir.c_str(), 0777);
  snprintf(namebuf, sizeof(namebuf), "/job%d/", (int)job);
  dir += namebuf;
  mkdir(dir.c_str(), 0777);

  // init() (MD:174-205): cubic lattice, Maxwellian velocities from std::mt19937 + normal_distribution in the reference's order
  mdqt_params p;
  CKP(mdqt_params_md(&p, MDQT_SCHEME_NONE, N, kappa, n, timeStep, 0.0, 0.0, 0));
  p.traj0 = (int)job; p.seed = seed; p.device = atoi(opt["device"].c_str());
  const double L = p.L;
  std::mt19937 rng(seed);
  std::normal_distribution<double> velocityDistribution(0, sqrt(1 / Gamma));
  std::uniform_real_distribution<double> uni(0, 1);
  std::vector<double> R((size_t)3 * N, 0.0), V((size_t)3 * N, 0.0);
  {
    int N0 = 0;
    const int side = (int)round(pow(N, 1. / 3));
    for (int i = 0; i < side; i++)
      for (int j = 0; j < side; j++)
        for (int k = 0; k < side; k++) {
          if (N0 >= N) break;
          R[N0] = i * L / pow(N, 1 / 3.) + 0.5; R[(size_t)N + N0] = j * L / pow(N, 1 / 3.) + 0.5; R[(size_t)2 * N + N0] = k * L / pow(N, 1 / 3.) + 0.5;
          V[N0] = velocityDistribution(rng); V[(size_t)N + N0] = velocityDistribution(rng); V[(size_t)2 * N + N0] = velocityDistribution(rng);
          N0++;
        }
    if (N0 != N) { fprintf(stderr, "mdqt_run: N must be a cube (the reference's lattice init, MD:66)\n"); return 2; }
  }
  mdqt_handle* h = NULL;
  CKP(mdqt_create(&p, &h));
  CKP(mdqt_upload_state(h, R.data(), V.data(), NULL, NULL, N));
  // A = 0 until the first MDStep computes it, as in the reference (its global A[][] is never evaluated before MD:1089)
  const double sigma_v = sqrt(1 / Gamma), laser_coeff = 1.234e-6 * beta / sqrt(n);
  const double rmax = L / 2;
  auto wall0 = std::chrono::steady_clock::now();

  // stage 4: collisional MD (MD:1081-1090)
  if (preSteps > 0) CKP(mdqt_vv_steps(h, preSteps, 0, timeStep, collFreq, sigma_v, 0, 0.0));

  // stage 5: collisionless MD with the recorders (MD:1093-1105)
  {
    // tagParticles() (MD:809-921) on the host: one pass over v_x with the reference's draws
    CKP(mdqt_download_state(h, NULL, V.data(), NULL, NULL, N));
    std::vector<uint8_t> tags(N);
    const double vT = sqrt(1 / Gamma);
    for (int i = 0; i < N; i++) {
      const double v = V[i];
      double roll;
      bool t1, t2, t3, t4;
      if (v < -3 * vT) t1 = false;
      else if (v > 3 * vT) t1 = true;
      else { roll = uni(rng); t1 = roll < (.5 + v / vT / 6); }
      const double c2 = .5 / 9 / vT / vT;
      roll = uni(rng);
      if (v < -3 * vT || v > 3 * vT) t2 = !(roll < .5);
      else t2 = roll < (c2 * v * v);
      const double c3 = .5 / 27 / vT / vT / vT;
      if (v < -3 * vT) t3 = false;
      else if (v > 3 * vT) t3 = true;
      else { roll = uni(rng); t3 = roll < (.5 + c3 * v * v * v); }
      const double c4 = .5 / 81 / vT / vT / vT / vT;
      roll = uni(rng);
      if (v < -3 * vT || v > 3 * vT) t4 = !(roll < .5);
      else t4 = roll < (c4 * v * v * v * v);
      tags[i] = (uint8_t)((t1 ? 1 : 0) | (t2 ? 2 : 0) | (t3 ? 4 : 0) | (t4 ? 8 : 0));
    }
    if (recSteps > 0) {
      CKP(mdqt_set_tags(h, tags.data()));
      CKP(mdqt_moments_begin(h, recSteps));
      CKP(mdqt_vstore_begin(h, recSteps));
      if (stress) CKP(mdqt_stress_begin(h, recSteps));
      if (heat) CKP(mdqt_heat_begin(h, recSteps));
      std::vector<int32_t> nvec((size_t)9 * modes, 0);  // the axis vectors: q = 3 (n - 1) + a is n along axis a
      for (int q = 0; q < 3 * modes; q++) nvec[(size_t)3 * q + q % 3] = q / 3 + 1;
      if (modes) CKP(mdqt_modes_begin(h, nvec.data(), 3 * modes, recSteps));
      for (int k = 0; k < recSteps; k++) {
        CKP(mdqt_moments_record(h, k));                          // recordTaggedParticleMoments(k), recordTemperature()
        if (stress) CKP(mdqt_stress_record(h, k));               // the pressure tensor of the same state: row k of temperature.dat
        if (heat) CKP(mdqt_heat_record(h, k));                   // the heat current of the same state
        if (modes) CKP(mdqt_modes_record(h, k));                 // rho_k and j_k of the same state
        if (k % 100 == 0) { if (!quiet) printf("%d\n", k); write_gr(h, dir, k, pairPairStep, rmax); }  // MD:1097-1100
        CKP(mdqt_vv_step(h, timeStep, 0.0, sigma_v, 0, 0.0));    // MDStep(k)
        CKP(mdqt_vstore_record(h, k));                           // recordVelsForAutocorrelations(k)
      }
      std::vector<double> rec((size_t)recSteps * 23);
      CKP(mdqt_moments_download(h, rec.data(), recSteps));
      static const char* names[4] = {"taggedVOneMoments.dat", "taggedVTwoMoments.dat", "taggedVThreeMoments.dat", "taggedVFourMoments.dat"};
      FILE* ft = open_in(dir, "temperature.dat", "a");
      FILE* fm[4];
      for (int s = 0; s < 4; s++) fm[s] = open_in(dir, names[s], "a");
      for (int k = 0; k < recSteps; k++) {
        const double* r = &rec[(size_t)k * 23];
        for (int s = 0; s < 4; s++) {  // MD:976-1026
          const double cnt = r[3 + 5 * s];
          fprintf(fm[s], "%lg\t%lg\t%lg\t%lg\t%lg\n", k * timeStep, r[4 + 5 * s] / cnt, r[5 + 5 * s] / cnt - 1 / (Gamma), r[6 + 5 * s] / cnt,
                  r[7 + 5 * s] / cnt - 3 / (Gamma * Gamma));
        }
        fprintf(ft, "%lg\n", (r[0] + r[1] + r[2]) / (3.0 * N));  // MD:536-544
      }
      fclose(ft);
      for (int s = 0; s < 4; s++) fclose(fm[s]);
      // stage 6: recordVAF, recordLongViscAutoCorr, recordVCubeAutoCorr, recordVFourthAutoCorr (MD:1107-1110)
      std::vector<double> ac[4];
      for (auto& a : ac) a.resize(recSteps);
      CKP(mdqt_autocorrelations(h, Gamma, ac[0].data(), ac[1].data(), ac[2].data(), ac[3].data()));
      static const char* acn[4] = {"VAF.dat", "longViscAutoCorr.dat", "vCubeAutoCorr.dat", "vFourthAutoCorr.dat"};
      for (int s = 0; s < 4; s++) {
        FILE* fa = open_in(dir, acn[s], "w");
        for (int tD = 0; tD < recSteps; tD++) fprintf(fa, "%lg\t%lg\n", tD * timeStep, ac[s][tD]);
        fclose(fa);
      }
      if (stress) write_stress(h, dir, recSteps, N, L, timeStep);
      if (heat) write_heat(h, dir, recSteps, N, L, timeStep);
      if (modes) write_modes(h, dir, recSteps, modes, L, timeStep);
      CKP(mdqt_set_tags(h, NULL));
    }
  }

  // stage 7: instantaneous anisotropy (MD:1113-1123), then collisional re-equilibration (MD:1125-1135)
  auto axis_stage = [&](const char* file, int nsteps, int laser) {
    if (nsteps <= 0) return;
    CKP(mdqt_moments_begin(h, nsteps));
    for (int k = 0; k < nsteps; k++) {
      CKP(mdqt_moments_record(h, k));                                                    // recordTempForEachAxis(fileName, k)
      CKP(mdqt_vv_step(h, timeStep, 0.0, sigma_v, laser, laser ? laser_coeff : 0.0));    // MDStep(k)
    }
    std::vector<double> rec((size_t)nsteps * 23);
    CKP(mdqt_moments_download(h, rec.data(), nsteps));
    write_axis_temps(dir, file, rec, nsteps, N, timeStep);
  };
  CKP(mdqt_scale_velocities(h, sqrt(1 + tempPercentDiff), sqrt(1 - tempPercentDiff / 2), sqrt(1 - tempPercentDiff / 2)));  // MD:548-558
  axis_stage("TemperaturesAlongAxesInstantaneous.dat", instSteps, 0);
  if (reeqSteps > 0) CKP(mdqt_vv_steps(h, reeqSteps, 0, timeStep, 0.25, sigma_v, 0, 0.0));

  // stage 8: anisotropy through the laser force, then relaxation (MD:1137-1165)
  axis_stage("TemperaturesAlongAxesDuringForcePeriod.dat", estSteps, oneAxis ? 2 : 1);
  axis_stage("TemperaturesAlongAxesAfterForcePeriod.dat", relaxSteps, 0);
  CKP(mdqt_sync(h));
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
  if (!quiet)
    fprintf(stderr, "mdqt_run: program md, job %u, N=%d: %d + %d + %d + %d + %d + %d MD steps in %.3f s; files in %s\n", job, N, preSteps, recSteps,
            instSteps, reeqSteps, estSteps, relaxSteps, wall, dir.c_str());
  mdqt_destroy(h);
  return 0;
}

// ---- randomFrozenStartTag408Linear.cpp ----------------------------------------------------------------------------------------
// main() (FZ408L:981-1076): frozen random start, leap-frog step() every `ratio` loop iterations, the 408 nm pump (7-level
// qstep(), frozen velocities) inside the window (tstartV0, tendV0), measureSpinUps() once at its end, then output() + Zfunc() +
// printVAF() every sampleFreq MD steps; writeConditions(c0) at the end. Files as the reference writes them: energies.dat
// (FZ408L:831), taggedMoments.dat (:871), vel_distX_timestep%06d.dat (4001 bins, the tagged ions only, :845-893), VAF.dat
// (:963-973), ions_/spinUpIonsList_/conditions_timestep%06d.dat (:667-707).
namespace {
struct FzOut {
  mdqt_handle* h; std::string dir; int N, ld; double Epot0; unsigned counter;
  std::vector<double> V; std::vector<int32_t> spin;
};
// output() (FZ408L:799-915)
void fz_output(FzOut& o, double t, int c0) {
  CKP(mdqt_download_state(o.h, NULL, o.V.data(), NULL, NULL, o.ld));
  double epot = 0.0;
  CKP(mdqt_epot(o.h, &epot));
  const int N = o.N, ld = o.ld;
  double ek[3] = {0, 0, 0};
  for (int c = 0; c < 3; c++) {
    for (int i = 0; i < N; i++) ek[c] += 0.5 * (o.V[(size_t)c * ld + i] * o.V[(size_t)c * ld + i]);
    ek[c] /= (double)N;
  }
  FILE* fa = open_in(o.dir, "energies.dat", "a");
  fprintf(fa, "%lg\t%lg\t%lg\t%lg\t%lg\t%lg\n", t, ek[0], ek[1], ek[2], epot, ek[0] + ek[1] + ek[2] + epot - o.Epot0);  // :831
  fclose(fa);
  // moments and the velocity distribution of the spin-up (tagged) ions: Gaussian weights of width 0.002 on 4001 bins (:835-893)
  const double V2 = 1. / (2. * 0.002 * 0.002);
  std::vector<double> pv(4001, 0.0);
  double m1 = 0, m2 = 0, m3 = 0, m4 = 0;
  unsigned numTagged = 0;
  for (int i = 0; i < N; i++) {
    const double v = o.V[i];
    if (!o.spin[i]) continue;
    m1 += v; m2 += v * v; m3 += v * v * v; m4 += v * v * v * v; numTagged += 1;
    if (o.spin[i] == 1)
      for (int j = 0; j < 4001; j++) { const double vel = (double)(j - 2000) * 0.0025; pv[j] += exp(-V2 * (vel - v) * (vel - v)); }
  }
  fa = open_in(o.dir, "taggedMoments.dat", "a");
  fprintf(fa, "%lg\t%lg\t%lg\t%lg\t%lg\n", t, m1 / numTagged, m2 / numTagged, m3 / numTagged, m4 / numTagged);  // :871
  fclose(fa);
  char name[64];
  snprintf(name, sizeof(name), "vel_distX_timestep%06d.dat", c0);
  fa = open_in(o.dir, name, "w");
  for (int j = 0; j < 4001; j++) fprintf(fa, "%lg\t%lg\n", (double)(j - 2000) * 0.0025, pv[j] / (6.0 * sqrt(2 * M_PI * 0.002 * 0.002)));  // :877-893
  fclose(fa);
  o.counter++;
}
void fz_print_vaf(const FzOut& o, double t, double vaf, const char* file = "VAF.dat") {
  FILE* fa = open_in(o.dir, file, "a");
  fprintf(fa, "%lg\t%lg\n", t, vaf);  // :971
  fclose(fa);
}
}  // namespace

// The same main() serves the two sibling programs (`variant`):
//   fz408q  randomFrozenStartTag408Quad.cpp: ONE circularly polarised resonant 408 nm laser -- the coupling keeps two of its four
//           terms (FZ408Q:441: the `quad` mask of the 7-level kernel), defaults detuning 0, Om 2, tpumpreal 1e-7 (FZ408Q:58-60), and
//           Zfunc() is the v_x^2 autocorrelation "LongKin" written to vSquareAutoCorr.dat (FZ408Q:942-979).
//   fz422l  randomFrozenStartTag422Linear.cpp: the 5-level 422 nm pump with its unit conversions (FZ422L:66-74: g2E x 0.894,
//           ratio = round(34.81 x 0.894 / sqrt(n)), velocity x 0.967, decayRatio 0.0754, vKick 0.001257), defaults detuning -1,
//           Om 1.3, tpumpreal 1e-7 (FZ422L:55-57), and NO output() at the measurement (FZ422L:1000-1005).
static int program_fz(int argc, char** argv, int variant) {
  const bool quadv = variant == 1, ca5 = variant == 2;
  const char* pname = quadv ? "fz408q" : ca5 ? "fz422l" : "fz408l";
  OptMap opt = {{"Ge", "0.1"}, {"density", "2"}, {"N0", "3500"}, {"detuning", quadv ? "0" : ca5 ? "-1" : "-2.5"}, {"Om", quadv ? "2" : ca5 ? "1.3" : "0.7"},
                {"tpumpreal", variant ? "0.0000001" : "0.0000002"}, {"tstartV0", "15"}, {"tmax", "25"}, {"sampleFreq", "40"}, {"seed", ""},
                {"saveDirectory", quadv ? "data/" : ca5 ? "data422/" : "dataTag408/"}, {"device", "0"}, {"program", pname}, {"quad", quadv ? "1" : "0"}};
  bool quiet = false;
  if (argc < 2 || argv[1][0] == '-') { fprintf(stderr, "usage: mdqt_run --program fz408l|fz408q|fz422l <job> [--Ge x] [--density x] [--N0 n] ...\n"); return 2; }
  const unsigned job = (unsigned)atof(argv[1]);
  if (!parse_opts(argc, argv, 2, opt, &quiet)) return 2;
  const double Ge = atof(opt["Ge"].c_str()), density = atof(opt["density"].c_str()), detuning = atof(opt["detuning"].c_str());
  const double Om = atof(opt["Om"].c_str()), tpumpreal = atof(opt["tpumpreal"].c_str()), tstartV0 = atof(opt["tstartV0"].c_str());
  const double tmax = atof(opt["tmax"].c_str());
  const int N0 = atoi(opt["N0"].c_str()), sampleFreq = atoi(opt["sampleFreq"].c_str());
  const long seed = opt["seed"].empty() ? (long)((unsigned)time(NULL) + job) : atol(opt["seed"].c_str());  // FZ408L:1022
  const double tpump = tpumpreal * 813490 * sqrt(density), tendV0 = tstartV0 + tpump;                      // FZ408L:77-78
  const int ld = N0 + 1000;

  std::string dir = opt["saveDirectory"];
  mkdir(dir.c_str(), 0777);
  char namebuf[256];
  snprintf(namebuf, sizeof(namebuf), "PumpTime%dPumpStart%dDet%dOm%dDensity%dGe%dNumIons%d", as_unsigned_printed(1000000000. * tpumpreal),
           as_unsigned_printed(tstartV0), as_unsigned_printed(100. * fabs(detuning)), as_unsigned_printed(100. * Om),
           as_unsigned_printed(10. * density), as_unsigned_printed(1000 * Ge), N0);  // FZ408L:990
  dir += namebuf;
  mkdir(dir.c_str(), 0777);
  snprintf(namebuf, sizeof(namebuf), "/job%d/", (int)job);
  dir += namebuf;
  mkdir(dir.c_str(), 0777);

  // init() (FZ408L:250-312): the SU family's frozen random start (same draw order), 7-level wavefunctions
  std::vector<double> R((size_t)3 * ld), V((size_t)3 * ld), psi12((size_t)ld * 24), tp(ld);
  double L = 0, lDeb = 0;
  const int N = mdqt_io_init_su(seed, N0, Ge, ld, R.data(), V.data(), psi12.data(), tp.data(), &L, &lDeb);
  if (N < 0) { fprintf(stderr, "mdqt_run: more than N0+1000 ions drawn\n"); return 1; }
  printf("%i\n", N);  // FZ408L:301
  const int S2 = ca5 ? 10 : 14;  // doubles per ion of the wavefunction: 5 or 7 states x (re, im)
  std::vector<double> psi((size_t)N * S2, 0.0);
  for (int i = 0; i < N; i++)
    for (int k = 0; k < 4; k++) psi[(size_t)i * S2 + k] = psi12[(size_t)i * 24 + k];  // S(-1/2), S(+1/2): the only non-zero amplitudes

  mdqt_params p;
  CKP(mdqt_params_su(&p, Ge, density, 4, 19, 0, detuning, 0, Om, 0, N0, N));
  p.scheme = ca5 ? MDQT_SCHEME_CA5 : MDQT_SCHEME_SR7; p.quad = atoi(opt["quad"].c_str());
  p.substeps_per_md = (int)round(34.81 / sqrt(density));  // FZ408L:73 rounds where SU takes the ceiling
  if (ca5) {                                              // FZ422L:66-74, 116-117
    p.g2E = 174.07 * .894 / sqrt(density);
    p.substeps_per_md = (int)round(34.81 * .894 / sqrt(density));
    p.pv2qv = 1.1821 * pow(density, 1. / 6) * .967;
    p.dR = 0.0754;
    p.vKick = 0.001257 / p.pv2qv;
  }
  p.dtq = 0.002 / p.substeps_per_md;
  p.traj0 = (int)job; p.seed = (uint64_t)seed; p.device = atoi(opt["device"].c_str());
  mdqt_handle* h = NULL;
  CKP(mdqt_create(&p, &h));
  CKP(mdqt_upload_state(h, R.data(), V.data(), psi.data(), NULL, ld));
  CKP(mdqt_set_time(h, 0.0, 0));
  FzOut o;
  o.h = h; o.dir = dir; o.N = N; o.ld = ld; o.counter = 0; o.V = V; o.spin.assign(N, 0);
  CKP(mdqt_epot(h, &o.Epot0));  // Epotential(); Epot0 = Epot (FZ408L:309-310)

  const int ratio = p.substeps_per_md;
  const double dtq = p.dtq;
  int c0 = -1, tsc = ratio, recorded = 0;
  double t = 0.0, vaf = 0.0;
  long pend_q = 0, pend_t = 0, iters = 0;
  auto flush = [&]() {  // consecutive pump sweeps between two events are one launch; t advances by the reference's repeated addition
    if (pend_q) { CKP(mdqt_qsteps(h, (int)pend_q)); pend_q = 0; }
    if (pend_t) { CKP(mdqt_advance_time(h, (int)pend_t)); pend_t = 0; }
  };
  const char* acfile = quadv ? "vSquareAutoCorr.dat" : "VAF.dat";  // printLongKin (FZ408Q:969-979) / printVAF (FZ408L:963-973)
  auto wall0 = std::chrono::steady_clock::now();
  while (t <= tmax + 0.0009) {  // FZ408L:1040
    if (!recorded && t >= tendV0) {
      flush();
      int32_t nup = 0;
      CKP(mdqt_tag_particles(h, o.spin.data(), &nup));  // measureSpinUps()
      recorded = 1;
      if (!ca5) fz_output(o, t, c0);                      // FZ408L:1045; the 422 nm program has no output() here (FZ422L:1000-1005)
      CKP(quadv ? mdqt_vsq_autocorr(h, 1, &vaf) : mdqt_vaf(h, 1, &vaf));  // Zfunc(0)
      fz_print_vaf(o, t, vaf, acfile);
    }
    if ((c0 + 1) % sampleFreq == 0 && tsc == 1 && recorded) {
      flush();
      fz_output(o, t, c0);
      CKP(quadv ? mdqt_vsq_autocorr(h, 0, &vaf) : mdqt_vaf(h, 0, &vaf));  // Zfunc(1)
      fz_print_vaf(o, t, vaf, acfile);
    }
    if (tsc == ratio) {
      flush();                                            // step() tests the clock (2nd-order start while t <= 0, FZ408L:321)
      CKP(mdqt_leapfrog_step(h, dtq * ratio));            // step(): dt = quantumTimestep * ratio (FZ408L:382)
      c0++; tsc = 0;
    }
    if (t < tendV0 && t > tstartV0) {                     // qstep() (which also does t += dtQuant, FZ408L:597)
      if (pend_t && !pend_q) flush();
      pend_q++;
    }
    pend_t++;
    t += dtq;
    tsc++;
    iters++;
  }
  flush();
  // writeConditions(c0) (FZ408L:667-707)
  CKP(mdqt_download_state(h, R.data(), V.data(), NULL, NULL, ld));
  {
    char name[64];
    snprintf(name, sizeof(name), "ions_timestep%06d.dat", c0);
    FILE* fa = open_in(dir, name, "w");
    fprintf(fa, "%i\t%i", N, o.counter);
    fclose(fa);
    snprintf(name, sizeof(name), "spinUpIonsList_timestep%06d.dat", c0);
    fa = open_in(dir, name, "w");
    for (int i = 0; i < N; i++) fprintf(fa, "%i\n", o.spin[i]);
    fclose(fa);
    snprintf(name, sizeof(name), "conditions_timestep%06d.dat", c0);
    fa = open_in(dir, name, "w");
    for (int i = 0; i < N; i++)
      fprintf(fa, "%lg\t%lg\t%lg\t%lg\t%lg\t%lg\t\n", R[i], R[(size_t)ld + i], R[(size_t)2 * ld + i], V[i], V[(size_t)ld + i], V[(size_t)2 * ld + i]);
    fclose(fa);
  }
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
  if (!quiet)
    fprintf(stderr, "mdqt_run: program %s, job %u, N=%d, t=%.6f, c0=%d: %ld loop iterations, %u outputs in %.3f s; files in %s\n", pname, job, N, t, c0,
            iters, o.counter, wall, dir.c_str());
  mdqt_destroy(h);
  return 0;
}
int mdqt_program_fz408l(int argc, char** argv) { return program_fz(argc, argv, 0); }
int mdqt_program_fz408q(int argc, char** argv) { return program_fz(argc, argv, 1); }
int mdqt_program_fz422l(int argc, char** argv) { return program_fz(argc, argv, 2); }

// ---- laserCoolNoPlasmaThreeState.cpp --------------------------------------------------------------------------------------------
// main() (TS:352-409): N0 non-interacting ions with Maxwellian velocities (std::mt19937 + normal_distribution, sigma = 1.0508
// sqrt(T[K]), TS:83, 115-131) in the ground state of a J = 0 -> J = 1 transition lit by two counter-propagating sigma+/sigma- beams;
// the loop is { t += dt; every sampleFreq-th iteration output(); qstep(); c0++ } until t > tmax, and output() appends
// "t <tab> <v_x^2>/2" to energies.dat (TS:296-322). No plasma forces at all: the whole run is the 3-level substep kernel, sampleFreq
// sweeps fused per launch. Directory: <save>/Om%d/Det%dNumIons%dInitialTemp%duK/job%d/ (TS:371-382; the (unsigned) cast of a
// negative detuning is printed as the reference prints it on x86-64).
int mdqt_program_ts(int argc, char** argv) {
  OptMap opt = {{"N0", "1000"}, {"detuning", "-0.5"}, {"Om", "0.5"}, {"tmax", "45000"}, {"sampleFreq", "1000"}, {"temperature", "0.01"},
                {"seed", ""}, {"saveDirectory", "dataLaserCoolTestDoppShift/"}, {"device", "0"}, {"program", "ts"}};
  bool quiet = false;
  if (argc < 2 || argv[1][0] == '-') { fprintf(stderr, "usage: mdqt_run --program ts <job> [--N0 n] [--detuning x] [--Om x] [--tmax x] ...\n"); return 2; }
  const unsigned job = (unsigned)atof(argv[1]);
  if (!parse_opts(argc, argv, 2, opt, &quiet)) return 2;
  const int N0 = atoi(opt["N0"].c_str()), sampleFreq = atoi(opt["sampleFreq"].c_str());
  const double detuning = atof(opt["detuning"].c_str()), Om = atof(opt["Om"].c_str()), tmax = atof(opt["tmax"].c_str());
  const double temperature = atof(opt["temperature"].c_str());
  const unsigned seed = opt["seed"].empty() ? (unsigned)time(NULL) + job : (unsigned)atol(opt["seed"].c_str());  // TS:388
  if (N0 < 1 || sampleFreq < 1) { fprintf(stderr, "mdqt_run: N0 and sampleFreq must be positive\n"); return 2; }

  std::string dir = opt["saveDirectory"];
  mkdir(dir.c_str(), 0777);
  char namebuf[256];
  snprintf(namebuf, sizeof(namebuf), "Om%d/", as_unsigned_printed(Om * 100));
  dir += namebuf;
  mkdir(dir.c_str(), 0777);
  snprintf(namebuf, sizeof(namebuf), "Det%dNumIons%dInitialTemp%duK", (int)(unsigned)(long long)(detuning * 100), N0, as_unsigned_printed(temperature * 1000000));
  dir += namebuf;
  mkdir(dir.c_str(), 0777);
  snprintf(namebuf, sizeof(namebuf), "/job%d/", (int)job);
  dir += namebuf;
  mkdir(dir.c_str(), 0777);

  // init() (TS:115-131)
  std::mt19937 rng(seed);
  std::normal_distribution<double> velocityDistribution(0, 1.0508 * sqrt(temperature));
  std::vector<double> V((size_t)3 * N0), R((size_t)3 * N0, 0.0), psi((size_t)N0 * 6, 0.0), tp(N0, 0.0);
  for (int i = 0; i < N0; i++) {
    V[i] = velocityDistribution(rng); V[(size_t)N0 + i] = velocityDistribution(rng); V[(size_t)2 * N0 + i] = velocityDistribution(rng);
    psi[(size_t)i * 6] = 1.0;
  }
  mdqt_params p;
  CKP(mdqt_params_ts(&p, N0, detuning, Om));
  p.traj0 = (int)job; p.seed = seed; p.device = atoi(opt["device"].c_str());
  mdqt_handle* h = NULL;
  CKP(mdqt_create(&p, &h));
  CKP(mdqt_upload_state(h, R.data(), V.data(), psi.data(), tp.data(), N0));
  CKP(mdqt_set_time(h, 0.0, 0));
  const double dt = 0.01;  // TS:390
  // the loop's schedule first (the reference's repeated addition t += dt decides where it ends), then the launches: every output()
  // is one reduction kernel appending sum v_x^2 to a device log -- nothing synchronises until the log is read back at the end
  std::vector<double> tout;
  std::vector<long> sweeps_before;  // qstep() sweeps between the previous output() and this one
  long c0 = 0, pend = 0;
  {
    double t = 0.0;
    while (t <= tmax) {  // TS:392
      t += dt;
      if ((c0 + 1) % sampleFreq == 0) { tout.push_back(t); sweeps_before.push_back(pend); pend = 0; }  // output() (TS:296-322)
      pend++;  // qstep()
      c0++;
    }
  }
  const long outputs = (long)tout.size();
  if (outputs > (1 << 22)) { fprintf(stderr, "mdqt_run: more than 2^22 outputs; raise --sampleFreq\n"); return 2; }
  auto wall0 = std::chrono::steady_clock::now();
  if (outputs) CKP(mdqt_moments_begin(h, (int)outputs));
  for (long k = 0; k < outputs; k++) {
    if (sweeps_before[k]) CKP(mdqt_qsteps(h, (int)sweeps_before[k]));
    CKP(mdqt_moments_record(h, (int)k));
  }
  if (pend) CKP(mdqt_qsteps(h, (int)pend));
  if (outputs) {
    std::vector<double> rec((size_t)outputs * 23);
    CKP(mdqt_moments_download(h, rec.data(), (int)outputs));
    FILE* fe = open_in(dir, "energies.dat", "a");
    for (long k = 0; k < outputs; k++) fprintf(fe, "%lg\t%lg\n", tout[k], 0.5 * rec[(size_t)k * 23] / (double)N0);  // TS:318: t, EkinX
    fclose(fe);
  }
  CKP(mdqt_sync(h));
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
  if (!quiet)
    fprintf(stderr, "mdqt_run: program ts, job %u, N0=%d: %ld sweeps, %ld outputs in %.3f s; files in %s\n", job, N0, c0, outputs, wall, dir.c_str());
  mdqt_destroy(h);
  return 0;
}

// ---- MonteCarloFollowedByQTTagging408Linear.cpp ---------------------------------------------------------------------------------
// main() (MC408L:1140-1254) without its Monte-Carlo stage: init() (lattice, Maxwellian velocities from std::mt19937, random S-manifold
// wavefunctions from the UNSEEDED drand48 stream the reference uses, Q14), collisional MD, the pump stage
// { ratio x qstep(); MDStep(k) } x pumpMDTimeSteps, tagParticles() (projective spin measurement), then the collisionless
// recording stage -- taggedMoments.dat and vel_distX_timestep%06d.dat every step (MC408L:1069-1137), g(r) every 100 steps,
// temperature.dat -- and the four autocorrelation files.
// The same main() serves MonteCarloFollowedByQTTagging422Linear.cpp (MC422L:1100-1222; `ca5`): the 5-level 422 nm pump scheme with
// its own unit conversions (mdqt_params_md, MC422L:113-122) and defaults (tpumpreal 5e-8, detuning -1, Om 1.3: MC422L:85-87), the
// same init() draws (MC422L:196-238) into a 5-state wavefunction, and a "Date%m%d%y" suffix on the run directory (MC422L:1127-1134).
static int program_mc_tagging(int argc, char** argv, bool ca5) {
  OptMap opt = {{"N", "4096"}, {"Gamma", "3"}, {"kappa", "0.5"}, {"density", "2"}, {"timeStep", "0.005"}, {"collisionFreq", "0.25"},
                {"preSteps", "200"}, {"recordSteps", "1500"}, {"pumpSteps", "-1"}, {"tpumpreal", ca5 ? "0.00000005" : "0.0000002"},
                {"detuning", ca5 ? "-1" : "-2.5"}, {"Om", ca5 ? "1.3" : "0.7"}, {"quad", "0"}, {"pairPairStep", "0.05"}, {"seed", ""},
                {"saveDirectory", "data/"}, {"device", "0"}, {"program", ca5 ? "mc422l" : "mc408l"}, {"dateSuffix", ca5 ? "1" : "0"}};
  bool quiet = false;
  if (argc < 2 || argv[1][0] == '-') { fprintf(stderr, "usage: mdqt_run --program mc408l|mc422l <job> [--N n] [--density x] [--tpumpreal x] ...\n"); return 2; }
  const unsigned job = (unsigned)atof(argv[1]);
  if (!parse_opts(argc, argv, 2, opt, &quiet)) return 2;
  const int N = atoi(opt["N"].c_str());
  const double Gamma = atof(opt["Gamma"].c_str()), kappa = atof(opt["kappa"].c_str()), n = atof(opt["density"].c_str());
  const double timeStep = atof(opt["timeStep"].c_str()), collFreq = atof(opt["collisionFreq"].c_str());
  const double tpumpreal = atof(opt["tpumpreal"].c_str()), detuning = atof(opt["detuning"].c_str()), Om = atof(opt["Om"].c_str());
  const int preSteps = atoi(opt["preSteps"].c_str()), recSteps = atoi(opt["recordSteps"].c_str());
  int pumpSteps = atoi(opt["pumpSteps"].c_str());
  if (pumpSteps < 0) pumpSteps = (int)round(tpumpreal * 813490 * sqrt(n) / timeStep);  // MC408L:119-120
  const double pairPairStep = atof(opt["pairPairStep"].c_str());
  const unsigned seed = opt["seed"].empty() ? (unsigned)time(NULL) + job : (unsigned)atol(opt["seed"].c_str());
  if (recSteps > 5000) { fprintf(stderr, "mdqt_run: recordSteps must be <= 5000\n"); return 2; }

  std::string dir = opt["saveDirectory"];
  mkdir(dir.c_str(), 0777);
  char namebuf[256];
  snprintf(namebuf, sizeof(namebuf), "Gamma%dKappa%dNumIons%dPumpTime%dDet%dOm%dDensity%d", as_unsigned_printed(Gamma * 100),
           as_unsigned_printed(kappa * 100), N, as_unsigned_printed(1000000000. * tpumpreal), as_unsigned_printed(100. * fabs(detuning)),
           as_unsigned_printed(100. * Om), as_unsigned_printed(10. * n));  // MC408L:1153
  dir += namebuf;
  if (atoi(opt["dateSuffix"].c_str())) {  // MC422L:1127-1134 (--dateSuffix 0 for a reproducible path)
    time_t rawtime;
    time(&rawtime);
    char st[80];
    strftime(st, sizeof(st), "Date%m%d%y", localtime(&rawtime));
    dir += st;
  }
  mkdir(dir.c_str(), 0777);
  snprintf(namebuf, sizeof(namebuf), "/job%d/", (int)job);
  dir += namebuf;
  mkdir(dir.c_str(), 0777);

  mdqt_params p;
  CKP(mdqt_params_md(&p, ca5 ? MDQT_SCHEME_CA5 : MDQT_SCHEME_SR7, N, kappa, n, timeStep, detuning, Om, atoi(opt["quad"].c_str())));
  const int S2 = ca5 ? 10 : 14;  // doubles per ion of the wavefunction: 5 or 7 states x (re, im)
  p.traj0 = (int)job; p.seed = seed; p.device = atoi(opt["device"].c_str());
  const double L = p.L;
  // init() (MC408L:196-250): per lattice site three normal draws (mt19937), then rand1..rand4 from drand48 in its default state
  std::mt19937 rng(seed);
  std::normal_distribution<double> velocityDistribution(0, sqrt(1 / Gamma));
  unsigned short xs[3] = {0x330E, 0xABCD, 0x1234};  // the initial state of an unseeded drand48 (the reference never calls srand48, Q14)
  std::vector<double> R((size_t)3 * N, 0.0), V((size_t)3 * N, 0.0), psi((size_t)N * S2, 0.0);
  {
    int N0 = 0;
    const int side = (int)round(pow(N, 1. / 3));
    for (int i = 0; i < side; i++)
      for (int j = 0; j < side; j++)
        for (int k = 0; k < side; k++) {
          if (N0 >= N) break;
          R[N0] = i * L / pow(N, 1 / 3.) + 0.5; R[(size_t)N + N0] = j * L / pow(N, 1 / 3.) + 0.5; R[(size_t)2 * N + N0] = k * L / pow(N, 1 / 3.) + 0.5;
          V[N0] = velocityDistribution(rng); V[(size_t)N + N0] = velocityDistribution(rng); V[(size_t)2 * N + N0] = velocityDistribution(rng);
          const double rand1 = erand48(xs), rand2 = erand48(xs), rand3 = erand48(xs);
          const double sign = rand3 < 0.5 ? -1 : 1;
          const double rand4 = erand48(xs);
          const double sign2 = rand4 < 0.5 ? -1 : 1;
          double* w = &psi[(size_t)N0 * S2];  // sqrt(rand1) |1> + (sign2 sqrt(..) + i sign sqrt(..)) |2>  (MC408L:232-236, MC422L:232-236)
          w[0] = sqrt(rand1); w[2] = sign2 * sqrt(1 - rand1) * sqrt(rand2); w[3] = sign * sqrt(1 - rand1) * sqrt(1 - rand2);
          N0++;
        }
    if (N0 != N) { fprintf(stderr, "mdqt_run: N must be a cube (the reference's lattice init, MC408L:79)\n"); return 2; }
  }
  mdqt_handle* h = NULL;
  CKP(mdqt_create(&p, &h));
  CKP(mdqt_upload_state(h, R.data(), V.data(), psi.data(), NULL, N));
  const double sigma_v = sqrt(1 / Gamma), rmax = L / 2;
  auto wall0 = std::chrono::steady_clock::now();
  if (preSteps > 0) CKP(mdqt_vv_steps(h, preSteps, 0, timeStep, collFreq, sigma_v, 0, 0.0));           // step 4 (MC408L:1211-1219)
  if (!quiet) printf("pumpMDTimeSteps=%d\nquantumStepsPerMD=%d\n", pumpSteps, p.substeps_per_md);        // MC408L:1225-1226
  if (pumpSteps > 0) CKP(mdqt_vv_steps(h, pumpSteps, p.substeps_per_md, timeStep, 0.0, sigma_v, 0, 0.0));  // step 5 (MC408L:1227-1232)
  std::vector<int32_t> spin(N);
  int32_t nup = 0;
  CKP(mdqt_tag_particles(h, spin.data(), &nup));                                                         // tagParticles()
  if (recSteps > 0) {
    std::vector<uint8_t> tags(N);
    for (int i = 0; i < N; i++) tags[i] = spin[i] ? 1 : 0;
    CKP(mdqt_set_tags(h, tags.data()));
    CKP(mdqt_moments_begin(h, recSteps));
    CKP(mdqt_vstore_begin(h, recSteps));
    std::vector<double> pv(4001);
    for (int k = 0; k < recSteps; k++) {  // step 6 (MC408L:1235-1244)
      CKP(mdqt_moments_record(h, k));     // recordTaggedParticleMoments(k): the moments; recordTemperature()
      CKP(mdqt_vel_dist_tagged(h, pv.data()));
      char name[64];
      snprintf(name, sizeof(name), "vel_distX_timestep%06d.dat", k);
      FILE* fa = open_in(dir, name, "w");
      for (int j = 0; j < 4001; j++) fprintf(fa, "%lg\t%lg\n", (double)(j - 2000) * 0.0025, pv[j]);      // MC408L:1131-1134
      fclose(fa);
      if (k % 100 == 0) { if (!quiet) printf("%d\n", k); write_gr(h, dir, k, pairPairStep, rmax); }
      CKP(mdqt_vv_step(h, timeStep, 0.0, sigma_v, 0, 0.0));
      CKP(mdqt_vstore_record(h, k));
    }
    std::vector<double> rec((size_t)recSteps * 23);
    CKP(mdqt_moments_download(h, rec.data(), recSteps));
    FILE* fm = open_in(dir, "taggedMoments.dat", "a");
    FILE* ft = open_in(dir, "temperature.dat", "a");
    for (int k = 0; k < recSteps; k++) {
      const double* r = &rec[(size_t)k * 23];
      const double cnt = r[3];
      fprintf(fm, "%lg\t%lg\t%lg\t%lg\t%lg\n", k * timeStep, r[4] / cnt, r[5] / cnt, r[6] / cnt, r[7] / cnt);  // MC408L:1106-1115
      fprintf(ft, "%lg\n", (r[0] + r[1] + r[2]) / (3.0 * N));
    }
    fclose(fm); fclose(ft);
    std::vector<double> ac[4];
    for (auto& a : ac) a.resize(recSteps);
    CKP(mdqt_autocorrelations(h, Gamma, ac[0].data(), ac[1].data(), ac[2].data(), ac[3].data()));  // step 7
    static const char* acn[4] = {"VAF.dat", "longViscAutoCorr.dat", "vCubeAutoCorr.dat", "vFourthAutoCorr.dat"};
    for (int s = 0; s < 4; s++) {
      FILE* fa = open_in(dir, acn[s], "w");
      for (int tD = 0; tD < recSteps; tD++) fprintf(fa, "%lg\t%lg\n", tD * timeStep, ac[s][tD]);
      fclose(fa);
    }
  }
  CKP(mdqt_sync(h));
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
  if (!quiet)
    fprintf(stderr, "mdqt_run: program %s, job %u, N=%d: %d collisional + %d pump (x %d qstep) + %d recorded MD steps, %d of %d ions tagged, %.3f s; files in %s\n",
            ca5 ? "mc422l" : "mc408l", job, N, preSteps, pumpSteps, p.substeps_per_md, recSteps, (int)nup, N, wall, dir.c_str());
  mdqt_destroy(h);
  return 0;
}
int mdqt_program_mc408l(int argc, char** argv) { return program_mc_tagging(argc, argv, false); }
int mdqt_program_mc422l(int argc, char** argv) { return program_mc_tagging(argc, argv, true); }
