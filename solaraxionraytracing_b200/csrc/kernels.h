// kernels.h — launcher prototypes shared by the kernel TUs and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>

#include "../../include/sart.h"
#include "device_params.h"
#include "fast_params.h"

namespace sart {

// Run-wide switches of a throughput launch, decided on the host and compiled into the kernel variants as template
// parameters.
struct LaunchVariant {
  bool wolter;    // Wolter-I optic (XMM, ABRIXAS) instead of two cones
  bool plain;     // solar source, vacuum stage, unturned telescope, no flags, a reflectivity table
  bool alias;     // alias sampler (solar source only: the X-ray test source draws no table values)
  bool margins;   // a re-trace queue is attached: the FP32 kernels test their decision margins
};
inline LaunchVariant launch_variant(const fast::FastParams& P, const fast::FastTables& T) {
  LaunchVariant v;
  v.wolter = P.telKind == SART_TK_XMM || P.telKind == SART_TK_ABRIXAS;
  v.plain = !P.testXray && P.stage == SART_SK_VACUUM && !P.rotated && P.flags == 0 && P.reflKind != SART_RK_EFFECTIVE_AREA;
  v.alias = T.sampler == SART_SAMPLER_ALIAS && !P.testXray && T.radiusAlias && T.energyAlias;
  v.margins = T.rq.cap != 0u;
  return v;
}

// The arrays of a per-ray record struct: f(a.field, b.field) for every pointer field of a pair of sart_ray_out_t (const or
// not) in declaration order. The only place that lists the fields; an element is sizeof(*field) bytes.
template <class A, class B, class F>
inline void ray_out_fields(A& a, B& b, F&& f) {
  f(a.x, b.x); f(a.y, b.y); f(a.w, b.w); f(a.code, b.code); f(a.shell, b.shell); f(a.energy, b.energy);
  f(a.reflect, b.reflect); f(a.transMagnet, b.transMagnet); f(a.yaw, b.yaw); f(a.alpha1, b.alpha1); f(a.alpha2, b.alpha2);
  f(a.pathCB, b.pathCB); f(a.r, b.r); f(a.deviationDet, b.deviationDet); f(a.transProbArgon, b.transProbArgon);
}
// The same for a pair of sart_passed_out_t.
template <class A, class B, class F>
inline void passed_out_fields(A& a, B& b, F&& f) {
  f(a.ray, b.ray); f(a.x, b.x); f(a.y, b.y); f(a.w, b.w); f(a.shell, b.shell); f(a.energy, b.energy); f(a.r, b.r);
  f(a.reflect, b.reflect); f(a.transMagnet, b.transMagnet); f(a.yaw, b.yaw); f(a.alpha1, b.alpha1); f(a.alpha2, b.alpha2);
  f(a.pathCB, b.pathCB); f(a.deviationDet, b.deviationDet); f(a.transProbArgon, b.transProbArgon);
}

// Grid of a grid-stride launch over n rays: one thread per ray, at most perSM blocks on each of smCount SMs. perSM = 0: one
// resident wave, i.e. the occupancy of `kern` with `smem` bytes of dynamic shared memory (at least one block per SM).
template <class K>
inline cudaError_t grid_size(K kern, int block, size_t smem, uint64_t n, int smCount, int perSM, unsigned* grid) {
  if (perSM == 0) {
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kern, block, smem);
    if (e != cudaSuccess) return e;
    if (perSM < 1) perSM = 1;
  }
  const uint64_t want = (n + block - 1) / block, cap = uint64_t(smCount) * perSM;
  *grid = unsigned(want < cap ? want : cap);
  return cudaSuccess;
}

// ---- FP64 "exact" pipeline (kernels_exact.cu)
cudaError_t launch_presampled_exact(const Params& P, const Tables& T, double mAxion, size_t n, const double* origin,
                                    const double* exitxy, const double* energy, const sart_ray_out_t& out,
                                    cudaStream_t s);
cudaError_t launch_mc_rays_exact(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n,
                                 uint64_t seed, const sart_ray_out_t& out, cudaStream_t s, const uint32_t* words = nullptr,
                                 int32_t* emit = nullptr);
cudaError_t launch_mc_image_exact(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                  uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                  sart_counters_t* counters, int smCount, cudaStream_t s, const BandImages& bands = {},
                                  const QuantityHists& qh = {}, const MassRows& rows = {});
// re-trace of the uncertain rays of an FP32 launch (fast_params.h: RetraceQueue) by the exact pipeline
cudaError_t launch_retrace_mc_image(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                    uint64_t seed, const fast::RetraceQueue& q, double* image, double* imageW2,
                                    sart_counters_t* counters, int smCount, cudaStream_t s, const BandImages& bands = {},
                                    const QuantityHists& qh = {}, const MassRows& rows = {});
cudaError_t launch_retrace_mc_rays(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n, uint64_t seed,
                                   const uint32_t* words, const fast::RetraceQueue& q, const sart_ray_out_t& out, int smCount,
                                   cudaStream_t s);
cudaError_t launch_retrace_mc_passed(const Params& P, const Tables& T, double mAxion, uint64_t first, uint64_t seed,
                                     const fast::RetraceQueue& q, const sart_passed_out_t& o, unsigned int* count, unsigned int cap,
                                     uint32_t idBase, sart_counters_t* counters, int smCount, cudaStream_t s);
cudaError_t launch_mc_passed_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                 uint64_t first, uint64_t nRays, uint64_t seed, const sart_passed_out_t& o, unsigned int* count,
                                 unsigned int cap, uint32_t idBase, sart_counters_t* counters, int smCount, cudaStream_t s);
cudaError_t launch_retrace_presampled(const Params& P, const Tables& T, double mAxion, size_t n, const double* origin,
                                      const double* exitxy, const double* energy, const fast::RetraceQueue& q,
                                      const sart_ray_out_t& out, int smCount, cudaStream_t s);
cudaError_t launch_build_cdfs(int nR, int nE, const double* radii, const double* energies, const double* emRates,
                              double* rowTotals, double* cdfs, double* radiusCDF, cudaStream_t s);

// rows: the per-mass radial histograms and band images of a mass scan (device_params.h: MassRows; off by default), the
// handle's rows for the exact launchers, mass-minor accumulators for the mass-scan launchers, which then run the kernel
// variants that fill them.
// ---- "fast" pipeline (kernels_fast.cu)
// bands: the band images (device_params.h: BandImages; w == nullptr: off), in modes 1 and 2 their replicas, which
// launch_fold_replicas adds up after the launch; with them on, the launchers run the kernel variants that fill them.
// qh: the quantity histograms (device_params.h: QuantityHists; w == nullptr: off), whose replicas rw / rw2 the caller folds
// after the launch as well; with them on, the launchers run the kernel variants that fill them and the band images.
cudaError_t launch_mc_image_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                 uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                 sart_counters_t* counters, int smCount, bool compact, cudaStream_t s,
                                 const BandImages& bands = {}, const QuantityHists& qh = {});

cudaError_t launch_mc_image_fast_masses(const fast::FastParams& P, const fast::FastTables& T, int nMasses,
                                        const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                        double* image, double* imageW2, sart_counters_t* counters, int smCount,
                                        cudaStream_t s, const MassRows& rows = {});
cudaError_t launch_mc_rays_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                uint64_t nRays, uint64_t seed, const sart_ray_out_t& o, int smCount, cudaStream_t s);
cudaError_t launch_emission_rates(int nR, int nE, const double* dTemp, const double* dRho, const double* dFrac,
                                  const double* dEnergies, unsigned processes, double gae, double gagamma, double ganuclei,
                                  void* dState /* 80 B per radius */, double* dEmRates, cudaStream_t s);
// ---- single-precision pipeline (kernels_f32.cu)
cudaError_t launch_mc_image_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                uint64_t first, uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                sart_counters_t* counters, int smCount, bool compact, cudaStream_t s,
                                const BandImages& bands = {}, const QuantityHists& qh = {});
cudaError_t launch_mc_image_f32_masses(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T,
                                       int nMasses, const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                       double* acc, double* accW2, sart_counters_t* counters, int smCount, cudaStream_t s,
                                       const MassRows& rows = {});
cudaError_t launch_presampled_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                  size_t n, const double* origin, const double* exitxy, const double* energy,
                                  const sart_ray_out_t& o, int smCount, cudaStream_t s);
cudaError_t launch_mc_rays_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                               uint64_t first, uint64_t nRays, uint64_t seed, const sart_ray_out_t& o, int smCount,
                               cudaStream_t s, const uint32_t* words = nullptr, bool lateEnergy = false,
                               int32_t* emit = nullptr);
cudaError_t launch_fold_replicas(double* rep, double* rep2, int nRep, size_t stride, size_t plane, double* image,
                                 double* imageW2, cudaStream_t s);
cudaError_t launch_fold_spectra(const Spectra& rep, int nE1, const Spectra& dst, cudaStream_t s);
cudaError_t launch_fold_mass_acc(double* acc, double* acc2, int nMasses, size_t plane, double* image, double* imageW2,
                                 cudaStream_t s);
cudaError_t launch_fold_mass_spectra(const Spectra& acc, int nMasses, int nE1, const Spectra& dst, cudaStream_t s);
cudaError_t launch_fold_mass_hist(double* accW, unsigned int* accN, int nMasses, int bins, double* dstW,
                                  unsigned long long* dstN, cudaStream_t s);
cudaError_t launch_heatmap(int rows, int cols, double start_x, double step_x, double start_y, double step_y, size_t n,
                           const double* X, const double* Y, const double* W, double norm, double* result,
                           unsigned long long* nBad, cudaStream_t s);

}  // namespace sart
