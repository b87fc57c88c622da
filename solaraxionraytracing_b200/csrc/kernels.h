// kernels.h — launcher prototypes shared by the kernel TUs and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>

#include "../../include/sart.h"
#include "device_params.h"
#include "fast_params.h"

namespace sart {

// ---- FP64 "exact" pipeline (kernels_exact.cu)
cudaError_t launch_presampled_exact(const Params& P, const Tables& T, double mAxion, size_t n, const double* origin,
                                    const double* exitxy, const double* energy, const sart_ray_out_t& out,
                                    cudaStream_t s);
cudaError_t launch_mc_rays_exact(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n,
                                 uint64_t seed, const sart_ray_out_t& out, cudaStream_t s, const uint32_t* words = nullptr,
                                 int32_t* emit = nullptr);
cudaError_t launch_mc_image_exact(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                  uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                  sart_counters_t* counters, int smCount, cudaStream_t s);
// re-trace of the uncertain rays of an FP32 launch (fast_params.h: RetraceQueue) by the exact pipeline
cudaError_t launch_retrace_mc_image(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                    uint64_t seed, const fast::RetraceQueue& q, double* image, double* imageW2,
                                    sart_counters_t* counters, int smCount, cudaStream_t s);
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

// ---- "fast" pipeline (kernels_fast.cu)
cudaError_t launch_mc_image_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                 uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                 sart_counters_t* counters, int smCount, bool compact, cudaStream_t s);

cudaError_t launch_mc_image_fast_masses(const fast::FastParams& P, const fast::FastTables& T, int nMasses,
                                        const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                        double* image, double* imageW2, sart_counters_t* counters, int smCount,
                                        cudaStream_t s);
cudaError_t launch_mc_rays_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                uint64_t nRays, uint64_t seed, const sart_ray_out_t& o, int smCount, cudaStream_t s);
cudaError_t launch_emission_rates(int nR, int nE, const double* dTemp, const double* dRho, const double* dFrac,
                                  const double* dEnergies, unsigned processes, double gae, double gagamma, double ganuclei,
                                  void* dState /* 80 B per radius */, double* dEmRates, cudaStream_t s);
// ---- single-precision pipeline (kernels_f32.cu)
cudaError_t launch_mc_image_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                uint64_t first, uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                sart_counters_t* counters, int smCount, bool compact, cudaStream_t s);
cudaError_t launch_mc_image_f32_masses(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T,
                                       int nMasses, const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                       double* acc, double* accW2, sart_counters_t* counters, int smCount, cudaStream_t s);
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
cudaError_t launch_heatmap(int rows, int cols, double start_x, double step_x, double start_y, double step_y, size_t n,
                           const double* X, const double* Y, const double* W, double norm, double* result,
                           unsigned long long* nBad, cudaStream_t s);

}  // namespace sart
