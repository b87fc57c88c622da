// comm.cu — the one collective of the path: the sum of the detector images and counters of all GPUs.
//
// Rays shard over GPUs by global ray index (Philox counter), with no exchange while tracing (SURVEY.md §8e); what has
// to be merged afterwards is additive: image [M][256][256], the sum-of-squares image and the counters. The handle keeps
// image and sum-of-squares image in ONE allocation followed by a small f64 area; sart_allreduce writes the counters into
// that area as f64 (exact below 2^53) and issues ONE ncclAllReduce(sum, f64) over the whole block into a separate
// "merged" block, so a rank's own accumulators stay untouched (no reset between steps) and the call can be repeated.
// sart_allreduce_outputs does the same for the optional accumulators (radial histogram, spectra, per-mass spectra, band
// images): the ranks first agree on which are on and their shapes, then sum them into merged copies, counts as u64 and sums
// as f64.
//
// NCCL is resolved with dlopen at first use: libsart.so has no link-time dependency on it, a process that already
// loaded NCCL (PyTorch) shares that copy, and a host without NCCL can use everything else.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <cstring>
#include <vector>

#include "host_cuda.h"
#include "kernels.h"
#include "sart_internal.h"

namespace sart {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi* nccl() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (api.lib) break;
    }
    if (api.lib) {
#define SART_SYM(field, sym) api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.lib, sym))
      SART_SYM(GetUniqueId, "ncclGetUniqueId");
      SART_SYM(CommInitRank, "ncclCommInitRank");
      SART_SYM(CommInitAll, "ncclCommInitAll");
      SART_SYM(AllReduce, "ncclAllReduce");
      SART_SYM(GroupStart, "ncclGroupStart");
      SART_SYM(GroupEnd, "ncclGroupEnd");
      SART_SYM(CommDestroy, "ncclCommDestroy");
      SART_SYM(GetErrorString, "ncclGetErrorString");
#undef SART_SYM
      if (!api.GetUniqueId || !api.CommInitRank || !api.CommInitAll || !api.AllReduce || !api.GroupStart || !api.GroupEnd ||
          !api.CommDestroy || !api.GetErrorString) {
        dlclose(api.lib);
        api.lib = nullptr;
      }
    }
  }
  return api.lib ? &api : nullptr;
}

static int nccl_fail(ncclResult_t r, const char* what) {
  NcclApi* n = nccl();
  return fail(SART_ERR_CUDA, "%s: %s", what, n ? n->GetErrorString(r) : "NCCL unavailable");
}
#define SART_NCCL(call)                                      \
  do {                                                       \
    ncclResult_t r__ = (call);                               \
    if (r__ != ncclSuccess) return nccl_fail(r__, #call);    \
  } while (0)

// counters -> f64 words behind the two images (pack), one thread per (mass, word)
__global__ void k_pack_counters(const sart_counters_t* __restrict__ c, int nMasses, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nMasses * kCounterWords) return;
  const int m = i / kCounterWords, w = i % kCounterWords;
  const unsigned long long* raw = reinterpret_cast<const unsigned long long*>(c + m);
  constexpr int nInt = int(offsetof(sart_counters_t, sum_w) / 8);
  out[i] = w < nInt ? double(raw[w]) : reinterpret_cast<const double*>(raw)[w];
}

// sart_allreduce_outputs: what a handle has on, in the words every rank must agree on, then an error word. All ranks send
// [d, -d] through one ncclMax, so each learns the largest and (negated) smallest value of every word. Words 0 .. kAccums - 1
// are the bins of each accumulator (0: off), then the bits of r_max, the number of masses and the bits of the
// SART_MAX_BANDS + 1 band edges (0 beyond the last edge; edges are >= 0, so their bits are non-negative int64 words), then
// per quantity histogram (0 beyond the last) a word of quantity | nbins << 8 | the sign bits of lo and hi << 20, 21, and
// the other 63 bits of lo and of hi (non-negative words, so that -d never overflows).
enum {
  kDescRadMax = kAccums, kDescMasses, kDescEdges, kDescQSpec = kDescEdges + SART_MAX_BANDS + 1,
  kDescQLo = kDescQSpec + SART_N_QUANTITIES, kDescQHi = kDescQLo + SART_N_QUANTITIES, kDescErr = kDescQHi + SART_N_QUANTITIES,
  kDescWords
};
static_assert(2 * kDescWords <= kDescCapacity, "the descriptor travels in sart_handle::d_desc");

static void describe_outputs(const sart_handle* h, long long d[kDescWords]) {
  for (AccumKind k : kAllAccums) d[k] = h->accum[k].bins;
  // a handle has at most one of the single-mass and the per-mass radial histogram on, and at most one of the band images:
  // the r_max and edge words are those of the one that is on (its bins word tells which)
  const AccumKind rad = h->accum[kMassRadialHist].blob ? kMassRadialHist : kRadialHist;
  const AccumKind band = h->accum[kMassBandImages].blob ? kMassBandImages : kBandImages;
  std::memcpy(&d[kDescRadMax], &h->accum[rad].rmax, sizeof(long long));
  d[kDescMasses] = h->n_masses;
  std::memcpy(&d[kDescEdges], h->accum[band].edges, (SART_MAX_BANDS + 1) * sizeof(long long));
  const Accum& q = h->accum[kQuantityHists];
  for (int j = 0; j < SART_N_QUANTITIES; ++j) {
    uint64_t lo = 0, hi = 0;
    long long spec = 0;
    if (j < q.n_qhists) {
      std::memcpy(&lo, &q.qspecs[j].lo, sizeof lo);
      std::memcpy(&hi, &q.qspecs[j].hi, sizeof hi);
      spec = (long long)q.qspecs[j].quantity | (long long)q.qspecs[j].nbins << 8 | (long long)(lo >> 63) << 20 |
             (long long)(hi >> 63) << 21;
    }
    d[kDescQSpec + j] = spec;
    d[kDescQLo + j] = (long long)(lo & ~(uint64_t(1) << 63));
    d[kDescQHi + j] = (long long)(hi & ~(uint64_t(1) << 63));
  }
  d[kDescErr] = 0;
}

static ncclDataType_t nccl_type(const double*) { return ncclDouble; }
static ncclDataType_t nccl_type(const unsigned long long*) { return ncclUint64; }

}  // namespace sart

using namespace sart;

extern "C" {

int sart_comm_unique_id(char id[SART_COMM_ID_BYTES]) {
  if (!id) return fail(SART_ERR_ARG, "sart_comm_unique_id: id is NULL");
  NcclApi* n = nccl();
  if (!n) return fail(SART_ERR_CONFIG, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror() ? dlerror() : "not found");
  static_assert(sizeof(ncclUniqueId) == SART_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  ncclUniqueId u;
  SART_NCCL(n->GetUniqueId(&u));
  std::memcpy(id, &u, sizeof u);
  return SART_OK;
}

int sart_comm_init_rank(sart_handle_t* h, int n_ranks, int rank, const char id[SART_COMM_ID_BYTES]) {
  if (!h || !id) return fail(SART_ERR_ARG, "sart_comm_init_rank: NULL argument");
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(SART_ERR_ARG, "sart_comm_init_rank: rank %d of %d", rank, n_ranks);
  if (h->comm) return fail(SART_ERR_ARG, "sart_comm_init_rank: the handle already has a communicator");
  NcclApi* n = nccl();
  if (!n) return fail(SART_ERR_CONFIG, "NCCL (libnccl.so.2) could not be loaded");
  DeviceGuard dg(h->device);
  ncclUniqueId u;
  std::memcpy(&u, id, sizeof u);
  ncclComm_t c = nullptr;
  const ncclResult_t r = n->CommInitRank(&c, n_ranks, u, rank);
  if (r != ncclSuccess) return nccl_fail(r, "ncclCommInitRank");
  h->comm = c; h->comm_ranks = n_ranks; h->comm_rank = rank;
  return SART_OK;
}

int sart_comm_init_all(sart_handle_t* const* handles, int n) {
  if (!handles || n < 1 || n > 64) return fail(SART_ERR_ARG, "sart_comm_init_all: need 1..64 handles");
  int devs[64];
  for (int i = 0; i < n; ++i) {
    if (!handles[i]) return fail(SART_ERR_ARG, "sart_comm_init_all: handle %d is NULL", i);
    if (handles[i]->comm) return fail(SART_ERR_ARG, "sart_comm_init_all: handle %d already has a communicator", i);
    devs[i] = handles[i]->device;
    for (int j = 0; j < i; ++j)
      if (devs[j] == devs[i]) return fail(SART_ERR_ARG, "sart_comm_init_all: handles %d and %d share device %d", j, i, devs[i]);
  }
  NcclApi* api = nccl();
  if (!api) return fail(SART_ERR_CONFIG, "NCCL (libnccl.so.2) could not be loaded");
  ncclComm_t comms[64];
  SART_NCCL(api->CommInitAll(comms, n, devs));
  for (int i = 0; i < n; ++i) { handles[i]->comm = comms[i]; handles[i]->comm_ranks = n; handles[i]->comm_rank = i; }
  return SART_OK;
}

void sart_comm_destroy(sart_handle_t* h) {
  if (!h || !h->comm) return;
  NcclApi* n = nccl();
  if (n) {
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    n->CommDestroy(static_cast<ncclComm_t>(h->comm));
  }
  h->comm = nullptr; h->comm_ranks = 0; h->comm_rank = 0;
}

int sart_allreduce(sart_handle_t* const* handles, int n) {
  if (!handles || n < 1) return fail(SART_ERR_ARG, "sart_allreduce: need at least one handle");
  NcclApi* api = nccl();
  if (!api) return fail(SART_ERR_CONFIG, "NCCL (libnccl.so.2) could not be loaded");
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    if (!h || !h->comm) return fail(SART_ERR_ARG, "sart_allreduce: handle %d has no communicator (sart_comm_init_rank / _all)", i);
    if (!h->d_image) return fail(SART_ERR_NOMEM, "sart_allreduce: handle %d has no image buffers", i);
    if (h->n_masses != handles[0]->n_masses) return fail(SART_ERR_ARG, "sart_allreduce: handles differ in their number of axion masses");
  }
  // the counters of every handle as f64 words behind its two images, then one all-reduce per handle inside one group
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    DeviceGuard dg(h->device);
    const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
    const size_t words = merged_words(h->n_masses);
    if (h->merged_masses != h->n_masses) {
      cudaFree(h->d_merged);
      h->d_merged = nullptr; h->merged_masses = 0;
      cudaError_t e = cudaMalloc(&h->d_merged, words * sizeof(double));
      if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(merged)");
      h->merged_masses = h->n_masses;
    }
    const int nw = h->n_masses * kCounterWords;
    k_pack_counters<<<(nw + 127) / 128, 128, 0, h->stream>>>(h->d_counters, h->n_masses, h->d_image + 2 * len);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "k_pack_counters");
  }
  ncclResult_t r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    DeviceGuard dg(h->device);
    r = api->AllReduce(h->d_image, h->d_merged, merged_words(h->n_masses), ncclDouble, ncclSum, static_cast<ncclComm_t>(h->comm),
                       h->stream);
  }
  const ncclResult_t r2 = api->GroupEnd();
  if (r != ncclSuccess) return nccl_fail(r, "ncclAllReduce");
  if (r2 != ncclSuccess) return nccl_fail(r2, "ncclGroupEnd");
  for (int i = 0; i < n; ++i) handles[i]->merged_valid = 1;
  return SART_OK;
}

int sart_read_merged(sart_handle_t* h, double* image, double* image_w2, sart_counters_t* counters) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!h->d_merged || !h->merged_valid || h->merged_masses != h->n_masses)
    return fail(SART_ERR_ARG, "sart_read_merged: no merged result (call sart_allreduce first)");
  DeviceGuard dg(h->device);
  const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  cudaError_t e = cudaSuccess;
  if (image) e = cudaMemcpyAsync(image, h->d_merged, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && image_w2) e = cudaMemcpyAsync(image_w2, h->d_merged + len, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  double words[SART_MAX_MASSES * kCounterWords];
  if (e == cudaSuccess && counters)
    e = cudaMemcpyAsync(words, h->d_merged + 2 * len, size_t(h->n_masses) * kCounterWords * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return cuda_fail(e, "sart_read_merged");
  if (counters) {
    constexpr int nInt = int(offsetof(sart_counters_t, sum_w) / 8);
    for (int m = 0; m < h->n_masses; ++m) {
      unsigned long long* raw = reinterpret_cast<unsigned long long*>(counters + m);
      for (int w = 0; w < kCounterWords; ++w) {
        const double v = words[m * kCounterWords + w];
        if (w < nInt) raw[w] = (unsigned long long)(v + 0.5);
        else reinterpret_cast<double*>(raw)[w] = v;
      }
    }
  }
  return SART_OK;
}

int sart_allreduce_outputs(sart_handle_t* const* handles, int n) {
  if (!handles || n < 1) return fail(SART_ERR_ARG, "sart_allreduce_outputs: need at least one handle");
  NcclApi* api = nccl();
  if (!api) return fail(SART_ERR_CONFIG, "NCCL (libnccl.so.2) could not be loaded");
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    if (!h || !h->comm)
      return fail(SART_ERR_ARG, "sart_allreduce_outputs: handle %d has no communicator (sart_comm_init_rank / _all)", i);
    if (!h->d_image) return fail(SART_ERR_NOMEM, "sart_allreduce_outputs: handle %d has no image buffers", i);
  }
  // [d, -d] of every handle; the handles of this process are compared here already, before any collective
  std::vector<long long> desc(size_t(n) * 2 * kDescWords), red(desc.size());
  for (int i = 0; i < n; ++i) describe_outputs(handles[i], &desc[size_t(i) * 2 * kDescWords]);
  for (int i = 1; i < n; ++i)
    for (int k = 0; k < kDescErr; ++k)
      if (desc[size_t(i) * 2 * kDescWords + k] != desc[k])
        return fail(SART_ERR_CONFIG, "sart_allreduce_outputs: handles 0 and %d differ in their radial histogram, spectra, "
                                     "per-mass spectra, band images, quantity histograms, per-mass radial histograms, "
                                     "per-mass band images or number of axion masses", i);
  auto desc_dev = [](sart_handle* h) { return h->d_desc; };
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    long long* d = &desc[size_t(i) * 2 * kDescWords];
    DeviceGuard dg(h->device);
    // the merged copy of every accumulator that is on, laid out like the handle's own; kept until the accumulator is
    // switched again (sart_enable_*)
    for (AccumKind k : kAllAccums) {
      const Accum& a = h->accum[k];
      Accum& m = h->merged_accum[k];
      m.valid = 0;
      if (a.blob && !m.blob && alloc_accum(k, a.bins, a.rmax, &m) != SART_OK) {
        cudaGetLastError();   // the failed allocation is reported by every rank below, not here
        d[kDescErr] = 1;
      }
    }
    for (int k = 0; k < kDescWords; ++k) d[kDescWords + k] = -d[k];
    const cudaError_t e = cudaMemcpyAsync(desc_dev(h), d, 2 * kDescWords * sizeof(long long), cudaMemcpyHostToDevice, h->stream);
    if (e != cudaSuccess) return cuda_fail(e, "sart_allreduce_outputs");
  }
  ncclResult_t r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    DeviceGuard dg(h->device);
    r = api->AllReduce(desc_dev(h), desc_dev(h), 2 * kDescWords, ncclInt64, ncclMax, static_cast<ncclComm_t>(h->comm), h->stream);
  }
  ncclResult_t r2 = api->GroupEnd();
  if (r != ncclSuccess) return nccl_fail(r, "ncclAllReduce (descriptor)");
  if (r2 != ncclSuccess) return nccl_fail(r2, "ncclGroupEnd");
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    DeviceGuard dg(h->device);
    cudaError_t e = cudaMemcpyAsync(&red[size_t(i) * 2 * kDescWords], desc_dev(h), 2 * kDescWords * sizeof(long long),
                                    cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return cuda_fail(e, "sart_allreduce_outputs");
  }
  // every rank holds the same reduced words, so every rank takes the same decision
  const long long* hi = &red[0];
  const long long* neg_lo = &red[kDescWords];
  if (hi[kDescErr]) return fail(SART_ERR_NOMEM, "sart_allreduce_outputs: a rank could not allocate its merged copies");
  static const char* const what[kDescEdges] = {"radial histogram bins", "spectra bins", "per-mass spectra bins",
                                               "number of energy bands", "quantity histogram entries",
                                               "per-mass radial histogram bins", "number of per-mass energy bands",
                                               "radial histogram r_max", "number of axion masses"};
  for (int k = 0; k < kDescErr; ++k)
    if (hi[k] != -neg_lo[k])
      return fail(SART_ERR_CONFIG, "sart_allreduce_outputs: the ranks differ in their %s",
                  k < kDescEdges ? what[k] : (k < kDescQSpec ? "energy band edges" : "quantity histogram specs"));
  bool any = false;
  for (AccumKind k : kAllAccums) any |= hi[k] != 0;
  if (!any)
    return fail(SART_ERR_ARG, "sart_allreduce_outputs: no radial histogram, spectra or per-mass spectra enabled, and no band "
                              "images, quantity histograms, per-mass radial histograms or per-mass band images");
  // the payload: counts as u64, sums as f64, of the per-mass rows only those of the M masses set, every all-reduce of every
  // handle in one group
  r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    DeviceGuard dg(h->device);
    for (AccumKind k : kAllAccums)
      if (h->accum[k].blob)
        accum_arrays(k, h->accum[k], h->merged_accum[k], accum_rows(k, h->n_masses), [&](auto* src, auto* dst, size_t count) {
          if (r == ncclSuccess)
            r = api->AllReduce(src, dst, count, nccl_type(src), ncclSum, static_cast<ncclComm_t>(h->comm), h->stream);
        });
  }
  r2 = api->GroupEnd();
  if (r != ncclSuccess) return nccl_fail(r, "ncclAllReduce");
  if (r2 != ncclSuccess) return nccl_fail(r2, "ncclGroupEnd");
  for (int i = 0; i < n; ++i)
    for (AccumKind k : kAllAccums) handles[i]->merged_accum[k].valid = handles[i]->accum[k].blob != nullptr;
  return SART_OK;
}

int sart_read_merged_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  return read_accum(h, kRadialHist, true, {sum_w, counts},
                    "sart_read_merged_radial_hist: no merged radial histogram (call sart_allreduce_outputs first)");
}

int sart_read_merged_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                             double* shell_sum_w, uint64_t* shell_counts) {
  return read_accum(h, kSpectra, true, {energy_sum_w, energy_sum_w2, energy_counts, shell_sum_w, shell_counts},
                    "sart_read_merged_spectra: no merged spectra (call sart_allreduce_outputs first)");
}

int sart_read_merged_band_images(sart_handle_t* h, double* image, double* image_w2, uint64_t* counts) {
  return read_accum(h, kBandImages, true, {image, image_w2, counts},
                    "sart_read_merged_band_images: no merged band images (call sart_allreduce_outputs first)");
}

int sart_read_merged_quantity_hists(sart_handle_t* h, double* sum_w, double* sum_w2, uint64_t* counts) {
  return read_accum(h, kQuantityHists, true, {sum_w, sum_w2, counts},
                    "sart_read_merged_quantity_hists: no merged quantity histograms (call sart_allreduce_outputs first)");
}

int sart_read_merged_mass_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  return read_accum(h, kMassRadialHist, true, {sum_w, counts},
                    "sart_read_merged_mass_radial_hist: no merged per-mass radial histograms (call sart_allreduce_outputs first)");
}

int sart_read_merged_mass_band_images(sart_handle_t* h, double* image, double* image_w2, uint64_t* counts) {
  return read_accum(h, kMassBandImages, true, {image, image_w2, counts},
                    "sart_read_merged_mass_band_images: no merged per-mass band images (call sart_allreduce_outputs first)");
}

int sart_read_merged_mass_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                                  double* shell_sum_w, uint64_t* shell_counts) {
  return read_accum(h, kMassSpectra, true, {energy_sum_w, energy_sum_w2, energy_counts, shell_sum_w, shell_counts},
                    "sart_read_merged_mass_spectra: no merged per-mass spectra (call sart_allreduce_outputs first)");
}

}  // extern "C"
