// comm.cu — the one collective of the path: the sum of the detector images and counters of all GPUs.
//
// Rays shard over GPUs by global ray index (Philox counter), with no exchange while tracing (SURVEY.md §8e); what has
// to be merged afterwards is additive: image [M][256][256], the sum-of-squares image and the counters. The handle keeps
// image and sum-of-squares image in ONE allocation followed by a small f64 area; sart_allreduce writes the counters into
// that area as f64 (exact below 2^53) and issues ONE ncclAllReduce(sum, f64) over the whole block into a separate
// "merged" block, so a rank's own accumulators stay untouched (no reset between steps) and the call can be repeated.
// sart_allreduce_outputs does the same for the optional accumulators (radial histogram, spectra, per-mass spectra): the
// ranks first agree on which are on and their shapes, then sum them into merged copies, counts as u64 and sums as f64.
//
// NCCL is resolved with dlopen at first use: libsart.so has no link-time dependency on it, a process that already
// loaded NCCL (PyTorch) shares that copy, and a host without NCCL can use everything else.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <cstring>
#include <initializer_list>
#include <vector>

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
// [d, -d] through one ncclMax, so each learns the largest and (negated) smallest value of every word.
enum { kDescRadBins, kDescRadMax, kDescSpecBins, kDescMassSpecBins, kDescMasses, kDescErr, kDescWords };
static_assert(2 * kDescWords <= kCounterWords, "the descriptor travels in the counter words behind the images");

static void describe_outputs(const sart_handle* h, long long d[kDescWords]) {
  long long rmax = 0;
  std::memcpy(&rmax, &h->rad_rmax, sizeof rmax);
  d[kDescRadBins] = h->rad_bins;
  d[kDescRadMax] = h->rad_bins ? rmax : 0;
  d[kDescSpecBins] = h->spec.eW ? h->spec_e1 : 0;
  d[kDescMassSpecBins] = h->mspec.eW ? h->mspec_e1 : 0;
  d[kDescMasses] = h->n_masses;
  d[kDescErr] = 0;
}

// (Re)allocates the handle's merged copies for what it has on; keeps them while the shapes stay. Returns a CUDA error.
static cudaError_t ensure_merged_outputs(sart_handle* h) {
  MergedOutputs& m = h->merged_out;
  const int spec_e1 = h->spec.eW ? h->spec_e1 : 0, mspec_e1 = h->mspec.eW ? h->mspec_e1 : 0;
  if (m.blob && m.rad_bins == h->rad_bins && m.spec_e1 == spec_e1 && m.mspec_e1 == mspec_e1) return cudaSuccess;
  auto layout = [&](unsigned char* base) {   // radial w | radial n | spectra | per-mass spectra, as the handle has them
    Carve c(base);
    c.take(m.rad_w, size_t(h->rad_bins)); c.take(m.rad_n, size_t(h->rad_bins));
    if (spec_e1) c.off += carve_spectra(base ? base + c.off : nullptr, spec_e1, 1, 1, &m.spec);
    if (mspec_e1) c.off += carve_mass_spectra(base ? base + c.off : nullptr, mspec_e1, &m.mspec);
    return c.off;
  };
  cudaFree(m.blob);
  m = MergedOutputs{};
  void* blob = nullptr;
  const cudaError_t e = cudaMalloc(&blob, layout(nullptr));
  if (e != cudaSuccess) { m = MergedOutputs{}; return e; }
  m.blob = blob;
  layout(static_cast<unsigned char*>(blob));
  m.rad_bins = h->rad_bins; m.spec_e1 = spec_e1; m.mspec_e1 = mspec_e1;
  return cudaSuccess;
}

// Copies device arrays of a handle's merged copies to host arrays (a NULL host array is skipped) and synchronises.
struct Part {
  void* host;
  const void* dev;
  size_t bytes;
};
static int read_merged_parts(sart_handle* h, const char* who, std::initializer_list<Part> parts) {
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(h->device);
  cudaError_t e = cudaSuccess;
  for (const Part& p : parts)
    if (p.host && e == cudaSuccess) e = cudaMemcpyAsync(p.host, p.dev, p.bytes, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaSetDevice(prev);
  return e == cudaSuccess ? SART_OK : fail(SART_ERR_CUDA, "%s: %s", who, cudaGetErrorString(e));
}

// `rows` rows of merged spectra: energy_* [rows][e1], shell_* [rows][SART_MAX_SHELLS].
static int read_merged_spectra(sart_handle* h, const char* who, const Spectra& s, int rows, int e1, double* eW, double* eW2,
                               uint64_t* eN, double* sW, uint64_t* sN) {
  const size_t e = size_t(rows) * e1 * 8, sh = size_t(rows) * SART_MAX_SHELLS * 8;
  return read_merged_parts(h, who, {{eW, s.eW, e}, {eW2, s.eW2, e}, {eN, s.eN, e}, {sW, s.sW, sh}, {sN, s.sN, sh}});
}

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
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(h->device);
  ncclUniqueId u;
  std::memcpy(&u, id, sizeof u);
  ncclComm_t c = nullptr;
  const ncclResult_t r = n->CommInitRank(&c, n_ranks, u, rank);
  cudaSetDevice(prev);
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
  int prev = 0;
  cudaGetDevice(&prev);
  // the counters of every handle as f64 words behind its two images, then one all-reduce per handle inside one group
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    cudaSetDevice(h->device);
    const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
    const size_t words = merged_words(h->n_masses);
    if (h->merged_masses != h->n_masses) {
      cudaFree(h->d_merged);
      h->d_merged = nullptr; h->merged_masses = 0;
      cudaError_t e = cudaMalloc(&h->d_merged, words * sizeof(double));
      if (e != cudaSuccess) { cudaSetDevice(prev); return fail(SART_ERR_CUDA, "cudaMalloc(merged): %s", cudaGetErrorString(e)); }
      h->merged_masses = h->n_masses;
    }
    const int nw = h->n_masses * kCounterWords;
    k_pack_counters<<<(nw + 127) / 128, 128, 0, h->stream>>>(h->d_counters, h->n_masses, h->d_image + 2 * len);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cudaSetDevice(prev); return fail(SART_ERR_CUDA, "k_pack_counters: %s", cudaGetErrorString(e)); }
  }
  ncclResult_t r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    cudaSetDevice(h->device);
    r = api->AllReduce(h->d_image, h->d_merged, merged_words(h->n_masses), ncclDouble, ncclSum, static_cast<ncclComm_t>(h->comm),
                       h->stream);
  }
  const ncclResult_t r2 = api->GroupEnd();
  cudaSetDevice(prev);
  if (r != ncclSuccess) return nccl_fail(r, "ncclAllReduce");
  if (r2 != ncclSuccess) return nccl_fail(r2, "ncclGroupEnd");
  for (int i = 0; i < n; ++i) handles[i]->merged_valid = 1;
  return SART_OK;
}

int sart_read_merged(sart_handle_t* h, double* image, double* image_w2, sart_counters_t* counters) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!h->d_merged || !h->merged_valid || h->merged_masses != h->n_masses)
    return fail(SART_ERR_ARG, "sart_read_merged: no merged result (call sart_allreduce first)");
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(h->device);
  const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  cudaError_t e = cudaSuccess;
  if (image) e = cudaMemcpyAsync(image, h->d_merged, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && image_w2) e = cudaMemcpyAsync(image_w2, h->d_merged + len, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  double words[SART_MAX_MASSES * kCounterWords];
  if (e == cudaSuccess && counters)
    e = cudaMemcpyAsync(words, h->d_merged + 2 * len, size_t(h->n_masses) * kCounterWords * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaSetDevice(prev);
  if (e != cudaSuccess) return fail(SART_ERR_CUDA, "sart_read_merged: %s", cudaGetErrorString(e));
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
                                     "per-mass spectra or number of axion masses", i);
  int prev = 0;
  cudaGetDevice(&prev);
  auto done = [&](int rc) { cudaSetDevice(prev); return rc; };
  // the descriptor travels in the counter words behind the images: sart_allreduce rewrites them before every use
  auto desc_dev = [](sart_handle* h) {
    return reinterpret_cast<long long*>(h->d_image + 2 * size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS);
  };
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    long long* d = &desc[size_t(i) * 2 * kDescWords];
    cudaSetDevice(h->device);
    MergedOutputs& m = h->merged_out;
    m.rad_valid = m.spec_valid = m.mspec_valid = 0;
    if ((d[kDescRadBins] || d[kDescSpecBins] || d[kDescMassSpecBins]) && ensure_merged_outputs(h) != cudaSuccess) {
      cudaGetLastError();   // the failed allocation is reported by every rank below, not here
      d[kDescErr] = 1;
    }
    for (int k = 0; k < kDescWords; ++k) d[kDescWords + k] = -d[k];
    const cudaError_t e = cudaMemcpyAsync(desc_dev(h), d, 2 * kDescWords * sizeof(long long), cudaMemcpyHostToDevice, h->stream);
    if (e != cudaSuccess) return done(fail(SART_ERR_CUDA, "sart_allreduce_outputs: %s", cudaGetErrorString(e)));
  }
  ncclResult_t r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    cudaSetDevice(h->device);
    r = api->AllReduce(desc_dev(h), desc_dev(h), 2 * kDescWords, ncclInt64, ncclMax, static_cast<ncclComm_t>(h->comm), h->stream);
  }
  ncclResult_t r2 = api->GroupEnd();
  if (r != ncclSuccess) return done(nccl_fail(r, "ncclAllReduce (descriptor)"));
  if (r2 != ncclSuccess) return done(nccl_fail(r2, "ncclGroupEnd"));
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    cudaSetDevice(h->device);
    cudaError_t e = cudaMemcpyAsync(&red[size_t(i) * 2 * kDescWords], desc_dev(h), 2 * kDescWords * sizeof(long long),
                                    cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return done(fail(SART_ERR_CUDA, "sart_allreduce_outputs: %s", cudaGetErrorString(e)));
  }
  // every rank holds the same reduced words, so every rank takes the same decision
  const long long* hi = &red[0];
  const long long* neg_lo = &red[kDescWords];
  if (hi[kDescErr]) return done(fail(SART_ERR_NOMEM, "sart_allreduce_outputs: a rank could not allocate its merged copies"));
  static const char* const what[kDescErr] = {"radial histogram bins", "radial histogram r_max", "spectra bins",
                                             "per-mass spectra bins", "number of axion masses"};
  for (int k = 0; k < kDescErr; ++k)
    if (hi[k] != -neg_lo[k]) return done(fail(SART_ERR_CONFIG, "sart_allreduce_outputs: the ranks differ in their %s", what[k]));
  if (!hi[kDescRadBins] && !hi[kDescSpecBins] && !hi[kDescMassSpecBins])
    return done(fail(SART_ERR_ARG, "sart_allreduce_outputs: no radial histogram, spectra or per-mass spectra enabled"));
  // the payload: counts as u64, sums as f64, every all-reduce of every handle in one group
  r = api->GroupStart();
  for (int i = 0; i < n && r == ncclSuccess; ++i) {
    sart_handle* h = handles[i];
    MergedOutputs& m = h->merged_out;
    cudaSetDevice(h->device);
    auto sum = [&](const void* src, void* dst, size_t count, ncclDataType_t t) {
      if (r == ncclSuccess) r = api->AllReduce(src, dst, count, t, ncclSum, static_cast<ncclComm_t>(h->comm), h->stream);
    };
    auto spectra = [&](const Spectra& s, const Spectra& d, size_t e, size_t sh) {
      sum(s.eW, d.eW, e, ncclDouble); sum(s.eW2, d.eW2, e, ncclDouble); sum(s.eN, d.eN, e, ncclUint64);
      sum(s.sW, d.sW, sh, ncclDouble); sum(s.sN, d.sN, sh, ncclUint64);
    };
    if (h->rad_bins) { sum(h->d_rad_w, m.rad_w, h->rad_bins, ncclDouble); sum(h->d_rad_n, m.rad_n, h->rad_bins, ncclUint64); }
    if (h->spec.eW) spectra(h->spec, m.spec, h->spec_e1, SART_MAX_SHELLS);
    // per-mass rows: only those of the M masses set
    if (h->mspec.eW) spectra(h->mspec, m.mspec, size_t(h->n_masses) * h->mspec_e1, size_t(h->n_masses) * SART_MAX_SHELLS);
  }
  r2 = api->GroupEnd();
  if (r != ncclSuccess) return done(nccl_fail(r, "ncclAllReduce"));
  if (r2 != ncclSuccess) return done(nccl_fail(r2, "ncclGroupEnd"));
  for (int i = 0; i < n; ++i) {
    sart_handle* h = handles[i];
    h->merged_out.rad_valid = h->rad_bins > 0;
    h->merged_out.spec_valid = h->spec.eW != nullptr;
    h->merged_out.mspec_valid = h->mspec.eW != nullptr;
  }
  return done(SART_OK);
}

int sart_read_merged_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  const MergedOutputs& m = h->merged_out;
  if (!m.rad_valid)
    return fail(SART_ERR_ARG, "sart_read_merged_radial_hist: no merged radial histogram (call sart_allreduce_outputs first)");
  const size_t nb = size_t(m.rad_bins);
  return read_merged_parts(h, "sart_read_merged_radial_hist", {{sum_w, m.rad_w, nb * 8}, {counts, m.rad_n, nb * 8}});
}

int sart_read_merged_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                             double* shell_sum_w, uint64_t* shell_counts) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  const MergedOutputs& m = h->merged_out;
  if (!m.spec_valid) return fail(SART_ERR_ARG, "sart_read_merged_spectra: no merged spectra (call sart_allreduce_outputs first)");
  return read_merged_spectra(h, "sart_read_merged_spectra", m.spec, 1, m.spec_e1, energy_sum_w, energy_sum_w2, energy_counts,
                             shell_sum_w, shell_counts);
}

int sart_read_merged_mass_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                                  double* shell_sum_w, uint64_t* shell_counts) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  const MergedOutputs& m = h->merged_out;
  if (!m.mspec_valid)
    return fail(SART_ERR_ARG, "sart_read_merged_mass_spectra: no merged per-mass spectra (call sart_allreduce_outputs first)");
  return read_merged_spectra(h, "sart_read_merged_mass_spectra", m.mspec, h->n_masses, m.mspec_e1, energy_sum_w,
                             energy_sum_w2, energy_counts, shell_sum_w, shell_counts);
}

}  // extern "C"
