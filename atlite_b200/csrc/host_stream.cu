// host_stream.cu -- the streaming behind the host-buffer entry points
// (atl_*_reduce_host): the cutout lives in host memory (NumPy arrays /
// NetCDF-backed), time slabs are streamed through a double-buffered device ring
// so H2D copies overlap the fused kernels, and the (time, bus) result is
// returned in host memory.  This is the call behind the reference-facing
// `Cutout.pv/wind/heat_demand(...)` when no device-resident copy of the cutout
// exists (bench.py "e2e").  Nothing here knows an operator: each one lists its
// fields (kernels.cuh: run_reduce_host, heat.cu).
//
// Pinned (cudaHostAlloc / cudaHostRegister'ed) inputs are DMA'd directly;
// pageable inputs go through a pinned staging ring (memcpy -> async H2D).
#include <sched.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "kernels.cuh"

namespace atl {

constexpr int NBUF = 2;

static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// Pinned staging buffers for pageable inputs are kept across calls (cudaHostAlloc
// of a few hundred MiB costs more than the transfer it serves); a call takes
// buffers out of the pool and puts them back when it returns.
struct StagePool {
  std::mutex mu;
  std::vector<std::pair<char*, size_t>> free_list;
  char* take(size_t bytes) {
    {
      std::lock_guard<std::mutex> lk(mu);
      int best = -1;
      for (int i = 0; i < (int)free_list.size(); ++i)
        if (free_list[i].second >= bytes && (best < 0 || free_list[i].second < free_list[best].second))
          best = i;
      if (best >= 0) {
        char* p = free_list[best].first;
        sizes.push_back({p, free_list[best].second});
        free_list.erase(free_list.begin() + best);
        return p;
      }
    }
    char* p = nullptr;
    if (cudaHostAlloc((void**)&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
      cudaGetLastError();
      release();  // drop cached buffers and retry once
      if (cudaHostAlloc((void**)&p, bytes, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    }
    std::lock_guard<std::mutex> lk(mu);
    sizes.push_back({p, bytes});
    return p;
  }
  void give(char* p) {
    std::lock_guard<std::mutex> lk(mu);
    for (size_t i = 0; i < sizes.size(); ++i)
      if (sizes[i].first == p) {
        free_list.push_back(sizes[i]);
        sizes.erase(sizes.begin() + i);
        return;
      }
  }
  void release() {
    std::lock_guard<std::mutex> lk(mu);
    for (auto& b : free_list) cudaFreeHost(b.first);
    free_list.clear();
  }
  std::vector<std::pair<char*, size_t>> sizes;  // buffers currently lent out
};
// One pool per device: its buffers are allocated (and first touched) by a thread bound to
// the CPUs next to that GPU, so they live on the GPU's NUMA node.
static StagePool g_stage_pool[64];
static StagePool& stage_pool(int device) { return g_stage_pool[(device >= 0 && device < 64) ? device : 0]; }

// ---- NUMA placement.  On a two-socket box half of the GPUs hang off each socket; a host
// thread that stages data for (or allocates pinned memory for) a GPU of the other socket
// pays the inter-socket link for every byte.  While a call streams slabs to device d, the
// calling thread -- and the staging-copy threads it spawns, which inherit the mask -- run on
// the CPUs the kernel lists as local to that PCI device
// (/sys/bus/pci/devices/<bus id>/local_cpulist).  ATL_NUMA_BIND=0 turns this off.
static bool device_local_cpus(int device, cpu_set_t* out) {
  static std::mutex mu;
  static bool known[64] = {false}, ok[64] = {false};
  static cpu_set_t sets[64];
  if (device < 0 || device >= 64) return false;
  std::lock_guard<std::mutex> lk(mu);
  if (!known[device]) {
    known[device] = true;
    const char* env = getenv("ATL_NUMA_BIND");
    char bus[64] = {0};
    if (!(env && atoi(env) == 0) && cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) {
      for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
      char path[160];
      snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/local_cpulist", bus);
      if (FILE* fh = fopen(path, "r")) {
        char line[4096] = {0};
        if (fgets(line, sizeof line, fh)) {
          CPU_ZERO(&sets[device]);
          int n = 0;
          for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
            int a = -1, b = -1;
            if (sscanf(tok, "%d-%d", &a, &b) == 2) {
            } else if (sscanf(tok, "%d", &a) == 1) {
              b = a;
            }
            for (int c = a; c >= 0 && c <= b && c < CPU_SETSIZE; ++c, ++n) CPU_SET(c, &sets[device]);
          }
          ok[device] = n > 0;
        }
        fclose(fh);
      }
    } else {
      cudaGetLastError();
    }
  }
  if (ok[device]) *out = sets[device];
  return ok[device];
}

// RAII: bind the calling thread to the device's local CPUs (intersected with the mask it
// already has), restore on scope exit.
struct NumaBind {
  cpu_set_t saved;
  bool active = false;
  explicit NumaBind(int device) {
    cpu_set_t local;
    if (!device_local_cpus(device, &local)) return;
    if (sched_getaffinity(0, sizeof saved, &saved) != 0) return;
    cpu_set_t both;
    CPU_AND(&both, &saved, &local);
    if (CPU_COUNT(&both) == 0) return;
    active = sched_setaffinity(0, sizeof both, &both) == 0;
  }
  ~NumaBind() {
    if (active) sched_setaffinity(0, sizeof saved, &saved);
  }
};

// Pageable -> pinned copy on several host threads (one thread moves ~10 GB/s, the
// PCIe link wants 50+).
static void par_memcpy(char* dst, const char* src, size_t bytes) {
  static const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t kMin = 1u << 20;  // measured: 4 threads move ~13 GB/s on the bench box
  unsigned nthr = (unsigned)std::min<size_t>(std::min(16u, hw), bytes / kMin);
  if (nthr <= 1) {
    std::memcpy(dst, src, bytes);
    return;
  }
  const size_t part = ((bytes / nthr) + 4095) & ~(size_t)4095;
  std::vector<std::thread> th;
  for (unsigned k = 1; k < nthr; ++k) {
    const size_t off = (size_t)k * part;
    if (off >= bytes) break;
    th.emplace_back([=] { std::memcpy(dst + off, src + off, std::min(part, bytes - off)); });
  }
  std::memcpy(dst, src, std::min(part, bytes));
  for (auto& t : th) t.join();
}

static void pool_keep_memory(int device) {
  static bool done[64] = {false};
  if (device < 0 || device >= 64 || done[device]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  done[device] = true;
}

// Stream `n_units` time units (steps, or days for heat demand) whose unit u
// starts at step unit_start(u) through the device ring.
int stream_slabs(const AtlOpBase* op, const AtlPlan* plan, const std::vector<SlabField>& fields,
                 int64_t n_units, const int64_t* unit_start, int64_t chunk_units, float* out_host,
                 const SlabLaunch& launch) {
  if (n_units <= 0) return ATL_OK;
  const int device = op->device;
  const int64_t S = op->grid.S;  // == ny * nx: check_host refuses padded operators
  const int32_t n_bus = plan->n_bus;
  ATL_CUDA(cudaSetDevice(device));
  NumaBind numa(device);
  StagePool& g_stage = stage_pool(device);
  pool_keep_memory(device);
  auto ustart = [&](int64_t u) { return unit_start ? unit_start[u] : u; };
  const int64_t total_steps = ustart(n_units) - ustart(0);
  size_t bytes_per_step = 0;
  for (const auto& f : fields)
    if (f.host) bytes_per_step += (size_t)S * f.elem;
  ATL_REQUIRE(bytes_per_step > 0, "no input fields");
  if (chunk_units <= 0) {
    // ~192 MiB of input per slab: long enough to amortise launch + copy setup,
    // short enough that the first kernel starts early
    const double steps_per_unit = (double)total_steps / (double)n_units;
    chunk_units = (int64_t)((192.0 * (1 << 20)) / ((double)bytes_per_step * steps_per_unit));
    if (chunk_units < 2) chunk_units = 2;
  }
  if (chunk_units > n_units) chunk_units = n_units;
  // widest slab in steps
  int64_t max_steps = 0;
  for (int64_t u = 0; u < n_units; u += chunk_units) {
    const int64_t e = u + chunk_units < n_units ? u + chunk_units : n_units;
    const int64_t n = ustart(e) - ustart(u);
    if (n > max_steps) max_steps = n;
  }

  cudaStream_t s_copy = nullptr, s_comp = nullptr;
  cudaEvent_t ev_copied[NBUF] = {nullptr}, ev_done[NBUF] = {nullptr}, ev_staged[NBUF] = {nullptr};
  std::vector<std::vector<void*>> dev(NBUF, std::vector<void*>(fields.size(), nullptr));
  std::vector<std::vector<char*>> stage(NBUF, std::vector<char*>(fields.size(), nullptr));
  float* out_dev = nullptr;
  int rc = ATL_OK;
  std::vector<bool> pinned(fields.size(), false);

#define SS_CUDA(call)                      \
  do {                                     \
    cudaError_t _e = (call);               \
    if (_e != cudaSuccess) {               \
      rc = cuda_fail(_e, #call);           \
      goto cleanup;                        \
    }                                      \
  } while (0)

  SS_CUDA(cudaStreamCreateWithFlags(&s_copy, cudaStreamNonBlocking));
  SS_CUDA(cudaStreamCreateWithFlags(&s_comp, cudaStreamNonBlocking));
  for (int b = 0; b < NBUF; ++b) {
    SS_CUDA(cudaEventCreateWithFlags(&ev_copied[b], cudaEventDisableTiming));
    SS_CUDA(cudaEventCreateWithFlags(&ev_done[b], cudaEventDisableTiming));
    SS_CUDA(cudaEventCreateWithFlags(&ev_staged[b], cudaEventDisableTiming));
  }
  for (size_t i = 0; i < fields.size(); ++i) {
    if (!fields[i].host) continue;
    pinned[i] = is_pinned(fields[i].host);
    const size_t bytes = (size_t)max_steps * S * fields[i].elem;
    for (int b = 0; b < NBUF; ++b) {
      SS_CUDA(cudaMallocAsync(&dev[b][i], bytes, s_copy));
      if (!pinned[i]) {
        stage[b][i] = g_stage.take(bytes);
        if (!stage[b][i]) {
          set_error("out of pinned host memory for the staging ring");
          rc = ATL_ERR_CUDA;
          goto cleanup;
        }
      }
    }
  }
  SS_CUDA(cudaMallocAsync((void**)&out_dev, (size_t)n_units * n_bus * sizeof(float) + 16, s_copy));
  SS_CUDA(cudaStreamSynchronize(s_copy));

  {
    int64_t it = 0;
    for (int64_t u = 0; u < n_units; u += chunk_units, ++it) {
      const int b = (int)(it % NBUF);
      const int64_t e = u + chunk_units < n_units ? u + chunk_units : n_units;
      const int64_t step0 = ustart(u), nsteps = ustart(e) - ustart(u);
      // the ring slot is free once the kernel that read it has finished
      if (it >= NBUF) SS_CUDA(cudaStreamWaitEvent(s_copy, ev_done[b], 0));
      for (size_t i = 0; i < fields.size(); ++i) {
        if (!fields[i].host) continue;
        const size_t off = (size_t)step0 * S * fields[i].elem;
        const size_t bytes = (size_t)nsteps * S * fields[i].elem;
        const char* src = fields[i].host + off;
        if (!pinned[i]) {
          if (it >= NBUF) SS_CUDA(cudaEventSynchronize(ev_staged[b]));  // staging slot drained
          par_memcpy(stage[b][i], src, bytes);
          src = stage[b][i];
        }
        SS_CUDA(cudaMemcpyAsync(dev[b][i], src, bytes, cudaMemcpyHostToDevice, s_copy));
      }
      SS_CUDA(cudaEventRecord(ev_staged[b], s_copy));
      SS_CUDA(cudaEventRecord(ev_copied[b], s_copy));
      SS_CUDA(cudaStreamWaitEvent(s_comp, ev_copied[b], 0));
      rc = launch(dev[b], u, e - u, out_dev + (size_t)u * n_bus, s_comp);
      if (rc != ATL_OK) goto cleanup;
      SS_CUDA(cudaEventRecord(ev_done[b], s_comp));
    }
  }
  SS_CUDA(cudaMemcpyAsync(out_host, out_dev, (size_t)n_units * n_bus * sizeof(float),
                          cudaMemcpyDeviceToHost, s_comp));
  SS_CUDA(cudaStreamSynchronize(s_comp));
  SS_CUDA(cudaStreamSynchronize(s_copy));

cleanup:
  if (s_comp) cudaStreamSynchronize(s_comp);
  if (s_copy) cudaStreamSynchronize(s_copy);
  for (int b = 0; b < NBUF; ++b) {
    for (size_t i = 0; i < fields.size(); ++i) {
      if (dev[b][i]) cudaFreeAsync(dev[b][i], s_copy ? s_copy : 0);
      if (stage[b][i]) g_stage.give(stage[b][i]);
    }
    if (ev_copied[b]) cudaEventDestroy(ev_copied[b]);
    if (ev_done[b]) cudaEventDestroy(ev_done[b]);
    if (ev_staged[b]) cudaEventDestroy(ev_staged[b]);
  }
  if (out_dev) cudaFreeAsync(out_dev, s_copy ? s_copy : 0);
  if (s_copy) {
    cudaStreamSynchronize(s_copy);
    cudaStreamDestroy(s_copy);
  }
  if (s_comp) cudaStreamDestroy(s_comp);
#undef SS_CUDA
  return rc;
}

}  // namespace atl

using namespace atl;

extern "C" {

void atl_release_host_staging(void) {
  for (auto& p : g_stage_pool) p.release();
}

int atl_device_local_cpus(int device, int32_t* cpus_out, int32_t capacity, int32_t* n_out) {
  ATL_REQUIRE(n_out, "n_out is NULL");
  *n_out = 0;
  cpu_set_t set;
  if (!device_local_cpus(device, &set)) return ATL_OK;  // unknown topology: empty list
  int32_t n = 0;
  for (int c = 0; c < CPU_SETSIZE; ++c)
    if (CPU_ISSET(c, &set)) {
      if (cpus_out && n < capacity) cpus_out[n] = c;
      ++n;
    }
  *n_out = n;
  return ATL_OK;
}

}  // extern "C"
