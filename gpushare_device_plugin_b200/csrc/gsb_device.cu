/*
 * gsb_device.cu — device layer of libgpushare_b200.so: lifecycle, inventory, arena, probe, cycle,
 * health events. Host code; the kernels live in hbm_probe_sm100a.cu.
 *
 * Replaces the reference's go-nvml use (vendor/github.com/NVIDIA/gpu-monitoring-tools/bindings/go/
 * nvml/{nvml.go,bindings.go,nvml_dl.c}) for the inventory+health path:
 *   - nvml.Init (nvml_dl.c:21-28: dlopen + nvmlInit_v2)             -> gsb_init
 *   - nvml.NewDevice's 11 getters + sysfs read (nvml.go:297-359)     -> 4 NVML calls per device
 *     (handle, UUID, minor, MemoryInfo v1) + 2 CUDA driver calls that cross-check identity; the
 *     eight getters whose values the plugin discards (name, power, PCI, BAR1, link gen/width,
 *     clocks, NUMA) are not made
 *   - total MiB = nvmlMemory_t.total / (1024*1024) (bindings.go:346-349): SAME call, SAME struct, so
 *     the slice count is bit-exact by construction. cuDeviceTotalMem is 762 839 040 B smaller on a
 *     B200 (profiles/envprobe_r01.txt: 178 vs 179 GiB) and is reported only as information.
 *   - RegisterEventForDevice x fake devices (nvidia.go:104-117; O(S*N^2) NVML calls) -> one
 *     nvmlDeviceRegisterEvents per GPU
 *   - WaitForEvent (bindings.go:134-146) -> gsb_health_wait over a queue fed by the XID thread and
 *     by the active HBM prober
 *
 * libcuda.so.1 and libnvidia-ml.so.1 are dlopen'ed at gsb_init, never linked: the library loads on
 * a GPU-less builder (symbol check in tests/test_abi.py) and reports GSB_ERR_LIBRARY_NOT_FOUND there.
 */
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvml.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <thread>
#include <vector>

#include "gsb_internal.h"

namespace {

// ------------------------------------------------------------------ error text

thread_local char tl_error[512];

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tl_error, sizeof tl_error, fmt, ap);
  va_end(ap);
}

uint64_t now_ns() {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec;
}

// ------------------------------------------------------------------ dlopen'ed entry points

struct DriverApi {
  void *lib = nullptr;
  CUresult (*cuInit)(unsigned) = nullptr;
  CUresult (*cuDeviceGet)(CUdevice *, int) = nullptr;
  CUresult (*cuDeviceGetUuid)(CUuuid *, CUdevice) = nullptr;
  CUresult (*cuDeviceTotalMem)(size_t *, CUdevice) = nullptr;
  CUresult (*cuMemGetInfo)(size_t *, size_t *) = nullptr;
  CUresult (*cuMemGetAllocationGranularity)(size_t *, const CUmemAllocationProp *,
                                            CUmemAllocationGranularity_flags) = nullptr;
  CUresult (*cuMemAddressReserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
  CUresult (*cuMemAddressFree)(CUdeviceptr, size_t) = nullptr;
  CUresult (*cuMemCreate)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *,
                          unsigned long long) = nullptr;
  CUresult (*cuMemRelease)(CUmemGenericAllocationHandle) = nullptr;
  CUresult (*cuMemMap)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
  CUresult (*cuMemUnmap)(CUdeviceptr, size_t) = nullptr;
  CUresult (*cuMemSetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t) = nullptr;
  CUresult (*cuGetErrorString)(CUresult, const char **) = nullptr;
};

struct NvmlApi {
  void *lib = nullptr;
  nvmlReturn_t (*init)(void) = nullptr;
  nvmlReturn_t (*shutdown)(void) = nullptr;
  const char *(*errorString)(nvmlReturn_t) = nullptr;
  nvmlReturn_t (*getCount)(unsigned *) = nullptr;
  nvmlReturn_t (*handleByIndex)(unsigned, nvmlDevice_t *) = nullptr;
  nvmlReturn_t (*getUUID)(nvmlDevice_t, char *, unsigned) = nullptr;
  nvmlReturn_t (*getMinor)(nvmlDevice_t, unsigned *) = nullptr;
  nvmlReturn_t (*getMemoryInfo)(nvmlDevice_t, nvmlMemory_t *) = nullptr;  // v1 struct: the reference's
  nvmlReturn_t (*getPciInfo)(nvmlDevice_t, nvmlPciInfo_t *) = nullptr;
  nvmlReturn_t (*eventSetCreate)(nvmlEventSet_t *) = nullptr;
  nvmlReturn_t (*registerEvents)(nvmlDevice_t, unsigned long long, nvmlEventSet_t) = nullptr;
  nvmlReturn_t (*eventSetWait)(nvmlEventSet_t, nvmlEventData_t *, unsigned) = nullptr;
  nvmlReturn_t (*eventSetFree)(nvmlEventSet_t) = nullptr;
};

template <typename F>
bool load_sym(void *lib, F &fn, const char *name, const char *alt = nullptr) {
  fn = reinterpret_cast<F>(dlsym(lib, name));
  if (!fn && alt) fn = reinterpret_cast<F>(dlsym(lib, alt));
  return fn != nullptr;
}

// ------------------------------------------------------------------ state

constexpr uint64_t kGranuleBytes = 64ull << 20;  // generation-table granularity
constexpr uint32_t kGranuleShiftWords = 22;      // log2(64 MiB / 16 B)

struct Chunk {
  CUmemGenericAllocationHandle handle;
  size_t size;
};

struct Snapshot {
  char uuid[GSB_UUID_BUFFER_SIZE] = {0};
  unsigned char uuid_bytes[16] = {0};  // the same UUID as the CUDA driver reports it (cuDeviceGetUuid)
  bool uuid_parsed = false;
  uint32_t minor = 0;
  uint64_t total = 0, free = 0;
  uint64_t taken_ns = 0;
  uint64_t refreshes = 0;
};

// what a device worker runs: plain data, no allocation per hand-off
struct Job {
  enum Kind { NONE, PROBE, CYCLE } kind = NONE;
  uint32_t idx = 0;
  const gsb_probe_cfg *cfg = nullptr;
  gsb_probe_result *probe_out = nullptr;
  uint64_t cycle_no = 0, window_bytes = 0;
  int unit_gib = 1;
  uint32_t variant = 0;
  gsb_cycle_result *cycle_out = nullptr;
  int rc = 0;
};

struct Device {
  nvmlDevice_t nvml{};
  int ordinal = -1;
  CUdevice cudev = 0;
  char uuid[GSB_UUID_BUFFER_SIZE] = {0};
  char bus_id[GSB_BUSID_BUFFER_SIZE] = {0};
  uint32_t minor = 0;
  uint32_t sm_count = 0, cc_major = 0, cc_minor = 0;
  uint64_t cuda_total = 0;

  std::mutex mu;  // serialises arena + launches of this device
  bool ready = false;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  gsb_kernel_out *out_host = nullptr, *out_dev = nullptr;
  gsb_partial *partials = nullptr;
  unsigned int *ticket = nullptr;
  unsigned long long *tile_counter = nullptr;
  uint32_t *seed_table = nullptr;  // device copy of gen[]
  uint32_t launch_seq = 0;

  CUdeviceptr va = 0;
  size_t va_size = 0;
  std::vector<Chunk> chunks;
  uint64_t arena_bytes = 0;
  std::map<uint64_t, gsb_launch_geom> geoms;  // (op, variant, grid request) -> resolved launch geometry
  std::vector<uint32_t> gen;  // host mirror of seed_table: generation that last wrote each granule
  uint32_t next_gen = 1;
  bool faulted = false;  // prober: sticky
  std::vector<uint8_t> bits_scratch;  // Unhealthy bit string of this device's own list (faulted devices only)
  bool transient_arena = false;  // the mapped arena is a transient window that could not be given back yet (wedged launch)
  bool wedged = false;   // a launch outlived the watchdog and is still on the stream: no new launches until it drains

  // inventory snapshot: what NVML said at the last (re)start-time query (server.go:39 -> nvidia.go:53-89 queries
  // once per plugin start, never per poll). The cycle serves identity/total from here and re-validates identity on
  // the CUDA side; gsb_device_info_get / gsb_inventory_refresh / the low-rate refresher rewrite it.
  std::mutex smu;
  Snapshot snap;
  gsb_health_stats hstats{};  // prober thread of this device; guarded by smu

  // persistent worker (gsb_cycle_all / gsb_probe_all): one host thread per device
  std::thread worker;
  std::mutex wmu;
  std::condition_variable wcv;
  Job job;
  bool job_ready = false, job_done = false, worker_quit = false;
  std::atomic<bool> job_flag{false}, done_flag{false}, quit_flag{false};  // lock-free mirrors for the spin phase
};

struct Global {
  // every device-touching entry point holds this shared; gsb_init/gsb_shutdown take it exclusively, so a
  // shutdown waits for calls still running on other threads (e.g. a start-up walk) instead of freeing
  // devices under them
  std::shared_mutex api_mu;
  std::mutex mu;
  bool inited = false;
  DriverApi cu;
  NvmlApi ml;
  std::vector<std::unique_ptr<Device>> devs;  // NVML index order

  // options (gsb_set_option)
  std::atomic<uint64_t> inventory_policy{GSB_INVENTORY_SNAPSHOT};
  std::atomic<uint64_t> wait_spin_us{2000};
  std::atomic<uint64_t> watchdog_ms{2000};
  std::atomic<uint64_t> inventory_refresh_ms{5000};
  std::atomic<uint64_t> transient_keep_free{1ull << 30};
  std::atomic<uint64_t> sweep_every{0};

  // node cycle (gsb_cycle_all / gsb_probe_all): one at a time; scratch of the join lives here, not on the heap per call
  std::mutex all_mu;
  std::vector<uint8_t> join_bits;

  // health
  // serialises gsb_health_start, gsb_health_stop and gsb_shutdown, so that one call's threads and event set are never
  // torn down by another's, nor devices freed under probers still running; taken before api_mu, never after it
  std::mutex life_mu;
  std::mutex hmu;
  std::condition_variable hcv;
  std::deque<gsb_event> events;
  bool health_running = false;
  std::atomic<bool> health_stop{false};
  std::atomic<uint32_t> recovery_cycles{0};
  uint64_t stop_gen = 0;  // bumped by every gsb_health_stop: wakes all gsb_health_wait callers
  std::vector<std::thread> health_threads;
  nvmlEventSet_t event_set{};
  bool have_event_set = false;
};

Global G;

const char *cu_err(CUresult r) {
  const char *s = nullptr;
  if (G.cu.cuGetErrorString && G.cu.cuGetErrorString(r, &s) == CUDA_SUCCESS && s) return s;
  return "unknown CUDA driver error";
}

#define CU_TRY(expr)                                                      \
  do {                                                                    \
    CUresult _r = (expr);                                                 \
    if (_r != CUDA_SUCCESS) {                                             \
      set_error("%s -> %d (%s)", #expr, (int)_r, cu_err(_r));             \
      return GSB_ERR_DRIVER;                                              \
    }                                                                     \
  } while (0)

#define RT_TRY(expr)                                                      \
  do {                                                                    \
    cudaError_t _r = (expr);                                              \
    if (_r != cudaSuccess) {                                              \
      set_error("%s -> %d (%s)", #expr, (int)_r, cudaGetErrorString(_r)); \
      return _r == cudaErrorMemoryAllocation ? GSB_ERR_OUT_OF_MEMORY : GSB_ERR_DRIVER; \
    }                                                                     \
  } while (0)

// "nvml: <nvmlErrorString>" is the reference's error text (bindings.go:52-58)
#define ML_TRY(expr)                                                      \
  do {                                                                    \
    nvmlReturn_t _r = (expr);                                             \
    if (_r != NVML_SUCCESS) {                                             \
      set_error("nvml: %s", G.ml.errorString ? G.ml.errorString(_r) : "?"); \
      return GSB_ERR_NVML;                                                \
    }                                                                     \
  } while (0)

void format_uuid(const CUuuid &u, char out[GSB_UUID_BUFFER_SIZE]) {
  const unsigned char *b = reinterpret_cast<const unsigned char *>(u.bytes);
  snprintf(out, GSB_UUID_BUFFER_SIZE,
           "GPU-%02x%02x%02x%02x-%02x%02x-%02x%02x-%02x%02x-%02x%02x%02x%02x%02x%02x", b[0], b[1], b[2],
           b[3], b[4], b[5], b[6], b[7], b[8], b[9], b[10], b[11], b[12], b[13], b[14], b[15]);
}

int load_libraries() {
  if (!G.cu.lib) {
    G.cu.lib = dlopen("libcuda.so.1", RTLD_LAZY | RTLD_GLOBAL);
    if (!G.cu.lib) {
      set_error("could not load CUDA driver library: %s", dlerror());
      return GSB_ERR_LIBRARY_NOT_FOUND;
    }
    DriverApi &c = G.cu;
    bool ok = load_sym(c.lib, c.cuInit, "cuInit") && load_sym(c.lib, c.cuDeviceGet, "cuDeviceGet") &&
              load_sym(c.lib, c.cuDeviceGetUuid, "cuDeviceGetUuid_v2", "cuDeviceGetUuid") &&
              load_sym(c.lib, c.cuDeviceTotalMem, "cuDeviceTotalMem_v2") &&
              load_sym(c.lib, c.cuMemGetInfo, "cuMemGetInfo_v2") &&
              load_sym(c.lib, c.cuMemGetAllocationGranularity, "cuMemGetAllocationGranularity") &&
              load_sym(c.lib, c.cuMemAddressReserve, "cuMemAddressReserve") &&
              load_sym(c.lib, c.cuMemAddressFree, "cuMemAddressFree") &&
              load_sym(c.lib, c.cuMemCreate, "cuMemCreate") && load_sym(c.lib, c.cuMemRelease, "cuMemRelease") &&
              load_sym(c.lib, c.cuMemMap, "cuMemMap") && load_sym(c.lib, c.cuMemUnmap, "cuMemUnmap") &&
              load_sym(c.lib, c.cuMemSetAccess, "cuMemSetAccess") &&
              load_sym(c.lib, c.cuGetErrorString, "cuGetErrorString");
    if (!ok) {
      set_error("libcuda.so.1 lacks a required entry point");
      return GSB_ERR_LIBRARY_NOT_FOUND;
    }
  }
  if (!G.ml.lib) {
    // same library name and flags as the reference's shim (nvml_dl.c:23)
    G.ml.lib = dlopen("libnvidia-ml.so.1", RTLD_LAZY | RTLD_GLOBAL);
    if (!G.ml.lib) {
      set_error("could not load NVML library");  // bindings.go:63
      return GSB_ERR_LIBRARY_NOT_FOUND;
    }
    NvmlApi &m = G.ml;
    bool ok = load_sym(m.lib, m.init, "nvmlInit_v2") && load_sym(m.lib, m.shutdown, "nvmlShutdown") &&
              load_sym(m.lib, m.errorString, "nvmlErrorString") &&
              load_sym(m.lib, m.getCount, "nvmlDeviceGetCount_v2") &&
              load_sym(m.lib, m.handleByIndex, "nvmlDeviceGetHandleByIndex_v2") &&
              load_sym(m.lib, m.getUUID, "nvmlDeviceGetUUID") &&
              load_sym(m.lib, m.getMinor, "nvmlDeviceGetMinorNumber") &&
              load_sym(m.lib, m.getMemoryInfo, "nvmlDeviceGetMemoryInfo") &&
              load_sym(m.lib, m.getPciInfo, "nvmlDeviceGetPciInfo_v3");
    if (!ok) {
      set_error("libnvidia-ml.so.1 lacks a required entry point");
      return GSB_ERR_LIBRARY_NOT_FOUND;
    }
    // optional (health): absence only disables the XID half
    load_sym(m.lib, m.eventSetCreate, "nvmlEventSetCreate");
    load_sym(m.lib, m.registerEvents, "nvmlDeviceRegisterEvents");
    load_sym(m.lib, m.eventSetWait, "nvmlEventSetWait_v2", "nvmlEventSetWait");
    load_sym(m.lib, m.eventSetFree, "nvmlEventSetFree");
  }
  return GSB_OK;
}

Device *device_at(uint32_t idx) {
  if (!G.inited) {
    set_error("gsb_init has not succeeded");
    return nullptr;
  }
  if (idx >= G.devs.size()) {
    set_error("nvml: device not found (index %u of %zu)", idx, G.devs.size());
    return nullptr;
  }
  return G.devs[idx].get();
}

// per-device CUDA resources, created on first probe/arena use (primary context via the runtime)
int ensure_ready(Device *d) {
  if (d->ordinal < 0) {
    set_error("device %s is not visible to the CUDA driver in this process", d->uuid);
    return GSB_ERR_NO_DEVICE;
  }
  if (d->cc_major != 10) {
    set_error("device %s is compute capability %u.%u; this library carries sm_100a code only", d->uuid,
              d->cc_major, d->cc_minor);
    return GSB_ERR_UNSUPPORTED_ARCH;
  }
  RT_TRY(cudaSetDevice(d->ordinal));
  if (d->ready) return GSB_OK;
  RT_TRY(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  RT_TRY(cudaEventCreate(&d->ev0));
  RT_TRY(cudaEventCreate(&d->ev1));
  RT_TRY(cudaHostAlloc(reinterpret_cast<void **>(&d->out_host), sizeof(gsb_kernel_out),
                       cudaHostAllocMapped | cudaHostAllocPortable));
  memset(d->out_host, 0, sizeof(gsb_kernel_out));
  RT_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&d->out_dev), d->out_host, 0));
  RT_TRY(cudaMalloc(reinterpret_cast<void **>(&d->partials),
                    sizeof(gsb_partial) * gsb_kernel_max_grid((int)d->sm_count)));
  RT_TRY(cudaMalloc(reinterpret_cast<void **>(&d->ticket), sizeof(unsigned int)));
  RT_TRY(cudaMemset(d->ticket, 0, sizeof(unsigned int)));
  RT_TRY(cudaMalloc(reinterpret_cast<void **>(&d->tile_counter), sizeof(unsigned long long)));
  RT_TRY(cudaMemset(d->tile_counter, 0, sizeof(unsigned long long)));
  d->ready = true;
  return GSB_OK;
}

int arena_destroy_locked(Device *d) {
  if (!d->va) return GSB_OK;
  cudaSetDevice(d->ordinal);
  if (d->wedged && cudaStreamQuery(d->stream) == cudaErrorNotReady) {
    // unmapping under a kernel that may never end would block for ever: keep the mapping (the process is about to
    // report this GPU Unhealthy or exit; the driver reclaims the memory with the context)
    set_error("%s: arena kept, a wedged launch still uses it", d->uuid);
    return GSB_ERR_TIMEOUT;
  }
  cudaStreamSynchronize(d->stream);
  size_t off = 0;
  for (const Chunk &c : d->chunks) {
    G.cu.cuMemUnmap(d->va + off, c.size);
    G.cu.cuMemRelease(c.handle);
    off += c.size;
  }
  d->chunks.clear();
  G.cu.cuMemAddressFree(d->va, d->va_size);
  d->va = 0;
  d->va_size = 0;
  d->arena_bytes = 0;
  d->transient_arena = false;
  if (d->seed_table) cudaFree(d->seed_table);
  d->seed_table = nullptr;
  d->gen.clear();
  return GSB_OK;
}

int run_probe_locked(Device *d, const gsb_probe_cfg *cfg, gsb_probe_result *out);

int arena_create_locked(Device *d, uint64_t max_bytes, uint64_t keep_free, uint64_t *arena_bytes,
                        gsb_probe_result *fill_res = nullptr) {
  int rc = ensure_ready(d);
  if (rc) return rc;
  if ((rc = arena_destroy_locked(d)) != GSB_OK) return rc;

  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof prop);
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = d->ordinal;
  size_t gran = 0;
  CU_TRY(G.cu.cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM));
  size_t free_b = 0, total_b = 0;
  CU_TRY(G.cu.cuMemGetInfo(&free_b, &total_b));
  uint64_t target = free_b > keep_free ? free_b - keep_free : 0;
  if (max_bytes && max_bytes < target) target = max_bytes;
  target = target / gran * gran;
  if (target == 0) {
    set_error("nothing allocatable on %s (free %zu, keep_free %llu)", d->uuid, free_b,
              (unsigned long long)keep_free);
    return GSB_ERR_OUT_OF_MEMORY;
  }
  CU_TRY(G.cu.cuMemAddressReserve(&d->va, target, 0, 0, 0));
  d->va_size = target;

  // Map physical chunks, largest first, until the driver refuses: what got mapped IS the
  // "actually allocatable" figure.
  const size_t ladder[] = {8ull << 30, 1ull << 30, 128ull << 20, 16ull << 20, 2ull << 20};
  uint64_t mapped = 0;
  for (size_t want : ladder) {
    size_t sz = want / gran * gran;
    if (sz == 0) sz = gran;
    while (mapped + sz <= target) {
      CUmemGenericAllocationHandle h;
      CUresult r = G.cu.cuMemCreate(&h, sz, &prop, 0);
      if (r != CUDA_SUCCESS) break;  // try the next smaller rung
      r = G.cu.cuMemMap(d->va + mapped, sz, 0, h, 0);
      if (r != CUDA_SUCCESS) {
        G.cu.cuMemRelease(h);
        set_error("cuMemMap -> %d (%s)", (int)r, cu_err(r));
        arena_destroy_locked(d);
        return GSB_ERR_DRIVER;
      }
      d->chunks.push_back({h, sz});
      mapped += sz;
    }
  }
  if (mapped == 0) {
    arena_destroy_locked(d);
    set_error("driver refused every allocation on %s", d->uuid);
    return GSB_ERR_OUT_OF_MEMORY;
  }
  CUmemAccessDesc acc;
  memset(&acc, 0, sizeof acc);
  acc.location = prop.location;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  CUresult r = G.cu.cuMemSetAccess(d->va, mapped, &acc, 1);
  if (r != CUDA_SUCCESS) {
    set_error("cuMemSetAccess -> %d (%s)", (int)r, cu_err(r));
    arena_destroy_locked(d);
    return GSB_ERR_DRIVER;
  }
  d->arena_bytes = mapped;
  const size_t n_gran = (size_t)((mapped + kGranuleBytes - 1) / kGranuleBytes);
  d->gen.assign(n_gran, 0u);
  if (cudaMalloc(reinterpret_cast<void **>(&d->seed_table), n_gran * sizeof(uint32_t)) != cudaSuccess) {
    arena_destroy_locked(d);
    set_error("cudaMalloc(seed table) failed");
    return GSB_ERR_OUT_OF_MEMORY;
  }
  cudaMemset(d->seed_table, 0, n_gran * sizeof(uint32_t));

  // First generation: write every word once (proves every mapped byte is writable) so that all
  // later cycles are VERIFY_REFILL.
  gsb_probe_cfg fill;
  memset(&fill, 0, sizeof fill);
  fill.op = GSB_OP_FILL;
  fill.variant = GSB_VARIANT_AUTO;
  fill.seed_write = d->next_gen;
  fill.flags = GSB_PROBE_SEED_TABLE;
  fill.flags = GSB_PROBE_SEED_TABLE | (fill_res ? GSB_PROBE_TIMED : 0u);
  gsb_probe_result res;
  rc = run_probe_locked(d, &fill, &res);
  if (fill_res) *fill_res = res;
  if (rc) {
    arena_destroy_locked(d);
    return rc;
  }
  d->next_gen++;
  if (d->next_gen == 0) d->next_gen = 1;
  if (arena_bytes) *arena_bytes = mapped;
  return GSB_OK;
}

struct ProbeFlight {
  gsb_probe_cfg cfg;
  gsb_launch_geom geom;
  gsb_kernel_args args;
  uint64_t bytes = 0;
  uint64_t t_begin = 0;
  bool timed = false;
  bool launched = false;
};

// validate + enqueue (does not wait)
int probe_begin_locked(Device *d, const gsb_probe_cfg *cfg, gsb_probe_result *out, ProbeFlight *fl) {
  fl->t_begin = now_ns();
  fl->cfg = *cfg;
  memset(out, 0, sizeof *out);
  out->first_bad_offset = UINT64_MAX;
  int rc = ensure_ready(d);
  if (rc) return out->status = rc;
  if (!d->va) {
    set_error("no arena on %s: call gsb_arena_create first", d->uuid);
    return out->status = GSB_ERR_NO_ARENA;
  }
  if (d->wedged) {  // a launch that outlived the watchdog: queue nothing behind it until it has drained
    if (cudaStreamQuery(d->stream) == cudaErrorNotReady) {
      set_error("%s: an earlier probe launch is still running (wedged)", d->uuid);
      return out->status = GSB_ERR_TIMEOUT;
    }
    d->wedged = false;
  }
  if (cfg->op < GSB_OP_FILL || cfg->op > GSB_OP_VERIFY_REFILL || (cfg->window_offset & 15) ||
      (cfg->window_bytes & 15) || cfg->window_offset > d->arena_bytes) {
    set_error("invalid probe window/op (op %u, offset %llu, bytes %llu)", cfg->op,
              (unsigned long long)cfg->window_offset, (unsigned long long)cfg->window_bytes);
    return out->status = GSB_ERR_INVALID_ARGUMENT;
  }
  const uint64_t bytes = cfg->window_bytes ? cfg->window_bytes : d->arena_bytes - cfg->window_offset;
  if (cfg->window_offset + bytes > d->arena_bytes) {
    set_error("probe window [%llu, +%llu) exceeds arena of %llu bytes", (unsigned long long)cfg->window_offset,
              (unsigned long long)bytes, (unsigned long long)d->arena_bytes);
    return out->status = GSB_ERR_INVALID_ARGUMENT;
  }
  const bool table = (cfg->flags & GSB_PROBE_SEED_TABLE) != 0;
  if (table && (cfg->window_offset & 0xFFFF)) {
    set_error("seed-table probes need a 64 KiB aligned window offset");
    return out->status = GSB_ERR_INVALID_ARGUMENT;
  }
  // occupancy + function attributes are queried once per (op, variant, grid) and device, not per launch
  const uint64_t gkey = ((uint64_t)cfg->op << 48) | ((uint64_t)cfg->variant << 32) | cfg->grid_ctas;
  int e = 0;
  auto git = d->geoms.find(gkey);
  if (git != d->geoms.end()) {
    fl->geom = git->second;
  } else {
    e = gsb_kernel_geometry(cfg->op, cfg->variant, cfg->grid_ctas, (int)d->sm_count, &fl->geom);
    if (!e) d->geoms.emplace(gkey, fl->geom);
  }
  if (e) {
    set_error("kernel geometry: %s", cudaGetErrorString((cudaError_t)e));
    return out->status = (e == (int)cudaErrorInvalidDeviceFunction || e == (int)cudaErrorNoKernelImageForDevice)
                             ? GSB_ERR_UNSUPPORTED_ARCH
                             : GSB_ERR_DRIVER;
  }
  gsb_kernel_args &a = fl->args;
  memset(&a, 0, sizeof a);
  a.base = reinterpret_cast<uint4 *>(d->va);
  a.first_word = cfg->window_offset >> 4;
  a.n_words = bytes >> 4;
  a.seed_expect = cfg->seed_expect;
  a.seed_write = cfg->seed_write;
  a.seed_table = table ? d->seed_table : nullptr;
  a.table_update = (table && cfg->op != GSB_OP_VERIFY) ? d->seed_table : nullptr;
  a.arena_words = d->arena_bytes >> 4;
  a.granule_shift = kGranuleShiftWords;
  a.launch_seq = ++d->launch_seq;
  a.partials = d->partials;
  a.ticket = d->ticket;
  a.tile_counter = d->tile_counter;
  a.out = d->out_dev;
  fl->bytes = bytes;
  fl->timed = (cfg->flags & GSB_PROBE_TIMED) != 0;
  if (bytes > 0) {
    if (fl->timed) RT_TRY(cudaEventRecord(d->ev0, d->stream));
    e = gsb_kernel_launch(cfg->op, &fl->geom, &a, d->stream);
    if (e) {
      set_error("kernel launch: %s", cudaGetErrorString((cudaError_t)e));
      return out->status = GSB_ERR_DRIVER;
    }
    if (fl->timed) RT_TRY(cudaEventRecord(d->ev1, d->stream));
    fl->launched = true;
  }
  return GSB_OK;
}

// wait for the launch and collect what the last CTA wrote into pinned host memory
//
// Three phases, none of which can park the thread for ever:
//   1. spin on the sequence word the last CTA stores into pinned host memory (option GSB_OPT_WAIT_SPIN_US, default
//      2000; a prober thread with a period >= 10 ms passes 0): a sleeping wait costs 10-30 us of wake-up latency, a
//      tenth of a 1 GiB-window cycle, which matters to a caller cycling back to back and not at all to a 1 Hz prober
//      inside a 1-CPU pod (device-plugin-ds.yaml:34-40);
//   2. sleep-poll the same word (50 us naps, the stream queried every ~1 ms so a faulted launch is noticed) against
//      the completion watchdog: GSB_OPT_WATCHDOG_MS (default 2000) + 1 ns per 10 window bytes (10 GB/s is "wedged").
//      The reference's WaitForEvent returns every 5 s whatever the GPU does (nvidia.go:126); a kernel that never
//      finishes must not keep this thread — and the GPU's Healthy flag — for ever;
//   3. cudaStreamSynchronize, which by then returns at once and orders the events.
thread_local bool tl_wait_blocking = false;  // set by prober threads that have milliseconds to spare

int probe_end_locked(Device *d, ProbeFlight *fl, gsb_probe_result *out) {
  const gsb_probe_cfg *cfg = &fl->cfg;
  const gsb_kernel_args &a = fl->args;
  if (fl->launched) {
    const volatile uint32_t *flag = &d->out_host->done_flag;
    const uint64_t spin_ns = tl_wait_blocking ? 0 : G.wait_spin_us.load(std::memory_order_relaxed) * 1000ull;
    if (spin_ns) {
      const uint64_t deadline = now_ns() + spin_ns;
      while (*flag != a.launch_seq) {
        for (int i = 0; i < 8; i++) __builtin_ia32_pause();
        if (now_ns() > deadline) break;
      }
    }
    const uint64_t wd_ms = G.watchdog_ms.load(std::memory_order_relaxed);
    if (wd_ms && *flag != a.launch_seq) {
      const uint64_t budget = wd_ms * 1000000ull + fl->bytes / 10;
      const uint64_t deadline = fl->t_begin + budget;
      unsigned naps = 0;
      while (*flag != a.launch_seq) {
        if ((++naps & 15u) == 0 && cudaStreamQuery(d->stream) != cudaErrorNotReady) break;  // finished or faulted
        if (now_ns() > deadline) {
          d->wedged = true;  // the launch is still on the stream: nothing new is queued behind it
          set_error("probe kernel on %s did not finish within %llu ms: device wedged?", d->uuid,
                    (unsigned long long)(budget / 1000000ull));
          out->wall_ns = now_ns() - fl->t_begin;
          return out->status = GSB_ERR_TIMEOUT;
        }
        struct timespec ts = {0, 50000};
        nanosleep(&ts, nullptr);
      }
    }
    cudaError_t se = cudaStreamSynchronize(d->stream);
    if (se != cudaSuccess) {
      set_error("probe kernel failed: %s", cudaGetErrorString(se));
      return out->status = GSB_ERR_DRIVER;
    }
    gsb_kernel_out ko;
    memcpy(&ko, d->out_host, sizeof ko);  // written by the last CTA; the stream sync above orders it
    if (ko.done_flag != a.launch_seq || ko.words_done != a.n_words) {
      set_error("probe kernel did not complete the window (seq %u/%u, words %llu/%llu)", ko.done_flag,
                a.launch_seq, ko.words_done, a.n_words);
      return out->status = GSB_ERR_DRIVER;
    }
    out->mismatch_words = ko.mismatch_words;
    out->mismatch_bits = ko.mismatch_bits;
    out->first_bad_offset = ko.first_bad_word == ~0ull ? UINT64_MAX : ko.first_bad_word << 4;
    out->checksum_xor = ko.checksum_xor;
    out->checksum_sum = ko.checksum_sum;
    if (fl->timed) {
      float ms = 0.f;
      RT_TRY(cudaEventElapsedTime(&ms, d->ev0, d->ev1));
      out->kernel_ns = (uint64_t)((double)ms * 1e6);
    }
    if (a.table_update) {  // host mirror of what the kernel's last CTA wrote
      const uint64_t g0 = (cfg->window_offset + kGranuleBytes - 1) / kGranuleBytes;
      const uint64_t g1 = (cfg->window_offset + fl->bytes) / kGranuleBytes;
      const bool tail = cfg->window_offset + fl->bytes == d->arena_bytes && (d->arena_bytes % kGranuleBytes);
      for (uint64_t g = g0; g < g1 + (tail ? 1 : 0) && g < d->gen.size(); g++) d->gen[g] = cfg->seed_write;
    }
  }
  out->variant = fl->geom.variant;
  out->grid_ctas = fl->geom.grid;
  out->block_threads = fl->geom.block;
  out->bytes_walked = fl->bytes;
  out->bytes_read = cfg->op == GSB_OP_FILL ? 0 : fl->bytes;
  out->bytes_written = cfg->op == GSB_OP_VERIFY ? 0 : fl->bytes;
  out->wall_ns = now_ns() - fl->t_begin;
  return out->status = GSB_OK;
}

int run_probe_locked(Device *d, const gsb_probe_cfg *cfg, gsb_probe_result *out) {
  ProbeFlight fl;
  int rc = probe_begin_locked(d, cfg, out, &fl);
  if (rc) return rc;
  return probe_end_locked(d, &fl, out);
}

// diagnostic knob GSB_NVML_SERIAL=1: one NVML/driver query at a time across this process's device threads
// (GSB_INVENTORY_LIVE only; profiles/node_cycle_8gpu_bimodal_r01.txt)
std::mutex g_nvml_serial_mu;
const bool kNvmlSerial = [] {
  const char *e = getenv("GSB_NVML_SERIAL");
  return e && atoi(e) != 0;
}();

// "GPU-xxxxxxxx-xxxx-xxxx-xxxx-xxxxxxxxxxxx" -> the 16 bytes cuDeviceGetUuid reports for the same device
bool parse_uuid(const char *s, unsigned char out[16]) {
  if (strncmp(s, "GPU-", 4) != 0) return false;
  s += 4;
  int n = 0;
  auto hex = [](char c) -> int {
    if (c >= '0' && c <= '9') return c - '0';
    if (c >= 'a' && c <= 'f') return c - 'a' + 10;
    if (c >= 'A' && c <= 'F') return c - 'A' + 10;
    return -1;
  };
  while (*s && n < 16) {
    if (*s == '-') {
      s++;
      continue;
    }
    const int hi = hex(s[0]), lo = hi < 0 ? -1 : hex(s[1]);
    if (lo < 0) return false;
    out[n++] = (unsigned char)(hi << 4 | lo);
    s += 2;
  }
  return n == 16 && *s == 0;
}

void fill_static_info(const Device *d, gsb_device_info *out) {
  snprintf(out->bus_id, sizeof out->bus_id, "%s", d->bus_id);
  out->cuda_ordinal = d->ordinal;
  out->sm_count = d->sm_count;
  out->cc_major = d->cc_major;
  out->cc_minor = d->cc_minor;
  out->cuda_total_bytes = d->cuda_total;
}

// LIVE inventory of one device: the reference's source (NVML UUID, minor, MemoryInfo v1) re-read and the identity
// cross-checked against the CUDA driver. This is what nvml.NewDevice does at every plugin (re)start
// (server.go:39 -> nvidia.go:60); it also rewrites the device's snapshot.
int query_info(Device *d, gsb_device_info *out) {
  memset(out, 0, sizeof *out);
  std::unique_lock<std::mutex> serial(g_nvml_serial_mu, std::defer_lock);
  if (kNvmlSerial) serial.lock();
  char uuid[GSB_UUID_BUFFER_SIZE] = {0};
  ML_TRY(G.ml.getUUID(d->nvml, uuid, GSB_UUID_BUFFER_SIZE));
  unsigned minor = 0;
  ML_TRY(G.ml.getMinor(d->nvml, &minor));
  nvmlMemory_t mem;
  memset(&mem, 0, sizeof mem);
  ML_TRY(G.ml.getMemoryInfo(d->nvml, &mem));
  if (d->ordinal >= 0) {
    CUuuid cu;
    CU_TRY(G.cu.cuDeviceGetUuid(&cu, d->cudev));
    char cuda_uuid[GSB_UUID_BUFFER_SIZE];
    format_uuid(cu, cuda_uuid);
    if (strcmp(cuda_uuid, uuid) != 0) {
      set_error("identity mismatch on minor %u: CUDA %s vs NVML %s", d->minor, cuda_uuid, uuid);
      return GSB_ERR_IDENTITY_MISMATCH;
    }
  }
  snprintf(out->uuid, sizeof out->uuid, "%s", uuid);
  fill_static_info(d, out);
  out->minor = minor;
  out->total_bytes = mem.total;
  out->total_mib = mem.total / (1024ull * 1024ull);  // bindings.go:346-349
  out->free_bytes = mem.free;
  {
    std::lock_guard<std::mutex> lk(d->smu);
    Snapshot &sn = d->snap;
    snprintf(sn.uuid, sizeof sn.uuid, "%s", uuid);
    sn.uuid_parsed = parse_uuid(uuid, sn.uuid_bytes);
    sn.minor = minor;
    sn.total = mem.total;
    sn.free = mem.free;
    sn.taken_ns = now_ns();
    sn.refreshes++;
  }
  return GSB_OK;
}

// SNAPSHOT inventory: identity/total as NVML reported them at the last live query, with the identity re-validated
// against the CUDA driver on every call (cuDeviceGetUuid is answered by the user-mode driver: no ioctl, no
// driver-wide lock, ~0.1 us — unlike nvmlDeviceGetMemoryInfo, which serialises with every other NVML client of the
// box: 6 us idle, 0.2-2.3 ms beside an nvidia-smi or dcgm-exporter poller, BENCH_r01 e2e.inventory_us_per_step).
int snapshot_info(Device *d, gsb_device_info *out, uint64_t *age_ns) {
  memset(out, 0, sizeof *out);
  Snapshot sn;
  {
    std::lock_guard<std::mutex> lk(d->smu);
    sn = d->snap;
  }
  if (sn.refreshes == 0) return query_info(d, out);  // never queried: take the live path once
  if (d->ordinal >= 0 && sn.uuid_parsed) {
    CUuuid cu;
    CU_TRY(G.cu.cuDeviceGetUuid(&cu, d->cudev));
    if (memcmp(cu.bytes, sn.uuid_bytes, 16) != 0) {
      char cuda_uuid[GSB_UUID_BUFFER_SIZE];
      format_uuid(cu, cuda_uuid);
      set_error("identity mismatch on minor %u: CUDA %s vs NVML snapshot %s", sn.minor, cuda_uuid, sn.uuid);
      return GSB_ERR_IDENTITY_MISMATCH;
    }
  }
  memcpy(out->uuid, sn.uuid, sizeof out->uuid);
  fill_static_info(d, out);
  out->minor = sn.minor;
  out->total_bytes = sn.total;
  out->total_mib = sn.total / (1024ull * 1024ull);
  out->free_bytes = sn.free;
  if (age_ns) *age_ns = now_ns() - sn.taken_ns;
  return GSB_OK;
}

// Run a Job on the device's own persistent thread (created on first use). Hand-off is spin-then-block in both
// directions: a node cycle every few hundred microseconds never pays a futex wake-up (tens of us per hop, a tenth
// of a 1 GiB-window cycle), an idle daemon's workers park after ~200 us. The job is plain data (no std::function,
// no allocation per hand-off).
// knob GSB_WORKER_SPIN_US (default 200; 0 = pure condition-variable hand-off)
const uint64_t kSpinNs = [] {
  const char *e = getenv("GSB_WORKER_SPIN_US");
  return (uint64_t)(e ? atoi(e) : 200) * 1000ull;
}();

int cycle_impl(Device *d, uint32_t idx, uint64_t cycle_no, uint64_t window_bytes, int unit_gib, uint32_t variant,
               uint8_t *lw_buf, size_t lw_cap, bool encode_lw, gsb_cycle_result *out);

void run_job(Device *d, Job *j) {  // on the worker thread; the submitting call holds G.api_mu (shared) throughout
  switch (j->kind) {
    case Job::PROBE: {
      std::lock_guard<std::mutex> lk(d->mu);
      j->rc = run_probe_locked(d, j->cfg, j->probe_out);
      break;
    }
    case Job::CYCLE:
      // the node cycle's join re-encodes the whole node's list: the per-device list is not built here
      j->rc = cycle_impl(d, j->idx, j->cycle_no, j->window_bytes, j->unit_gib, j->variant, nullptr, 0, false,
                         j->cycle_out);
      break;
    default:
      j->rc = GSB_ERR_INVALID_ARGUMENT;
  }
}

void worker_submit(Device *d, const Job &job) {
  std::unique_lock<std::mutex> lk(d->wmu);
  if (!d->worker.joinable()) {
    d->worker = std::thread([d] {
      for (;;) {
        // spin for a job first
        const uint64_t until = now_ns() + kSpinNs;
        while (!d->job_flag.load(std::memory_order_acquire) && !d->quit_flag.load(std::memory_order_acquire) &&
               now_ns() < until)
          __builtin_ia32_pause();
        std::unique_lock<std::mutex> wl(d->wmu);
        d->wcv.wait(wl, [d] { return d->job_ready || d->worker_quit; });
        if (d->worker_quit) return;
        d->job_ready = false;
        d->job_flag.store(false, std::memory_order_relaxed);
        wl.unlock();
        run_job(d, &d->job);  // the submitter does not touch d->job until job_done
        wl.lock();
        d->job_done = true;
        d->done_flag.store(true, std::memory_order_release);
        d->wcv.notify_all();
      }
    });
  }
  d->job = job;
  d->job_done = false;
  d->done_flag.store(false, std::memory_order_relaxed);
  d->job_ready = true;
  d->job_flag.store(true, std::memory_order_release);
  d->wcv.notify_all();
}

int worker_wait(Device *d) {
  const uint64_t until = now_ns() + 5 * kSpinNs;
  while (!d->done_flag.load(std::memory_order_acquire) && now_ns() < until) __builtin_ia32_pause();
  std::unique_lock<std::mutex> lk(d->wmu);
  d->wcv.wait(lk, [d] { return d->job_done; });
  return d->job.rc;
}

void worker_stop(Device *d) {
  {
    std::lock_guard<std::mutex> lk(d->wmu);
    d->worker_quit = true;
    d->quit_flag.store(true, std::memory_order_release);
  }
  d->wcv.notify_all();
  if (d->worker.joinable()) d->worker.join();
}

void push_event(const gsb_event &ev) {
  {
    std::lock_guard<std::mutex> lk(G.hmu);
    G.events.push_back(ev);
  }
  G.hcv.notify_all();
}

void wake_health_waiters() {  // whether or not the internal threads are running
  {
    std::lock_guard<std::mutex> lk(G.hmu);
    G.stop_gen++;
  }
  G.hcv.notify_all();
}

int health_stop_locked() {  // the caller holds G.life_mu
  std::vector<std::thread> ts;
  {
    std::lock_guard<std::mutex> lk(G.mu);
    if (!G.health_running) return GSB_OK;
    G.health_stop = true;
    ts.swap(G.health_threads);
    G.health_running = false;
  }
  for (auto &t : ts) t.join();
  if (G.have_event_set) {
    G.ml.eventSetFree(G.event_set);
    G.have_event_set = false;
  }
  std::lock_guard<std::mutex> lk(G.hmu);
  G.events.clear();
  G.health_stop = false;
  return GSB_OK;
}

}  // namespace

// ====================================================================== C ABI

extern "C" {

int gsb_abi_version(void) { return (int)GSB_ABI_VERSION; }

const char *gsb_strerror(int status) {
  switch (status) {
    case GSB_OK: return "ok";
    case GSB_ERR_NOT_INITIALIZED: return "not initialized";
    case GSB_ERR_INVALID_ARGUMENT: return "invalid argument";
    case GSB_ERR_LIBRARY_NOT_FOUND: return "could not load NVML library";
    case GSB_ERR_DRIVER: return "CUDA driver error";
    case GSB_ERR_NVML: return "NVML error";
    case GSB_ERR_NO_DEVICE: return "nvml: device not found";
    case GSB_ERR_IDENTITY_MISMATCH: return "CUDA/NVML device identity mismatch";
    case GSB_ERR_BUFFER_TOO_SMALL: return "buffer too small";
    case GSB_ERR_OUT_OF_MEMORY: return "out of device memory";
    case GSB_ERR_UNSUPPORTED_ARCH: return "device is not sm_100: no kernel image, no fallback";
    case GSB_ERR_TIMEOUT: return "timeout";
    case GSB_ERR_NO_ARENA: return "no probe arena";
    case GSB_ERR_MALFORMED: return "malformed protobuf";
    case GSB_ERR_STOPPED: return "health queue stopped";
    default: return "unknown gsb status";
  }
}

int gsb_last_error(char *buf, size_t cap) {
  if (!buf || cap == 0) return GSB_ERR_INVALID_ARGUMENT;
  snprintf(buf, cap, "%s", tl_error);
  return GSB_OK;
}

int gsb_init(void) {
  std::unique_lock<std::shared_mutex> api_lk(G.api_mu);
  std::lock_guard<std::mutex> lk(G.mu);
  if (G.inited) return GSB_OK;
  int rc = load_libraries();
  if (rc) return rc;
  ML_TRY(G.ml.init());
  CU_TRY(G.cu.cuInit(0));

  unsigned n_ml = 0;
  ML_TRY(G.ml.getCount(&n_ml));
  int n_cu = 0;
  RT_TRY(cudaGetDeviceCount(&n_cu));
  struct CudaDev {
    CUdevice dev;
    char uuid[GSB_UUID_BUFFER_SIZE];
  };
  std::vector<CudaDev> cds((size_t)n_cu);
  for (int i = 0; i < n_cu; i++) {
    CU_TRY(G.cu.cuDeviceGet(&cds[i].dev, i));
    CUuuid u;
    CU_TRY(G.cu.cuDeviceGetUuid(&u, cds[i].dev));
    format_uuid(u, cds[i].uuid);
  }
  G.devs.clear();
  for (unsigned i = 0; i < n_ml; i++) {  // NVML index order = the reference's order (nvidia.go:59)
    auto d = std::make_unique<Device>();
    ML_TRY(G.ml.handleByIndex(i, &d->nvml));
    ML_TRY(G.ml.getUUID(d->nvml, d->uuid, GSB_UUID_BUFFER_SIZE));
    unsigned minor = 0;
    ML_TRY(G.ml.getMinor(d->nvml, &minor));
    d->minor = minor;
    nvmlPciInfo_t pci;
    memset(&pci, 0, sizeof pci);
    ML_TRY(G.ml.getPciInfo(d->nvml, &pci));
    snprintf(d->bus_id, sizeof d->bus_id, "%s", pci.busId);
    for (int c = 0; c < n_cu; c++) {
      if (strcmp(cds[c].uuid, d->uuid) == 0) {
        d->ordinal = c;
        d->cudev = cds[c].dev;
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, c);
        d->sm_count = (uint32_t)v;
        cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, c);
        d->cc_major = (uint32_t)v;
        cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, c);
        d->cc_minor = (uint32_t)v;
        size_t tot = 0;
        G.cu.cuDeviceTotalMem(&tot, d->cudev);
        d->cuda_total = tot;
        break;
      }
    }
    G.devs.push_back(std::move(d));
  }
  // the (re)start-time inventory: every device's identity + memory read from NVML once, as getDevices does
  for (auto &d : G.devs) {
    gsb_device_info info;
    int qrc = query_info(d.get(), &info);
    if (qrc) {
      G.devs.clear();
      return qrc;
    }
  }
  if (const char *e = getenv("GSB_PROBE_WATCHDOG_MS")) G.watchdog_ms = (uint64_t)atoll(e);
  if (const char *e = getenv("GSB_INVENTORY_POLICY")) G.inventory_policy = strcmp(e, "live") == 0 ? GSB_INVENTORY_LIVE : GSB_INVENTORY_SNAPSHOT;
  G.inited = true;
  return GSB_OK;
}

int gsb_shutdown(void) {
  wake_health_waiters();
  std::lock_guard<std::mutex> life_lk(G.life_mu);
  health_stop_locked();
  std::unique_lock<std::shared_mutex> api_lk(G.api_mu);  // waits for in-flight calls of other threads
  std::lock_guard<std::mutex> lk(G.mu);
  if (!G.inited) return GSB_OK;
  for (auto &d : G.devs) {
    worker_stop(d.get());
    std::lock_guard<std::mutex> dl(d->mu);
    bool still_wedged = false;
    if (d->ready && d->wedged) {
      cudaSetDevice(d->ordinal);
      still_wedged = cudaStreamQuery(d->stream) == cudaErrorNotReady;
    }
    if (!still_wedged) arena_destroy_locked(d.get());
    if (d->ready && still_wedged) {
      // cudaFree and cudaStreamDestroy wait for the device: under a launch that never ends they would hang the
      // shutdown for ever. The resources go with the process / the context instead.
      d->ready = false;
    }
    if (d->ready) {
      cudaSetDevice(d->ordinal);
      cudaStreamDestroy(d->stream);
      cudaEventDestroy(d->ev0);
      cudaEventDestroy(d->ev1);
      cudaFreeHost(d->out_host);
      cudaFree(d->partials);
      cudaFree(d->ticket);
      cudaFree(d->tile_counter);
      d->ready = false;
    }
  }
  G.devs.clear();
  G.inited = false;
  nvmlReturn_t r = G.ml.shutdown();  // library handles stay open: re-init is cheap and safe
  if (r != NVML_SUCCESS) {
    set_error("nvml: %s", G.ml.errorString(r));
    return GSB_ERR_NVML;
  }
  return GSB_OK;
}

int gsb_device_count(uint32_t *n) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!n) return GSB_ERR_INVALID_ARGUMENT;
  if (!G.inited) {
    set_error("gsb_init has not succeeded");
    return GSB_ERR_NOT_INITIALIZED;
  }
  unsigned c = 0;
  ML_TRY(G.ml.getCount(&c));  // live query, like nvml.GetDeviceCount
  *n = c < G.devs.size() ? c : (uint32_t)G.devs.size();
  return GSB_OK;
}

int gsb_device_info_get(uint32_t idx, gsb_device_info *out) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!out) return GSB_ERR_INVALID_ARGUMENT;
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  int rc = query_info(d, out);
  out->index = idx;
  return rc;
}

int gsb_arena_create(uint32_t idx, uint64_t max_bytes, uint64_t keep_free_bytes, uint64_t *arena_bytes) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->mu);
  return arena_create_locked(d, max_bytes, keep_free_bytes, arena_bytes);
}

int gsb_arena_destroy(uint32_t idx) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->mu);
  return arena_destroy_locked(d);
}

int gsb_arena_bytes(uint32_t idx, uint64_t *arena_bytes) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d || !arena_bytes) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->mu);
  *arena_bytes = d->arena_bytes;
  return d->va ? GSB_OK : GSB_ERR_NO_ARENA;
}

int gsb_probe(uint32_t idx, const gsb_probe_cfg *cfg, gsb_probe_result *out) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!cfg || !out) return GSB_ERR_INVALID_ARGUMENT;
  Device *d = device_at(idx);
  if (!d) {
    memset(out, 0, sizeof *out);
    return out->status = G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  }
  std::lock_guard<std::mutex> lk(d->mu);
  return run_probe_locked(d, cfg, out);
}

int gsb_probe_all(uint32_t n, const uint32_t *idxs, const gsb_probe_cfg *cfg, gsb_probe_result *results) {
  if (!idxs || !cfg || !results || n > GSB_MAX_DEVICES) return GSB_ERR_INVALID_ARGUMENT;
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);  // held across the fan-out: a shutdown waits for it
  std::lock_guard<std::mutex> one(G.all_mu);             // each device worker has one job slot
  Device *ds[GSB_MAX_DEVICES];
  for (uint32_t i = 0; i < n; i++) {
    ds[i] = device_at(idxs[i]);
    for (uint32_t k = 0; k < i && ds[i]; k++)
      if (ds[k] == ds[i]) ds[i] = nullptr;  // a device listed twice runs once; the second slot reports the error
    if (!ds[i]) {
      memset(&results[i], 0, sizeof results[i]);
      results[i].status = !G.inited ? GSB_ERR_NOT_INITIALIZED : idxs[i] < G.devs.size() ? GSB_ERR_INVALID_ARGUMENT : GSB_ERR_NO_DEVICE;
      continue;
    }
    Job j;
    j.kind = Job::PROBE;
    j.idx = idxs[i];
    j.cfg = cfg;
    j.probe_out = &results[i];
    worker_submit(ds[i], j);
  }
  int rc = GSB_OK;
  for (uint32_t i = 0; i < n; i++) {
    if (ds[i]) worker_wait(ds[i]);
    if (results[i].status != GSB_OK) rc = results[i].status;
  }
  return rc;
}

int64_t gsb_cycle_all(uint32_t n, const uint32_t *idxs, uint64_t cycle_no, uint64_t window_bytes, int unit_gib,
                      uint32_t variant, uint8_t *lw_buf, size_t lw_cap, gsb_cycle_result *results) {
  if (!idxs || !results || n == 0 || n > GSB_MAX_DEVICES) return GSB_ERR_INVALID_ARGUMENT;
  if (window_bytes % kGranuleBytes) {
    set_error("cycle window must be a multiple of 64 MiB (or 0 = whole arena)");
    return GSB_ERR_INVALID_ARGUMENT;
  }
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  std::lock_guard<std::mutex> one(G.all_mu);
  Device *ds[GSB_MAX_DEVICES];
  int rcs[GSB_MAX_DEVICES];
  for (uint32_t i = 0; i < n; i++) {
    ds[i] = device_at(idxs[i]);
    if (!ds[i]) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
    for (uint32_t k = 0; k < i; k++)
      if (ds[k] == ds[i]) {
        set_error("device %u listed twice", idxs[i]);
        return GSB_ERR_INVALID_ARGUMENT;
      }
  }
  for (uint32_t i = 0; i < n; i++) {  // fan out: every device runs its own cycle on its own thread
    Job j;
    j.kind = Job::CYCLE;
    j.idx = idxs[i];
    j.cycle_no = cycle_no;
    j.window_bytes = window_bytes;
    j.unit_gib = unit_gib;
    j.variant = variant;
    j.cycle_out = &results[i];
    worker_submit(ds[i], j);
  }
  for (uint32_t i = 0; i < n; i++) rcs[i] = worker_wait(ds[i]);
  // the one join: concatenate in index order, slices from the first device, health from each verdict
  const uint32_t slices = results[0].slices;
  const char *uuids[GSB_MAX_DEVICES];
  bool any_bad = false;
  int rc_all = GSB_OK;
  for (uint32_t i = 0; i < n; i++) {
    // a failed or timed-out launch is a verdict (healthy = 0), not an API error
    if (rcs[i] < 0 && rcs[i] != GSB_ERR_DRIVER && rcs[i] != GSB_ERR_TIMEOUT) rc_all = rcs[i];
    uuids[i] = results[i].info.uuid;
    if (!results[i].healthy) any_bad = true;
  }
  if (rc_all) return rc_all;
  if (any_bad) {
    G.join_bits.assign(((size_t)n * slices + 7) / 8, 0);
    for (uint32_t i = 0; i < n; i++)
      if (!results[i].healthy)
        for (uint32_t j = 0; j < slices; j++) {  // every fake device of that GPU (nvidia.go:146-150)
          const size_t b = (size_t)i * slices + j;
          G.join_bits[b >> 3] |= (uint8_t)(1u << (b & 7));
        }
  }
  const int64_t len = gsb_encode_list_and_watch(uuids, n, slices, any_bad ? G.join_bits.data() : nullptr, lw_buf, lw_cap);
  if (len >= 0)
    for (uint32_t i = 0; i < n; i++) results[i].lw_len = i == 0 ? len : 0;  // the node's list is reported once
  return len;
}

int gsb_arena_read(uint32_t idx, uint64_t offset, void *dst, uint64_t bytes) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d || !dst) return GSB_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lk(d->mu);
  if (!d->va) return GSB_ERR_NO_ARENA;
  if (offset + bytes > d->arena_bytes) return GSB_ERR_INVALID_ARGUMENT;
  RT_TRY(cudaSetDevice(d->ordinal));
  RT_TRY(cudaMemcpy(dst, reinterpret_cast<const void *>(d->va + offset), bytes, cudaMemcpyDeviceToHost));
  return GSB_OK;
}

int gsb_arena_write(uint32_t idx, uint64_t offset, const void *src, uint64_t bytes) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d || !src) return GSB_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lk(d->mu);
  if (!d->va) return GSB_ERR_NO_ARENA;
  if (offset + bytes > d->arena_bytes) return GSB_ERR_INVALID_ARGUMENT;
  RT_TRY(cudaSetDevice(d->ordinal));
  RT_TRY(cudaMemcpy(reinterpret_cast<void *>(d->va + offset), src, bytes, cudaMemcpyHostToDevice));
  return GSB_OK;
}

int gsb_cycle(uint32_t idx, uint64_t cycle_no, uint64_t window_bytes, int unit_gib, uint32_t variant,
              uint8_t *lw_buf, size_t lw_cap, gsb_cycle_result *out) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!out) return GSB_ERR_INVALID_ARGUMENT;
  memset(out, 0, sizeof *out);
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  return cycle_impl(d, idx, cycle_no, window_bytes, unit_gib, variant, lw_buf, lw_cap, true, out);
}

int gsb_set_option(uint32_t key, uint64_t value) {
  switch (key) {
    case GSB_OPT_INVENTORY_POLICY:
      if (value != GSB_INVENTORY_SNAPSHOT && value != GSB_INVENTORY_LIVE) return GSB_ERR_INVALID_ARGUMENT;
      G.inventory_policy = value;
      return GSB_OK;
    case GSB_OPT_WAIT_SPIN_US: G.wait_spin_us = value; return GSB_OK;
    case GSB_OPT_WATCHDOG_MS: G.watchdog_ms = value; return GSB_OK;
    case GSB_OPT_INVENTORY_REFRESH_MS: G.inventory_refresh_ms = value; return GSB_OK;
    case GSB_OPT_TRANSIENT_KEEP_FREE_BYTES: G.transient_keep_free = value; return GSB_OK;
    case GSB_OPT_SWEEP_EVERY_CYCLES: G.sweep_every = value; return GSB_OK;
    default: set_error("unknown option %u", key); return GSB_ERR_INVALID_ARGUMENT;
  }
}

int gsb_get_option(uint32_t key, uint64_t *value) {
  if (!value) return GSB_ERR_INVALID_ARGUMENT;
  switch (key) {
    case GSB_OPT_INVENTORY_POLICY: *value = G.inventory_policy; return GSB_OK;
    case GSB_OPT_WAIT_SPIN_US: *value = G.wait_spin_us; return GSB_OK;
    case GSB_OPT_WATCHDOG_MS: *value = G.watchdog_ms; return GSB_OK;
    case GSB_OPT_INVENTORY_REFRESH_MS: *value = G.inventory_refresh_ms; return GSB_OK;
    case GSB_OPT_TRANSIENT_KEEP_FREE_BYTES: *value = G.transient_keep_free; return GSB_OK;
    case GSB_OPT_SWEEP_EVERY_CYCLES: *value = G.sweep_every; return GSB_OK;
    default: set_error("unknown option %u", key); return GSB_ERR_INVALID_ARGUMENT;
  }
}

int gsb_health_stats_get(uint32_t idx, gsb_health_stats *out) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!out) return GSB_ERR_INVALID_ARGUMENT;
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->smu);
  *out = d->hstats;
  return GSB_OK;
}

int gsb_inventory_refresh(uint32_t idx) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!G.inited) return GSB_ERR_NOT_INITIALIZED;
  gsb_device_info info;
  if (idx == GSB_ALL_DEVICES) {
    for (auto &d : G.devs) {
      int rc = query_info(d.get(), &info);
      if (rc) return rc;
    }
    return GSB_OK;
  }
  Device *d = device_at(idx);
  if (!d) return GSB_ERR_NO_DEVICE;
  return query_info(d, &info);
}

int gsb_inventory_snapshot(uint32_t idx, gsb_device_info *out, uint64_t *age_ns) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!out) return GSB_ERR_INVALID_ARGUMENT;
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  int rc = snapshot_info(d, out, age_ns);
  out->index = idx;
  return rc;
}

int gsb_test_stall(uint32_t idx, uint32_t ms) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->mu);
  int rc = ensure_ready(d);
  if (rc) return rc;
  const int e = gsb_kernel_stall((unsigned long long)ms * 1000000ull, d->stream);
  if (e) {
    set_error("stall kernel: %s", cudaGetErrorString((cudaError_t)e));
    return GSB_ERR_DRIVER;
  }
  return GSB_OK;
}

int gsb_test_skew_snapshot(uint32_t idx, uint64_t total_bytes) {
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  Device *d = device_at(idx);
  if (!d) return G.inited ? GSB_ERR_NO_DEVICE : GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(d->smu);
  d->snap.total = total_bytes;
  return GSB_OK;
}

}  // extern "C"

namespace {

// One inventory + health-probe cycle of one device. The caller holds G.api_mu (shared).
int cycle_impl(Device *d, uint32_t idx, uint64_t cycle_no, uint64_t window_bytes, int unit_gib, uint32_t variant,
               uint8_t *lw_buf, size_t lw_cap, bool encode_lw, gsb_cycle_result *out) {
  memset(out, 0, sizeof *out);
  if (window_bytes % kGranuleBytes) {
    set_error("cycle window must be a multiple of 64 MiB (or 0 = whole arena)");
    return GSB_ERR_INVALID_ARGUMENT;
  }
  std::lock_guard<std::mutex> lk(d->mu);
  // Transient window (SURVEY §7 hard-part 2, the tenant-safe steady state): with no standing arena the cycle
  // allocates the window, fills it, verifies it and gives it back, so between cycles the plugin holds no HBM beyond
  // its CUDA context and the 179 advertised slices are not oversold. "Nothing free to probe" (tenants hold the
  // HBM) is not a GPU fault.
  if (d->va && d->transient_arena) {
    // a transient window that a wedged launch kept mapped: give it back now if the stream has drained, otherwise this
    // cycle's verdict is the same wedge (nothing new is queued, nothing more is allocated)
    if (d->wedged && cudaStreamQuery(d->stream) != cudaErrorNotReady) d->wedged = false;
    if (arena_destroy_locked(d) == GSB_OK) d->transient_arena = false;
  }
  const bool leftover = d->va && d->transient_arena;
  const bool transient = !d->va || leftover;
  gsb_probe_result fill_res;
  memset(&fill_res, 0, sizeof fill_res);
  int prc = GSB_OK;
  bool skip_probe = false;
  if (transient) {
    if (window_bytes == 0) {
      set_error("no arena on %s: call gsb_arena_create first (or pass a window for a transient probe)", d->uuid);
      return GSB_ERR_NO_ARENA;
    }
    out->transient = 1;
    uint64_t got = 0;
    if (leftover) {
      set_error("%s: the previous transient window is still held by a wedged launch", d->uuid);
      prc = GSB_ERR_TIMEOUT;
    } else {
      prc = arena_create_locked(d, window_bytes, G.transient_keep_free.load(), &got, &fill_res);
      if (prc != GSB_OK && d->va) d->transient_arena = true;  // could not be unmapped under a wedged launch: retried next cycle
    }
    if (prc == GSB_ERR_OUT_OF_MEMORY) {
      out->probe.status = GSB_ERR_OUT_OF_MEMORY;
      prc = GSB_OK;
      skip_probe = true;
    } else if (prc) {
      out->probe = fill_res;
      out->probe.status = prc;
      skip_probe = true;
    }
  }
  // 1. health: enqueue this cycle's walk (asynchronous). Standing arena: VERIFY_REFILL of the cycle's window.
  //    Transient window: the FILL above wrote generation g, VERIFY reads it back.
  gsb_probe_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.op = transient ? GSB_OP_VERIFY : GSB_OP_VERIFY_REFILL;
  cfg.variant = variant;
  cfg.flags = GSB_PROBE_TIMED | GSB_PROBE_SEED_TABLE;
  if (!transient) {
    if (window_bytes && window_bytes < d->arena_bytes) {
      const uint64_t n_win = d->arena_bytes / window_bytes;
      cfg.window_offset = (cycle_no % n_win) * window_bytes;
      cfg.window_bytes = window_bytes;
    }
    cfg.seed_write = d->next_gen++;
    if (d->next_gen == 0) d->next_gen = 1;
  }
  // diagnostic knob GSB_CYCLE_ORDER (tools/cycle_breakdown.py): 0 = launch, then inventory while the kernel
  // runs (shipped); 1 = inventory first, then launch
  static const int order = [] {
    const char *e = getenv("GSB_CYCLE_ORDER");
    return e ? atoi(e) : 0;
  }();
  ProbeFlight fl;
  if (!skip_probe && order != 1) prc = probe_begin_locked(d, &cfg, &out->probe, &fl);

  // 2. inventory while the kernel walks HBM: identity + total (policy SNAPSHOT: NVML's (re)start-time answer,
  //    identity re-validated on the CUDA side; policy LIVE: a fresh NVML query), slices, S fake devices, wire bytes
  //    (optimistically with the health this device had going into the cycle)
  const uint64_t t0 = now_ns();
  int rc;
  if (G.inventory_policy.load(std::memory_order_relaxed) == GSB_INVENTORY_LIVE) {
    rc = query_info(d, &out->info);
    out->inventory_live = 1;
  } else {
    rc = snapshot_info(d, &out->info, &out->snapshot_age_ns);
  }
  if (rc == GSB_OK) {
    out->info.index = idx;
    out->slices = gsb_slices(out->info.total_mib, unit_gib);
  }
  const char *uuids[1] = {out->info.uuid};
  auto encode = [&](bool unhealthy) -> int64_t {
    if (!encode_lw) return 0;
    const uint8_t *bits = nullptr;
    if (unhealthy) {  // every fake device of a faulted GPU (nvidia.go:146-150)
      d->bits_scratch.assign((out->slices + 7) / 8, 0xFF);
      bits = d->bits_scratch.data();
    }
    return gsb_encode_list_and_watch(uuids, 1, out->slices, bits, lw_buf, lw_cap);
  };
  if (rc == GSB_OK) out->lw_len = encode(d->faulted);
  out->inventory_ns = now_ns() - t0;
  if (!skip_probe && order == 1) prc = probe_begin_locked(d, &cfg, &out->probe, &fl);

  // 3. verdict
  if (!skip_probe && prc == GSB_OK) prc = probe_end_locked(d, &fl, &out->probe);
  if (transient) {
    if (!skip_probe && prc == GSB_OK) {  // one figure for the window: FILL wrote it, VERIFY read it
      out->probe.kernel_ns += fill_res.kernel_ns;
      out->probe.bytes_written = fill_res.bytes_written;
    }
    if (!leftover && d->va && arena_destroy_locked(d) != GSB_OK) d->transient_arena = true;  // wedged: kept, retried next cycle
  }
  if (rc) return rc;
  if (out->lw_len < 0) return (int)out->lw_len;
  out->healthy = (prc == GSB_OK && out->probe.mismatch_words == 0 && !d->faulted) ? 1u : 0u;
  if (!(prc == GSB_OK && out->probe.mismatch_words == 0) && !d->faulted) {
    d->faulted = true;  // sticky (server.go:180 FIXME): the list this cycle reports already carries it
    out->lw_len = encode(true);
    if (out->lw_len < 0) return (int)out->lw_len;
  }
  return prc;
}

}  // namespace

extern "C" {

// ---------------------------------------------------------------------- health

int gsb_xid_is_benign(uint64_t xid) { return xid == 31 || xid == 43 || xid == 45; }

int gsb_health_set_recovery(uint32_t clean_cycles) {
  G.recovery_cycles = clean_cycles;
  return GSB_OK;
}

int gsb_health_inject(const gsb_event *ev) {
  if (!ev) return GSB_ERR_INVALID_ARGUMENT;
  push_event(*ev);
  return GSB_OK;
}

int gsb_health_wait(uint32_t timeout_ms, gsb_event *ev) {
  if (!ev) return GSB_ERR_INVALID_ARGUMENT;
  std::unique_lock<std::mutex> lk(G.hmu);
  const uint64_t gen = G.stop_gen;
  G.hcv.wait_for(lk, std::chrono::milliseconds(timeout_ms), [&] { return !G.events.empty() || G.stop_gen != gen; });
  if (!G.events.empty()) {
    *ev = G.events.front();
    G.events.pop_front();
    return GSB_OK;
  }
  return G.stop_gen != gen ? GSB_ERR_STOPPED : GSB_ERR_TIMEOUT;
}

int gsb_health_start(uint32_t probe_period_ms, uint64_t window_bytes) {
  std::lock_guard<std::mutex> life_lk(G.life_mu);
  std::shared_lock<std::shared_mutex> api_lk(G.api_mu);
  if (!G.inited) return GSB_ERR_NOT_INITIALIZED;
  std::lock_guard<std::mutex> lk(G.mu);
  if (G.health_running) return GSB_OK;
  G.health_stop = false;
  // XID half: one registration per GPU (the reference registers the same GPU once per fake device)
  if (G.ml.eventSetCreate && G.ml.registerEvents && G.ml.eventSetWait && G.ml.eventSetFree) {
    nvmlReturn_t cr = G.ml.eventSetCreate(&G.event_set);
    if (cr != NVML_SUCCESS) {
      set_error("nvml: %s (nvmlEventSetCreate)", G.ml.errorString(cr));
      return GSB_ERR_NVML;
    }
    G.have_event_set = true;
    for (auto &d : G.devs) {
      nvmlReturn_t r = G.ml.registerEvents(d->nvml, nvmlEventTypeXidCriticalError, G.event_set);
      if (r == NVML_ERROR_NOT_SUPPORTED) {
        // nvidia.go:107-112: too old to support health checking -> marked unhealthy
        gsb_event ev;
        memset(&ev, 0, sizeof ev);
        snprintf(ev.uuid, sizeof ev.uuid, "%s", d->uuid);
        ev.etype = GSB_EVENT_XID;
        ev.edata = ~0ull;
        push_event(ev);
      } else if (r != NVML_SUCCESS) {
        // nvidia.go:114-116: any other registration error is fatal (log.Fatalf) — a GPU without XID coverage must
        // not stay silently Healthy. The caller decides what fatal means; nothing is left half started.
        set_error("nvml: %s (nvmlDeviceRegisterEvents on %s)", G.ml.errorString(r), d->uuid);
        G.ml.eventSetFree(G.event_set);
        G.have_event_set = false;
        std::lock_guard<std::mutex> hl(G.hmu);
        G.events.clear();
        return GSB_ERR_NVML;
      }
    }
    G.health_threads.emplace_back([] {
      uint64_t last_refresh = now_ns();
      while (!G.health_stop.load()) {
        // low-rate inventory refresh (GSB_OPT_INVENTORY_REFRESH_MS, default 5000 = the reference's WaitForEvent
        // period; 0 = never): NVML is re-asked off the cycle's path, and an answer that differs from the snapshot
        // (a different GPU behind the handle, a different total) is reported as an event, not papered over
        const uint64_t period = G.inventory_refresh_ms.load() * 1000000ull;
        if (period && now_ns() - last_refresh >= period) {
          last_refresh = now_ns();
          for (auto &d : G.devs) {
            Snapshot before;
            {
              std::lock_guard<std::mutex> sl(d->smu);
              before = d->snap;
            }
            gsb_device_info info;
            const int qrc = query_info(d.get(), &info);
            uint64_t what = 0;
            if (qrc == GSB_ERR_IDENTITY_MISMATCH || (qrc == GSB_OK && strcmp(before.uuid, info.uuid) != 0))
              what = GSB_INVENTORY_IDENTITY_CHANGED;
            else if (qrc == GSB_OK && before.total != info.total_bytes)
              what = GSB_INVENTORY_TOTAL_CHANGED;
            if (what) {
              gsb_event ev;
              memset(&ev, 0, sizeof ev);
              snprintf(ev.uuid, sizeof ev.uuid, "%s", before.uuid);
              ev.etype = GSB_EVENT_INVENTORY;
              ev.edata = what;
              push_event(ev);
            }
          }
        }
        nvmlEventData_t data;
        memset(&data, 0, sizeof data);
        nvmlReturn_t r = G.ml.eventSetWait(G.event_set, &data, 200);
        if (r != NVML_SUCCESS) {
          if (r != NVML_ERROR_TIMEOUT) std::this_thread::sleep_for(std::chrono::milliseconds(200));
          continue;
        }
        if (data.eventType != nvmlEventTypeXidCriticalError) continue;  // nvidia.go:127-129
        gsb_event ev;
        memset(&ev, 0, sizeof ev);
        if (data.device) G.ml.getUUID(data.device, ev.uuid, GSB_UUID_BUFFER_SIZE);
        ev.etype = data.eventType;
        ev.edata = data.eventData;
        push_event(ev);
      }
    });
  }
  // active half: rotate a window probe over each device's arena
  if (probe_period_ms > 0) {
    for (uint32_t i = 0; i < G.devs.size(); i++) {
      G.health_threads.emplace_back([i, probe_period_ms, window_bytes] {
        // a prober with milliseconds between cycles sleeps through the kernel instead of spinning a core: the
        // DaemonSet gives the whole plugin one CPU (device-plugin-ds.yaml:34-40)
        tl_wait_blocking = probe_period_ms >= 10;
        std::vector<uint8_t> buf(1 << 16);
        uint64_t cycle = 0;
        bool reported = false;
        uint32_t clean = 0;
        {
          std::lock_guard<std::mutex> sl(G.devs[i]->smu);
          G.devs[i]->hstats = gsb_health_stats{};
        }
        while (!G.health_stop.load()) {
          gsb_cycle_result cr;
          // every Nth cycle of a device WITHOUT a standing arena is a sweep: a transient window as large as whatever is
          // allocatable right now (minus the keep-free margin) — all free HBM walked, then given back (SURVEY §7
          // hard-part 2: "full walk only at start-up / idle"). With a standing arena the request is just a whole-arena cycle.
          const uint64_t every = G.sweep_every.load(std::memory_order_relaxed);
          const bool sweep = every > 0 && window_bytes > 0 && (cycle + 1) % every == 0;
          const uint64_t t_cycle = now_ns();
          int rc = gsb_cycle(i, cycle++, sweep ? (1ull << 46) : window_bytes, 1, GSB_VARIANT_AUTO, buf.data(), buf.size(), &cr);
          {
            std::lock_guard<std::mutex> sl(G.devs[i]->smu);
            gsb_health_stats &st = G.devs[i]->hstats;
            st.cycles++;
            st.last_bytes_walked = cr.probe.bytes_walked;
            st.last_kernel_ns = cr.probe.kernel_ns;
            if (cr.probe.status == GSB_ERR_OUT_OF_MEMORY) st.skipped++;
            if (!(rc == GSB_OK && cr.probe.mismatch_words == 0) && rc != GSB_ERR_NO_ARENA) st.faults++;
            if (sweep && cr.transient) {
              st.sweeps++;
              st.last_sweep_bytes = cr.probe.bytes_walked;
              st.last_sweep_ns = now_ns() - t_cycle;
            }
          }
          // with no standing arena the cycle probes a transient window (allocate -> fill -> verify -> free); a
          // window that could not be allocated (tenants hold the HBM) is silence, not a fault
          const bool this_cycle_clean = rc == GSB_OK && cr.probe.mismatch_words == 0;
          if (rc != GSB_ERR_NO_ARENA && !this_cycle_clean && !reported) {
            gsb_event ev;
            memset(&ev, 0, sizeof ev);
            snprintf(ev.uuid, sizeof ev.uuid, "%s", G.devs[i]->uuid);
            ev.etype = GSB_EVENT_PROBE;
            ev.edata = rc == GSB_OK ? GSB_PROBE_FAULT_MISMATCH : rc == GSB_ERR_TIMEOUT ? GSB_PROBE_FAULT_WEDGED : GSB_PROBE_FAULT_LAUNCH;
            push_event(ev);
            reported = true;
            clean = 0;
          } else if (reported) {
            clean = this_cycle_clean ? clean + 1 : 0;
            const uint32_t need = G.recovery_cycles.load();
            if (need > 0 && clean >= need) {  // optional recovery: the refills since the fault all verified
              {
                std::lock_guard<std::mutex> dl(G.devs[i]->mu);
                G.devs[i]->faulted = false;
              }
              gsb_event ev;
              memset(&ev, 0, sizeof ev);
              snprintf(ev.uuid, sizeof ev.uuid, "%s", G.devs[i]->uuid);
              ev.etype = GSB_EVENT_PROBE;
              ev.edata = GSB_PROBE_RECOVERED;
              push_event(ev);
              reported = false;
              clean = 0;
            }
          }
          for (uint32_t slept = 0; slept < probe_period_ms && !G.health_stop.load(); slept += 10)
            std::this_thread::sleep_for(std::chrono::milliseconds(10));
        }
      });
    }
  }
  G.health_running = true;
  return GSB_OK;
}

int gsb_health_stop(void) {
  wake_health_waiters();
  std::lock_guard<std::mutex> life_lk(G.life_mu);
  return health_stop_locked();
}

}  // extern "C"
