// context.cu -- process-wide state: device binding, stream, exp table, error strings.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "gibbs.cuh"

namespace kdeb200 {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char *get_error() { return g_err; }

// Slot 0 is the primary context (the device the process is bound to: kdeb200_init / first use); slots 1.. are the
// other GPUs of an in-process multi-GPU set (kdeb200_init_multi).  A host thread that drives one of them binds it with
// ScopedDevice; ctx() then returns that context, so every internal routine works unchanged on any device.
static Context g_ctx[KDEB200_MAX_GPUS];
static int g_nctx = 1;
static thread_local Context *tl_ctx = nullptr;

Context &ctx() { return tl_ctx ? *tl_ctx : g_ctx[0]; }
Context &ctx_at(int slot) { return g_ctx[slot]; }
int multi_count() { return (g_ctx[0].ready && g_nctx > 1) ? g_nctx : 1; }

ScopedDevice::ScopedDevice(int slot) : prev_(tl_ctx) {
  cudaGetDevice(&prev_dev_);
  tl_ctx = &g_ctx[slot];
  cudaSetDevice(g_ctx[slot].device);
}
ScopedDevice::~ScopedDevice() {
  tl_ctx = static_cast<Context *>(prev_);
  cudaSetDevice(prev_dev_);
}

static std::mutex g_mu;

static void drop_context(Context &c) {
  if (!c.ready) return;
  cudaSetDevice(c.device);
  cudaDeviceSynchronize();
  gibbs_drop_schedules(c.slot);
  gibbs_batch_drop(c.slot);
  cudaStreamSynchronize(c.stream);
  cudaFree(c.d_exptab);
  cudaEventDestroy(c.ev0);
  cudaEventDestroy(c.ev1);
  cudaStreamDestroy(c.stream);
  c = Context();
}

static int make_context(Context &c, int device, int slot) {
  KDE_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  KDE_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) KDE_FAIL(22, "libkdeb200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
  c.device = device;
  c.slot = slot;
  c.sm_count = prop.multiProcessorCount;
  KDE_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
  {  // keep up to 1 GiB of freed blocks in the stream-ordered pool (the default returns everything to the driver
     // at every sync, which made tree create / destroy cost tens of milliseconds)
    cudaMemPool_t pool;
    KDE_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = 1ull << 30;  // bounded: multi-GB staging buffers (injected randU) go back to the driver
    KDE_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
  }
  KDE_CUDA(cudaEventCreate(&c.ev0));
  KDE_CUDA(cudaEventCreate(&c.ev1));
  double tab[KDE_EXP_TAB];
  for (int j = 0; j < KDE_EXP_TAB; ++j) {  // 2^(j/TAB), high word biased by -(j << SHL): see kde_exp_core
    const double v = (double)exp2l((long double)j / (long double)KDE_EXP_TAB);
    uint64_t bits;
    std::memcpy(&bits, &v, sizeof(bits));
    bits -= (uint64_t)((uint32_t)j << KDE_EXP_SHL) << 32;
    std::memcpy(&tab[j], &bits, sizeof(bits));
  }
  KDE_CUDA(cudaMalloc(&c.d_exptab, sizeof(tab)));
  KDE_CUDA(cudaMemcpy(c.d_exptab, tab, sizeof(tab), cudaMemcpyHostToDevice));
  c.ready = true;
  return 0;
}

static int init_device(int device) {
  Context &c = g_ctx[0];
  int count = 0;
  KDE_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) KDE_FAIL(20, "no CUDA device visible: libkdeb200 has no CPU fallback");
  if (device < 0 || device >= count) KDE_FAIL(21, "kdeb200_init: device %d out of range (0..%d)", device, count - 1);
  if (c.ready && c.device == device) {
    KDE_CUDA(cudaSetDevice(device));
    return 0;
  }
  for (int s = g_nctx - 1; s >= 0; --s) drop_context(g_ctx[s]);  // re-bind: the multi-GPU set goes with it
  g_nctx = 1;
  return make_context(c, device, 0);
}

// devices[0] becomes (or must already be) the primary; the others follow in the given order.  Repeating a device is
// allowed: several contexts (streams, host threads, tree replicas) then share one GPU -- no speed-up, but the whole
// sharding path can be exercised on a single-GPU box (tests) and small GPUs can be oversubscribed deliberately.
static int init_multi_devices(const int *devices, int n) {
  int count = 0;
  KDE_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) KDE_FAIL(20, "no CUDA device visible: libkdeb200 has no CPU fallback");
  if (n < 1 || n > KDEB200_MAX_GPUS) KDE_FAIL(21, "kdeb200_init_multi: between 1 and %d GPUs (got %d)", KDEB200_MAX_GPUS, n);
  for (int i = 0; i < n; ++i)
    if (devices[i] < 0 || devices[i] >= count)
      KDE_FAIL(21, "kdeb200_init_multi: device %d out of range (0..%d)", devices[i], count - 1);
  if (int rc = init_device(devices[0])) return rc;  // no-op when already bound there; otherwise a full re-bind
  for (int s = g_nctx - 1; s >= 1; --s) drop_context(g_ctx[s]);
  g_nctx = 1;
  for (int i = 1; i < n; ++i) {
    if (int rc = make_context(g_ctx[i], devices[i], i)) {
      for (int s = i; s >= 1; --s) drop_context(g_ctx[s]);
      cudaSetDevice(g_ctx[0].device);
      return rc;
    }
    g_nctx = i + 1;
  }
  for (int a = 0; a < g_nctx; ++a)  // peer access for the tree replication copies (ignored where unsupported)
    for (int b = 0; b < g_nctx; ++b) {
      if (g_ctx[a].device == g_ctx[b].device) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, g_ctx[a].device, g_ctx[b].device);
      if (can) {
        cudaSetDevice(g_ctx[a].device);
        if (cudaDeviceEnablePeerAccess(g_ctx[b].device, 0) != cudaSuccess) cudaGetLastError();  // already enabled
        // stream-ordered allocations come from the device's memory pool, which has its own access list: without this
        // every peer copy of pool memory (tree replicas, the LOO contribution vectors) is staged through the host
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, g_ctx[a].device) == cudaSuccess) {
          cudaMemAccessDesc desc = {};
          desc.location.type = cudaMemLocationTypeDevice;
          desc.location.id = g_ctx[b].device;
          desc.flags = cudaMemAccessFlagsProtReadWrite;
          if (cudaMemPoolSetAccess(pool, &desc, 1) != cudaSuccess) cudaGetLastError();
        }
      }
    }
  KDE_CUDA(cudaSetDevice(g_ctx[0].device));
  return 0;
}

// The primary plus the next visible devices (in index order) until `ngpus` contexts exist; ngpus <= 0: every visible device.
static int init_multi(int ngpus) {
  int count = 0;
  KDE_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) KDE_FAIL(20, "no CUDA device visible: libkdeb200 has no CPU fallback");
  if (ngpus <= 0) ngpus = count < KDEB200_MAX_GPUS ? count : KDEB200_MAX_GPUS;
  if (ngpus > count) KDE_FAIL(21, "kdeb200_init_multi: %d GPUs requested, %d visible", ngpus, count);
  int primary = 0;
  if (g_ctx[0].ready) primary = g_ctx[0].device;
  else if (cudaGetDevice(&primary) != cudaSuccess) primary = 0;
  std::vector<int> devs{primary};
  for (int dev = 0; dev < count && (int)devs.size() < ngpus; ++dev)
    if (dev != primary) devs.push_back(dev);
  return init_multi_devices(devs.data(), (int)devs.size());
}

int ensure_init() {
  std::lock_guard<std::mutex> lk(g_mu);
  Context &c = ctx();
  if (c.ready) {
    KDE_CUDA(cudaSetDevice(c.device));
    return 0;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  return init_device(dev);
}

}  // namespace kdeb200

using namespace kdeb200;

extern "C" {

const char *kdeb200_last_error(void) { return get_error(); }
int kdeb200_version(void) { return 100; }

int kdeb200_device_count(int *count) {
  if (!count) KDE_FAIL(2, "device_count: NULL");
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) {
    *count = 0;
    KDE_FAIL(100 + (int)e, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  return 0;
}

int kdeb200_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  return init_device(device);
}

int kdeb200_init_multi(int ngpus) {
  std::lock_guard<std::mutex> lk(g_mu);
  return init_multi(ngpus);
}

int kdeb200_init_multi_devices(const int *devices, int n) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!devices) KDE_FAIL(2, "init_multi_devices: NULL");
  return init_multi_devices(devices, n);
}

int kdeb200_multi_count(int *ngpus) {
  if (!ngpus) KDE_FAIL(2, "multi_count: NULL");
  *ngpus = multi_count();
  return 0;
}

int kdeb200_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  for (int s = g_nctx - 1; s >= 0; --s) drop_context(g_ctx[s]);
  g_nctx = 1;
  return 0;
}

int kdeb200_device_props(int *sm_count, int *cc_major, int *cc_minor, int *clock_khz, size_t *free_bytes) {
  if (int rc = ensure_init()) return rc;
  cudaDeviceProp prop;
  KDE_CUDA(cudaGetDeviceProperties(&prop, ctx().device));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (clock_khz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx().device);
    *clock_khz = khz;
  }
  if (free_bytes) {
    size_t fr = 0, tot = 0;
    KDE_CUDA(cudaMemGetInfo(&fr, &tot));
    *free_bytes = fr;
  }
  return 0;
}

int kdeb200_last_kernel_ms(double *ms, int *launches) {
  if (ms) *ms = ctx().last_ms;
  if (launches) *launches = ctx().last_launches;
  return 0;
}

}  // extern "C"
