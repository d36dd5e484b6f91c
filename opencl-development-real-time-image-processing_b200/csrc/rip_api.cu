// rip_api.cu -- the C ABI of librip_cuda.so (include/rip_cuda.h): discovery, handles, memory,
// device-resident ops and the host-buffer pipeline that Controller::PerformCL* drives.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "rip_common.cuh"
#include "rip_internal.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

// ============================================================================================
// error plumbing / counters
// ============================================================================================
namespace rip {

static thread_local char g_err[512] = "no error";
static std::atomic<uint64_t> g_launches{0};

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
    return (int)e;
}

void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static Options g_options;
static std::once_flag g_options_once;
static const struct { const char *name; int Options::*field; } kOptionTable[] = {
    {"RIP_FUSED_SEG", &Options::fused_seg}, {"RIP_FUSED_NPX", &Options::fused_npx}, {"RIP_FUSED_GENERIC", &Options::fused_generic},
    {"RIP_BLUR_EXACT", &Options::blur_exact}, {"RIP_BLUR_TILED", &Options::blur_tiled}, {"RIP_BLUR_STREAM", &Options::blur_stream},
};

static void load_options_from_env()
{
    for (const auto &o : kOptionTable)
        if (const char *e = getenv(o.name)) {
            const int v = atoi(e);
            g_options.*(o.field) = (v != 0 || e[0] == '0') ? v : 1;   // "RIP_X=" or "RIP_X=yes" mean on
        }
}

const Options &options()
{
    std::call_once(g_options_once, load_options_from_env);
    return g_options;
}

int sm_count(int device)
{
    static int cache[64];
    static std::atomic<bool> have[64];
    if (device < 0 || device >= 64) return 148;
    if (!have[device].load(std::memory_order_acquire)) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
        cache[device] = v;
        have[device].store(true, std::memory_order_release);
    }
    return cache[device];
}

static int check_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(RIP_ENODEV, "no CUDA device available (%s); librip_cuda has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return fail(RIP_EINVAL, "device index %d out of range [0,%d)", device, n);
    return RIP_OK;
}

// 0 = not a format
static int channels_of(int fmt)
{
    const Format *f = format_of(fmt);
    return f ? f->channels : 0;
}

static int load_weights(Weights &dst, int ksize, const float *weights, const char *who)
{
    if (ksize < 1 || ksize > RIP_MAX_KSIZE || (ksize & 1) == 0)
        return fail(RIP_EINVAL, "%s: kernel size must be odd and in [1,%d] (got %d)", who, RIP_MAX_KSIZE, ksize);
    if (!weights) return fail(RIP_EINVAL, "%s: weights is NULL", who);
    memcpy(dst.w, weights, sizeof(float) * ksize * ksize);
    return RIP_OK;
}

}  // namespace rip

using namespace rip;

// ============================================================================================
// handle types
// ============================================================================================
namespace {
constexpr int kSets = 3;  // chunk buffers in flight per device (H2D / kernel / D2H overlap)

struct Part;

struct BufSet {
    cudaStream_t stream = nullptr;
    void *d_in = nullptr, *d_out = nullptr;
    size_t in_cap = 0, out_cap = 0;
    // frames of a decoded format decoded to RGBA8 (GAUSSIAN) or GRAY8 (EDGE / FUSED) for the kernel that follows
    void *d_mid = nullptr;
    size_t mid_cap = 0;
    // pinned staging for callers that hand in pageable memory (std::vector, cv::Mat): allocated on first need
    void *stage_in = nullptr, *stage_out = nullptr;
    size_t stage_in_cap = 0, stage_out_cap = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // write start/end = kernel start, kernel end = read start, read end
    // what is in flight on this set (the worker thread's bookkeeping)
    Part *owner = nullptr;
    uint8_t *copyout_dst = nullptr;   // pageable destination of the staged D2H (NULL: the D2H went straight to the caller)
    size_t copyout_bytes = 0;
    bool timed = false;
};

int ensure(void **p, size_t *cap, size_t need)
{
    if (need <= *cap) return RIP_OK;
    if (*p) RIP_CUDA(cudaFree(*p));
    *p = nullptr;
    *cap = 0;
    // grow in 1 MiB steps so slightly different frame sizes reuse the allocation
    const size_t want = (need + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    RIP_CUDA(cudaMalloc(p, want));
    *cap = want;
    return RIP_OK;
}

int ensure_pinned(void **p, size_t *cap, size_t need)
{
    if (need <= *cap) return RIP_OK;
    if (*p) RIP_CUDA(cudaFreeHost(*p));
    *p = nullptr;
    *cap = 0;
    const size_t want = (need + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    RIP_CUDA(cudaHostAlloc(p, want, cudaHostAllocPortable));
    *cap = want;
    return RIP_OK;
}

struct DevState;
}  // namespace

// One submitted job: shared by the parts (one per device) it was cut into.
struct rip_ticket {
    std::mutex mu;
    std::condition_variable cv;
    int remaining = 0;          // parts not yet finished
    int rc = RIP_OK;
    std::string err;
    double prof_ms[3] = {0, 0, 0};
    bool want_prof = false;
    // the job, copied at submit time (the caller's descriptor and weights need not outlive the call)
    rip_op_desc desc;
    std::vector<float> weights;
    int W = 0, H = 0, cn = 0;
    size_t in_frame_bytes = 0, out_frame_bytes = 0;
    const uint8_t *h_in = nullptr;
    uint8_t *h_out = nullptr;
    bool in_pinned = false, out_pinned = false;
    bool banded = false;
    int n_parts = 0;
};

namespace {
struct Part {
    rip_ticket *t = nullptr;
    int index = 0;              // part number within the ticket (0 carries the profile)
    int f0 = 0, f1 = 0;         // frames [f0, f1) of the batch (frame mode)
    int in_row0 = 0, in_rows = 0, out_row0 = 0, out_rows = 0;   // row band (banded mode)
    int outstanding = 0;        // buffer sets still in flight for this part
    bool issued = false;        // all chunks enqueued
    int rc = RIP_OK;
    std::string err;
};

struct DevState {
    int device = 0;
    BufSet set[kSets];
    int next_set = 0;
    // worker
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<Part *> queue;
    bool stop = false;
};
}  // namespace

struct rip_ctx {
    std::vector<std::unique_ptr<DevState>> devs;
};
struct rip_module {
    rip_ctx *ctx;
    int op;
    std::string variant;
};
struct rip_kernel {
    rip_module *module;
    int op;
    std::string name;
};
struct rip_event {
    int device;
    cudaEvent_t ev;
};

static void worker_main(DevState *dev);

// ============================================================================================
// discovery
// ============================================================================================
extern "C" int rip_abi_version(void) { return RIP_ABI_VERSION; }
extern "C" const char *rip_last_error_string(void) { return g_err; }

extern "C" int rip_launch_count(uint64_t *launches)
{
    if (!launches) return fail(RIP_EINVAL, "rip_launch_count: NULL");
    *launches = g_launches.load(std::memory_order_relaxed);
    return RIP_OK;
}

extern "C" int rip_device_count(int *count)
{
    if (!count) return fail(RIP_EINVAL, "rip_device_count: NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count = 0;
        return fail(RIP_ENODEV, "no CUDA device available (%s); librip_cuda has no CPU fallback", cudaGetErrorString(e));
    }
    *count = n;
    return RIP_OK;
}

extern "C" int rip_device_get_info(int device, rip_device_info *info)
{
    if (!info) return fail(RIP_EINVAL, "rip_device_get_info: NULL");
    if (int rc = check_device(device)) return rc;
    cudaDeviceProp p;
    RIP_CUDA(cudaGetDeviceProperties(&p, device));
    memset(info, 0, sizeof(*info));
    snprintf(info->name, sizeof(info->name), "%s", p.name);
    info->sm_count = p.multiProcessorCount;
    info->cc_major = p.major;
    info->cc_minor = p.minor;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
    info->clock_khz = khz;
    info->l2_bytes = p.l2CacheSize;
    info->global_mem_bytes = p.totalGlobalMem;
    info->smem_per_sm_bytes = p.sharedMemPerMultiprocessor;
    return RIP_OK;
}

extern "C" int rip_device_pci_bus_id(int device, char *buf, size_t buf_len)
{
    if (int rc = check_device(device)) return rc;
    if (!buf || buf_len < 13) return fail(RIP_EINVAL, "rip_device_pci_bus_id: buffer of at least 13 bytes needed");
    RIP_CUDA(cudaDeviceGetPCIBusId(buf, (int)buf_len, device));
    return RIP_OK;
}

extern "C" int rip_device_name(int device, char *buf, size_t buf_len)
{
    if (!buf || buf_len == 0) return fail(RIP_EINVAL, "rip_device_name: NULL buffer");
    rip_device_info info;
    if (int rc = rip_device_get_info(device, &info)) return rc;
    snprintf(buf, buf_len, "%s", info.name);
    return RIP_OK;
}

// ============================================================================================
// context / module / kernel
// ============================================================================================
extern "C" int rip_ctx_create(const int *devices, int n_devices, rip_ctx **out)
{
    if (!out) return fail(RIP_EINVAL, "rip_ctx_create: NULL");
    *out = nullptr;
    int count = 0;
    if (int rc = rip_device_count(&count)) return rc;
    if (count <= 0) return fail(RIP_ENODEV, "no CUDA device available; librip_cuda has no CPU fallback");
    std::vector<int> devs;
    if (!devices || n_devices <= 0) {
        devs.push_back(0);
    } else {
        for (int i = 0; i < n_devices; i++) {
            if (devices[i] < 0 || devices[i] >= count)
                return fail(RIP_EINVAL, "rip_ctx_create: device %d out of range [0,%d)", devices[i], count);
            devs.push_back(devices[i]);
        }
    }
    rip_ctx *ctx = new (std::nothrow) rip_ctx();
    if (!ctx) return fail(RIP_ENOMEM, "rip_ctx_create: out of host memory");
    for (size_t i = 0; i < devs.size(); i++) {
        ctx->devs.emplace_back(new DevState());
        DevState &d = *ctx->devs.back();
        d.device = devs[i];
        DeviceGuard g(d.device);
        if (!g.ok) {
            rip_ctx_destroy(ctx);
            return fail(RIP_ENODEV, "rip_ctx_create: cudaSetDevice(%d) failed", d.device);
        }
        for (int k = 0; k < kSets; k++) {
            cudaError_t e = cudaStreamCreateWithFlags(&d.set[k].stream, cudaStreamNonBlocking);
            for (int j = 0; j < 4 && e == cudaSuccess; j++) e = cudaEventCreate(&d.set[k].ev[j]);
            if (e != cudaSuccess) {
                rip_ctx_destroy(ctx);
                return cuda_fail(e, "cudaStreamCreateWithFlags / cudaEventCreate", __FILE__, __LINE__);
            }
        }
    }
    // one persistent worker thread per device: it owns the device's buffer sets and streams, so no call ever
    // creates a thread and two host threads may use the same context concurrently
    for (auto &d : ctx->devs) d->worker = std::thread(worker_main, d.get());
    *out = ctx;
    return RIP_OK;
}

extern "C" int rip_ctx_destroy(rip_ctx *ctx)
{
    if (!ctx) return RIP_OK;
    for (auto &dp : ctx->devs) {
        DevState &d = *dp;
        if (d.worker.joinable()) {
            {
                std::lock_guard<std::mutex> lk(d.mu);
                d.stop = true;   // (the worker drains its queue before it leaves)
            }
            d.cv.notify_all();
            d.worker.join();
        }
        DeviceGuard g(d.device);
        for (int k = 0; k < kSets; k++) {
            BufSet &b = d.set[k];
            if (b.stream) {
                cudaStreamSynchronize(b.stream);
                cudaStreamDestroy(b.stream);
            }
            if (b.d_in) cudaFree(b.d_in);
            if (b.d_out) cudaFree(b.d_out);
            if (b.d_mid) cudaFree(b.d_mid);
            if (b.stage_in) cudaFreeHost(b.stage_in);
            if (b.stage_out) cudaFreeHost(b.stage_out);
            for (int j = 0; j < 4; j++)
                if (b.ev[j]) cudaEventDestroy(b.ev[j]);
        }
    }
    delete ctx;
    return RIP_OK;
}

extern "C" int rip_ctx_device_count(const rip_ctx *ctx, int *n)
{
    if (!ctx || !n) return fail(RIP_EINVAL, "rip_ctx_device_count: NULL");
    *n = (int)ctx->devs.size();
    return RIP_OK;
}

extern "C" int rip_ctx_device(const rip_ctx *ctx, int index, int *device)
{
    if (!ctx || !device) return fail(RIP_EINVAL, "rip_ctx_device: NULL");
    if (index < 0 || index >= (int)ctx->devs.size()) return fail(RIP_EINVAL, "rip_ctx_device: index %d out of range", index);
    *device = ctx->devs[index]->device;
    return RIP_OK;
}

static int op_of_variant(const std::string &v)
{
    // the reference's kernel file names (RealtimeImageProcessing.cpp:28-30) select the operation
    if (v.find("grayscale") != std::string::npos) return RIP_OP_GRAY;
    if (v.find("gaussian") != std::string::npos) return RIP_OP_GAUSSIAN;
    if (v.find("edge") != std::string::npos || v.find("sobel") != std::string::npos) return RIP_OP_EDGE;
    if (v.find("fused") != std::string::npos) return RIP_OP_FUSED;
    return -1;
}

extern "C" int rip_module_load(rip_ctx *ctx, const char *variant, rip_module **module)
{
    if (!ctx || !variant || !module) return fail(RIP_EINVAL, "rip_module_load: NULL");
    *module = nullptr;
    const int op = op_of_variant(variant);
    if (op < 0) return fail(RIP_EINVAL, "rip_module_load: unknown kernel variant '%s'", variant);
    *module = new (std::nothrow) rip_module{ctx, op, variant};
    return *module ? RIP_OK : fail(RIP_ENOMEM, "rip_module_load: out of host memory");
}

extern "C" int rip_module_release(rip_module *m)
{
    delete m;
    return RIP_OK;
}

extern "C" int rip_kernel_get(rip_module *module, const char *kernel_name, rip_kernel **kernel)
{
    if (!module || !kernel_name || !kernel) return fail(RIP_EINVAL, "rip_kernel_get: NULL");
    *kernel = nullptr;
    // entry-point names of the reference kernels (ProgramHandler.cpp:69-78)
    int op = -1;
    if (!strcmp(kernel_name, "grayscale")) op = RIP_OP_GRAY;
    else if (!strcmp(kernel_name, "gaussian_blur")) op = RIP_OP_GAUSSIAN;
    else if (!strcmp(kernel_name, "sobel_edge_detection")) op = RIP_OP_EDGE;
    else if (!strcmp(kernel_name, "fused")) op = RIP_OP_FUSED;
    if (op < 0 || op != module->op)
        return fail(RIP_EINVAL, "rip_kernel_get: module '%s' has no kernel '%s'", module->variant.c_str(), kernel_name);
    *kernel = new (std::nothrow) rip_kernel{module, op, kernel_name};
    return *kernel ? RIP_OK : fail(RIP_ENOMEM, "rip_kernel_get: out of host memory");
}

extern "C" int rip_kernel_release(rip_kernel *k)
{
    delete k;
    return RIP_OK;
}

extern "C" int rip_kernel_op(const rip_kernel *k, int *op)
{
    if (!k || !op) return fail(RIP_EINVAL, "rip_kernel_op: NULL");
    *op = k->op;
    return RIP_OK;
}

// ============================================================================================
// streams, events, memory
// ============================================================================================
extern "C" int rip_stream_create(int device, rip_stream *stream)
{
    if (!stream) return fail(RIP_EINVAL, "rip_stream_create: NULL");
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    cudaStream_t s;
    RIP_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = s;
    return RIP_OK;
}

extern "C" int rip_stream_destroy(int device, rip_stream stream)
{
    if (!stream) return RIP_OK;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaStreamDestroy((cudaStream_t)stream));
    return RIP_OK;
}

extern "C" int rip_stream_sync(int device, rip_stream stream)
{
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return RIP_OK;
}

extern "C" int rip_device_sync(int device)
{
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaDeviceSynchronize());
    return RIP_OK;
}

extern "C" int rip_event_create(int device, rip_event **event)
{
    if (!event) return fail(RIP_EINVAL, "rip_event_create: NULL");
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    cudaEvent_t e;
    RIP_CUDA(cudaEventCreate(&e));
    *event = new (std::nothrow) rip_event{device, e};
    return *event ? RIP_OK : fail(RIP_ENOMEM, "rip_event_create: out of host memory");
}

extern "C" int rip_event_destroy(rip_event *event)
{
    if (!event) return RIP_OK;
    DeviceGuard g(event->device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", event->device);
    cudaEventDestroy(event->ev);
    delete event;
    return RIP_OK;
}

extern "C" int rip_event_record(rip_event *event, rip_stream stream)
{
    if (!event) return fail(RIP_EINVAL, "rip_event_record: NULL");
    DeviceGuard g(event->device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", event->device);
    RIP_CUDA(cudaEventRecord(event->ev, (cudaStream_t)stream));
    return RIP_OK;
}

extern "C" int rip_event_sync(rip_event *event)
{
    if (!event) return fail(RIP_EINVAL, "rip_event_sync: NULL");
    DeviceGuard g(event->device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", event->device);
    RIP_CUDA(cudaEventSynchronize(event->ev));
    return RIP_OK;
}

extern "C" int rip_event_elapsed_ns(rip_event *start, rip_event *stop, uint64_t *ns)
{
    if (!start || !stop || !ns) return fail(RIP_EINVAL, "rip_event_elapsed_ns: NULL");
    DeviceGuard g(start->device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", start->device);
    float ms = 0.f;
    RIP_CUDA(cudaEventElapsedTime(&ms, start->ev, stop->ev));
    *ns = (uint64_t)llround((double)ms * 1e6);
    return RIP_OK;
}

extern "C" int rip_malloc_device(int device, size_t bytes, void **d_ptr)
{
    if (!d_ptr) return fail(RIP_EINVAL, "rip_malloc_device: NULL");
    *d_ptr = nullptr;
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaMalloc(d_ptr, bytes ? bytes : 1));
    return RIP_OK;
}

extern "C" int rip_free_device(int device, void *d_ptr)
{
    if (!d_ptr) return RIP_OK;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaFree(d_ptr));
    return RIP_OK;
}

extern "C" int rip_malloc_pinned(size_t bytes, void **h_ptr)
{
    if (!h_ptr) return fail(RIP_EINVAL, "rip_malloc_pinned: NULL");
    *h_ptr = nullptr;
    if (int rc = check_device(0)) return rc;
    RIP_CUDA(cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocPortable));
    return RIP_OK;
}

extern "C" int rip_free_pinned(void *h_ptr)
{
    if (!h_ptr) return RIP_OK;
    RIP_CUDA(cudaFreeHost(h_ptr));
    return RIP_OK;
}

extern "C" int rip_memcpy_h2d_async(int device, void *d_dst, const void *h_src, size_t bytes, rip_stream stream)
{
    if (!d_dst || !h_src) return fail(RIP_EINVAL, "rip_memcpy_h2d_async: NULL");
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return RIP_OK;
}

extern "C" int rip_memcpy_d2h_async(int device, void *h_dst, const void *d_src, size_t bytes, rip_stream stream)
{
    if (!h_dst || !d_src) return fail(RIP_EINVAL, "rip_memcpy_d2h_async: NULL");
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return RIP_OK;
}

extern "C" int rip_memset_device_async(int device, void *d_dst, int value, size_t bytes, rip_stream stream)
{
    if (!d_dst) return fail(RIP_EINVAL, "rip_memset_device_async: NULL");
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    RIP_CUDA(cudaMemsetAsync(d_dst, value, bytes, (cudaStream_t)stream));
    return RIP_OK;
}

// ============================================================================================
// Gaussian weights.  Same typing as the reference generator (Controller.cpp:352-372): the exponent
// argument is a float quotient, exp() is the double overload, the 2*pi*sigma^2 divisor is double,
// each tap is rounded to float when stored, the running sum and the normalising divide are float.
// ============================================================================================
extern "C" int rip_gauss_weights(int ksize, float sigma, float *weights)
{
    if (!weights) return fail(RIP_EINVAL, "rip_gauss_weights: NULL");
    if (ksize < 1 || ksize > RIP_MAX_KSIZE || (ksize & 1) == 0)
        return fail(RIP_EINVAL, "rip_gauss_weights: kernel size must be odd and in [1,%d] (got %d)", RIP_MAX_KSIZE, ksize);
    if (!(sigma > 0.0f)) return fail(RIP_EINVAL, "rip_gauss_weights: sigma must be positive");
    const int r = ksize / 2;
    const float two_sigma_sq = 2 * sigma * sigma;
    const double norm = 2 * M_PI * sigma * sigma;
    volatile float total = 0.0f;  // volatile: keep the accumulation in float on every compiler
    float *w = weights;
    for (int dy = -r; dy <= r; dy++)
        for (int dx = -r; dx <= r; dx++) {
            const float e = (float)(-(dx * dx + dy * dy)) / two_sigma_sq;
            const float tap = (float)(std::exp((double)e) / norm);
            *w++ = tap;
            total = total + tap;
        }
    const float t = total;
    for (int i = 0; i < ksize * ksize; i++) weights[i] = weights[i] / t;
    return RIP_OK;
}

// ============================================================================================
// device-resident ops
// ============================================================================================
static int check_image(const char *who, const void *in, const void *out, int w, int h, int n)
{
    if (!in || !out) return fail(RIP_EINVAL, "%s: NULL device pointer", who);
    if (w <= 0 || h <= 0 || n <= 0) return fail(RIP_EINVAL, "%s: width, height and n_frames must be positive (got %d x %d x %d)", who, w, h, n);
    return RIP_OK;
}

extern "C" int rip_gray(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                        int n_frames, int in_format, int out_mode)
{
    if (int rc = check_device(device)) return rc;
    if (int rc = check_image("rip_gray", d_in, d_out, width, height, n_frames)) return rc;
    if (out_mode != RIP_GRAY_OUT_U8 && out_mode != RIP_GRAY_OUT_RGBA) return fail(RIP_EINVAL, "rip_gray: bad out_mode %d", out_mode);
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    if (decodes_to_color(in_format))
        return launch_yuv((cudaStream_t)stream, d_in, d_out, width, height, n_frames, in_format,
                          out_mode == RIP_GRAY_OUT_RGBA ? YUV_TO_GRAY_RGBA : YUV_TO_GRAY);
    return launch_gray((cudaStream_t)stream, d_in, d_out, (long long)width * height * n_frames, in_format, out_mode, device);
}

extern "C" int rip_convert(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                           int n_frames, int in_format, int out_format)
{
    if (int rc = check_device(device)) return rc;
    if (int rc = check_image("rip_convert", d_in, d_out, width, height, n_frames)) return rc;
    if (!decodes_to_color(in_format))
        return fail(RIP_EUNSUPPORTED, "rip_convert: input format %d (RIP_FMT_NV12_COLOR, YUYV, UYVY, I420, BAYER_*8 ... BAYER_*16 or BAYER_*P_*)", in_format);
    YuvOut to;
    switch (out_format) {
    case RIP_FMT_RGB8: to = YUV_TO_RGB; break;
    case RIP_FMT_BGR8: to = YUV_TO_BGR; break;
    case RIP_FMT_RGBA8: to = YUV_TO_RGBA; break;
    case RIP_FMT_BGRA8: to = YUV_TO_BGRA; break;
    default: return fail(RIP_EUNSUPPORTED, "rip_convert: output format %d (RGB8, BGR8, RGBA8 or BGRA8)", out_format);
    }
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    return launch_yuv((cudaStream_t)stream, d_in, d_out, width, height, n_frames, in_format, to);
}

static int needs_gray_first(const char *who, int fmt)
{
    const char *name = format_of(fmt)->name;
    return fail(RIP_EUNSUPPORTED, "%s: RIP_FMT_%s is not taken here; decode with rip_gray(..., RIP_FMT_%s, RIP_GRAY_OUT_U8) "
                "and pass the result as RIP_FMT_GRAY8", who, name, name);
}

extern "C" int rip_gauss(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                         int n_frames, int channels, int ksize, const float *weights)
{
    if (int rc = check_device(device)) return rc;
    if (int rc = check_image("rip_gauss", d_in, d_out, width, height, n_frames)) return rc;
    Weights wts;
    if (int rc = load_weights(wts, ksize, weights, "rip_gauss")) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    return launch_blur((cudaStream_t)stream, d_in, d_out, width, height, n_frames, channels, ksize, wts, 0, height, 0, height);
}

extern "C" int rip_sobel(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                         int n_frames, int in_format)
{
    if (int rc = check_device(device)) return rc;
    if (int rc = check_image("rip_sobel", d_in, d_out, width, height, n_frames)) return rc;
    if (decodes_to_color(in_format)) return needs_gray_first("rip_sobel", in_format);
    if (channels_of(in_format) == 0) return fail(RIP_EINVAL, "rip_sobel: unsupported input format %d", in_format);
    if (in_format == RIP_FMT_NV12 && (height & 1)) return fail(RIP_EINVAL, "rip_sobel: NV12 frames need an even height (got %d)", height);
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    if (fused_supported(width, height, in_format, 0, d_in, d_out))
        return launch_fused((cudaStream_t)stream, d_in, d_out, width, height, n_frames, in_format, false, nullptr, 0, height, 0,
                            height, device);
    return launch_sobel((cudaStream_t)stream, d_in, d_out, width, height, n_frames, in_format, 0, height, 0, height);
}

extern "C" int rip_fused_workspace_bytes(int width, int in_rows, int n_frames, int ksize, size_t *bytes)
{
    if (!bytes) return fail(RIP_EINVAL, "rip_fused_workspace_bytes: NULL");
    if (width <= 0 || in_rows <= 0 || n_frames <= 0) return fail(RIP_EINVAL, "rip_fused_workspace_bytes: bad shape");
    (void)ksize;
    *bytes = 0;   // every shape and kernel size runs as a single kernel
    return RIP_OK;
}

extern "C" int rip_fused(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                         int n_frames, int in_format, int ksize, const float *weights, int in_row0, int in_rows,
                         int out_row0, int out_rows, void * /* d_workspace: unused */, size_t /* workspace_bytes: unused */)
{
    if (int rc = check_device(device)) return rc;
    if (int rc = check_image("rip_fused", d_in, d_out, width, height, n_frames)) return rc;
    if (decodes_to_color(in_format)) return needs_gray_first("rip_fused", in_format);
    if (channels_of(in_format) == 0) return fail(RIP_EINVAL, "rip_fused: unsupported input format %d", in_format);
    if (in_format == RIP_FMT_NV12 && (height & 1)) return fail(RIP_EINVAL, "rip_fused: NV12 frames need an even height (got %d)", height);
    Weights wts;
    if (int rc = load_weights(wts, ksize, weights, "rip_fused")) return rc;
    const int half = ksize / 2;
    if (out_row0 < 0 || out_rows <= 0 || out_row0 + out_rows > height)
        return fail(RIP_EINVAL, "rip_fused: output rows [%d,%d) outside the image (height %d)", out_row0, out_row0 + out_rows, height);
    // blurred rows the Sobel stage needs, then gray rows the blur stage needs (both clipped to the image)
    const int b0 = max(0, out_row0 - 1), b1 = min(height, out_row0 + out_rows + 1);
    const int g0 = max(0, b0 - half), g1 = min(height, b1 + half);
    if (in_row0 < 0 || in_rows <= 0 || in_row0 > g0 || in_row0 + in_rows < g1 || in_row0 + in_rows > height)
        return fail(RIP_EINVAL, "rip_fused: input band [%d,%d) does not cover rows [%d,%d) needed for output rows [%d,%d)",
                    in_row0, in_row0 + in_rows, g0, g1, out_row0, out_row0 + out_rows);
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    cudaStream_t s = (cudaStream_t)stream;
    {
        float g3[3], thr;  // single-kernel path: 5x5, aligned shape, and weights the guard band can cover
        if (ksize == 5 && !options().fused_generic && fused_supported(width, height, in_format, 5, d_in, d_out) && fused_plan_weights(wts.w, g3, &thr))
            return launch_fused(s, d_in, d_out, width, height, n_frames, in_format, true, wts.w, in_row0, in_rows, out_row0, out_rows, device);
    }
    // every other shape, kernel size and weight set: still one kernel, the reference's arithmetic throughout
    return launch_fused_tile(s, d_in, d_out, width, height, n_frames, in_format, ksize, wts, in_row0, in_rows, out_row0, out_rows);
}

// ============================================================================================
// diagnostics
// ============================================================================================
static unsigned long long *g_d_slow = nullptr;

extern "C" int rip_debug_slow_path_stats(int device, int enable, uint64_t *slow_pixels)
{
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    if (slow_pixels) *slow_pixels = 0;
    if (g_d_slow && slow_pixels) {
        unsigned long long v = 0;
        RIP_CUDA(cudaDeviceSynchronize());
        RIP_CUDA(cudaMemcpy(&v, g_d_slow, sizeof(v), cudaMemcpyDeviceToHost));
        *slow_pixels = v;
    }
    if (enable && !g_d_slow) {
        RIP_CUDA(cudaMalloc(&g_d_slow, sizeof(unsigned long long)));
    }
    if (g_d_slow) RIP_CUDA(cudaMemset(g_d_slow, 0, sizeof(unsigned long long)));
    if (!enable && g_d_slow) {
        fused_set_slow_counter(nullptr);
        blur_sep_set_slow_counter(nullptr);
        RIP_CUDA(cudaFree(g_d_slow));
        g_d_slow = nullptr;
    }
    if (enable) {
        fused_set_slow_counter(g_d_slow);
        blur_sep_set_slow_counter(g_d_slow);
    }
    return RIP_OK;
}

extern "C" int rip_debug_set_option(const char *name, int value)
{
    if (!name) return fail(RIP_EINVAL, "rip_debug_set_option: NULL");
    options();   // (the environment is read first, so that a later first use cannot overwrite this call)
    for (const auto &o : kOptionTable)
        if (!strcmp(name, o.name) || !strcmp(name, o.name + 4)) {
            g_options.*(o.field) = value;
            return RIP_OK;
        }
    return fail(RIP_EINVAL, "rip_debug_set_option: unknown option '%s'", name);
}

extern "C" int rip_debug_selftest(int device, uint64_t *checked, uint64_t *mismatches)
{
    if (!checked || !mismatches) return fail(RIP_EINVAL, "rip_debug_selftest: NULL");
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    unsigned long long c = 0, m = 0;
    if (int rc = fused_selftest(device, &c, &m)) return rc;
    *checked = c;
    *mismatches = m;
    return RIP_OK;
}

// ============================================================================================
// host-buffer pipeline
// ============================================================================================
extern "C" int rip_out_bytes_per_frame(const rip_op_desc *desc, int width, int height, size_t *bytes)
{
    if (!desc || !bytes) return fail(RIP_EINVAL, "rip_out_bytes_per_frame: NULL");
    const size_t px = (size_t)width * height;
    switch (desc->op) {
    case RIP_OP_GRAY: *bytes = desc->gray_out == RIP_GRAY_OUT_RGBA ? px * 4 : px; return RIP_OK;
    case RIP_OP_EDGE: case RIP_OP_FUSED: *bytes = px; return RIP_OK;
    case RIP_OP_GAUSSIAN: *bytes = px * (decodes_to_color(desc->in_format) ? 4 : channels_of(desc->in_format)); return RIP_OK;
    default: return fail(RIP_EINVAL, "unknown op %d", desc->op);
    }
}

namespace {

int validate_desc(const rip_op_desc *desc, int *cn_out)
{
    if (!desc) return fail(RIP_EINVAL, "rip_process_host: NULL descriptor");
    const Format *f = format_of(desc->in_format);
    if (!f) return fail(RIP_EINVAL, "rip_process_host: unsupported input format %d", desc->in_format);
    const int cn = f->channels;
    switch (desc->op) {
    case RIP_OP_GRAY:
        if (cn < 3) return fail(RIP_EINVAL, "GRAYSCALE needs a colour input");
        break;
    case RIP_OP_EDGE:
        break;
    case RIP_OP_GAUSSIAN:
        if (!(f->layout == LAYOUT_INTERLEAVED && (cn == 1 || cn == 4)) && !decodes_to_color(desc->in_format))
            return fail(RIP_EINVAL, "GAUSSIAN runs on GRAY8, RGBA8/BGRA8, NV12_COLOR, YUYV, UYVY, I420 or Bayer input");
        if (!desc->weights) return fail(RIP_EINVAL, "GAUSSIAN needs weights");
        break;
    case RIP_OP_FUSED:
        if (!desc->weights) return fail(RIP_EINVAL, "FUSED needs weights");
        break;
    default:
        return fail(RIP_EINVAL, "unknown op %d", desc->op);
    }
    *cn_out = cn;
    return RIP_OK;
}

// gray -> Sobel on one row band of a single frame (the band's input rows are device-resident at d_in)
int rip_sobel_rows(int device, cudaStream_t s, const uint8_t *d_in, uint8_t *d_out, int W, int H, int fmt, int in_row0, int in_rows,
                   int out_row0, int out_rows)
{
    DeviceGuard g(device);
    if (!g.ok) return fail(RIP_ENODEV, "cudaSetDevice(%d) failed", device);
    if (fused_supported(W, H, fmt, 0, d_in, d_out))
        return launch_fused(s, d_in, d_out, W, H, 1, fmt, false, nullptr, in_row0, in_rows, out_row0, out_rows, device);
    return launch_sobel(s, d_in, d_out, W, H, 1, fmt, in_row0, in_rows, out_row0, out_rows);
}

// ---- the worker side ----------------------------------------------------------------------------------------

// enqueue one operation on device-resident data: `n_frames` whole frames, or one row band of a single frame
int enqueue_op(const rip_ticket &t, int device, const BufSet &b, int n_frames, const Part *band)
{
    const rip_op_desc &d = t.desc;
    cudaStream_t s = b.stream;
    const uint8_t *in = (const uint8_t *)b.d_in;
    uint8_t *out = (uint8_t *)b.d_out;
    if (band) {
        if (d.op == RIP_OP_FUSED)
            return rip_fused(device, s, in, out, t.W, t.H, 1, d.in_format, d.ksize, d.weights, band->in_row0, band->in_rows,
                             band->out_row0, band->out_rows, nullptr, 0);
        return rip_sobel_rows(device, s, in, out, t.W, t.H, d.in_format, band->in_row0, band->in_rows, band->out_row0, band->out_rows);
    }
    if (decodes_to_color(d.in_format) && d.op != RIP_OP_GRAY) {
        // decode into the chunk's middle buffer (RGBA8 for the blur, GRAY8 for Sobel / fused), then the existing kernel on it
        uint8_t *mid = (uint8_t *)b.d_mid;
        if (d.op == RIP_OP_GAUSSIAN) {
            if (int rc = rip_convert(device, s, in, mid, t.W, t.H, n_frames, d.in_format, RIP_FMT_RGBA8)) return rc;
            return rip_gauss(device, s, mid, out, t.W, t.H, n_frames, 4, d.ksize, d.weights);
        }
        if (int rc = rip_gray(device, s, in, mid, t.W, t.H, n_frames, d.in_format, RIP_GRAY_OUT_U8)) return rc;
        in = mid;
        if (d.op == RIP_OP_EDGE) return rip_sobel(device, s, in, out, t.W, t.H, n_frames, RIP_FMT_GRAY8);
        return rip_fused(device, s, in, out, t.W, t.H, n_frames, RIP_FMT_GRAY8, d.ksize, d.weights, 0, t.H, 0, t.H, nullptr, 0);
    }
    switch (d.op) {
    case RIP_OP_GRAY:
        return rip_gray(device, s, in, out, t.W, t.H, n_frames, d.in_format, d.gray_out);
    case RIP_OP_EDGE:
        return rip_sobel(device, s, in, out, t.W, t.H, n_frames, d.in_format);
    case RIP_OP_GAUSSIAN:
        return rip_gauss(device, s, in, out, t.W, t.H, n_frames, t.cn, d.ksize, d.weights);
    case RIP_OP_FUSED:
        return rip_fused(device, s, in, out, t.W, t.H, n_frames, d.in_format, d.ksize, d.weights, 0, t.H, 0, t.H, nullptr, 0);
    default:
        return fail(RIP_EINVAL, "unknown op %d", d.op);
    }
}

void finish_part(Part *p)
{
    rip_ticket *t = p->t;
    bool last;
    {
        std::lock_guard<std::mutex> lk(t->mu);
        if (p->rc != RIP_OK && t->rc == RIP_OK) {
            t->rc = p->rc;
            t->err = p->err;
        }
        last = --t->remaining == 0;
        if (last) t->cv.notify_all();   // (under the lock: rip_collect may delete the ticket as soon as it sees 0)
    }
    delete p;
}

// Wait until buffer set `b` is free again: its stream has drained, a staged result has been copied out to the
// caller's pageable buffer, the profile (if this was the timed chunk) is read, and its part is told.
void retire_set(BufSet &b)
{
    if (!b.owner) return;
    Part *p = b.owner;
    cudaError_t e = cudaStreamSynchronize(b.stream);
    if (e != cudaSuccess && p->rc == RIP_OK) {
        p->rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
        p->err = rip_last_error_string();
    }
    if (p->rc == RIP_OK && b.copyout_dst) memcpy(b.copyout_dst, b.stage_out, b.copyout_bytes);
    if (p->rc == RIP_OK && b.timed) {
        float w = 0, k = 0, r = 0;
        cudaEventElapsedTime(&w, b.ev[0], b.ev[1]);
        cudaEventElapsedTime(&k, b.ev[1], b.ev[2]);
        cudaEventElapsedTime(&r, b.ev[2], b.ev[3]);
        std::lock_guard<std::mutex> lk(p->t->mu);
        p->t->prof_ms[0] = w; p->t->prof_ms[1] = k; p->t->prof_ms[2] = r;
    }
    b.owner = nullptr;
    b.copyout_dst = nullptr;
    b.timed = false;
    if (--p->outstanding == 0 && p->issued) finish_part(p);
}

// Enqueue every chunk of one part.  Chunks cycle through the kSets buffer sets, each with its own stream, so the H2D
// of chunk i+1 and the D2H of chunk i-1 overlap the kernel of chunk i -- and, because nothing here waits for the
// part's own completion, the first chunks of the NEXT part in the queue overlap the tail of this one.
void issue_part(DevState &dev, Part *p)
{
    rip_ticket &t = *p->t;
    const bool band = t.banded;
    const int n = band ? 1 : p->f1 - p->f0;
    // ~48 MiB of input per chunk keeps three chunks in flight without hoarding HBM
    int chunk = band ? 1 : (int)((size_t)(48u << 20) / (t.in_frame_bytes ? t.in_frame_bytes : 1));
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    const size_t row_in = (size_t)t.W * t.cn;
    int rc = RIP_OK;
    p->outstanding = 1;   // (guards against finishing while still issuing)
    for (int c0 = 0; c0 < n && rc == RIP_OK; c0 += chunk) {
        const int cf = (n - c0 < chunk) ? n - c0 : chunk;
        BufSet &b = dev.set[dev.next_set];
        dev.next_set = (dev.next_set + 1) % kSets;
        retire_set(b);   // previous user of this set (of this part or of an earlier one) is done
        const size_t in_bytes = band ? row_in * p->in_rows : t.in_frame_bytes * cf;
        const size_t out_bytes = band ? (size_t)t.W * p->out_rows : t.out_frame_bytes * cf;
        const uint8_t *src = band ? t.h_in + row_in * p->in_row0 : t.h_in + (size_t)(p->f0 + c0) * t.in_frame_bytes;
        uint8_t *dst = band ? t.h_out + (size_t)t.W * p->out_row0 : t.h_out + (size_t)(p->f0 + c0) * t.out_frame_bytes;
        if ((rc = ensure(&b.d_in, &b.in_cap, in_bytes))) break;
        if ((rc = ensure(&b.d_out, &b.out_cap, out_bytes))) break;
        if (decodes_to_color(t.desc.in_format) && t.desc.op != RIP_OP_GRAY &&
            (rc = ensure(&b.d_mid, &b.mid_cap, (size_t)t.W * t.H * cf * (t.desc.op == RIP_OP_GAUSSIAN ? 4 : 1))))
            break;
        if (!t.in_pinned) {   // pageable source: stage through pinned memory (the copy overlaps the DMA of the previous chunk)
            if ((rc = ensure_pinned(&b.stage_in, &b.stage_in_cap, in_bytes))) break;
            memcpy(b.stage_in, src, in_bytes);
            src = (const uint8_t *)b.stage_in;
        }
        uint8_t *d2h_dst = dst;
        if (!t.out_pinned) {
            if ((rc = ensure_pinned(&b.stage_out, &b.stage_out_cap, out_bytes))) break;
            d2h_dst = (uint8_t *)b.stage_out;
        }
        const bool timed = t.want_prof && p->index == 0 && c0 == 0;
        cudaError_t e = cudaSuccess;
        if (timed) cudaEventRecord(b.ev[0], b.stream);
        if ((e = cudaMemcpyAsync(b.d_in, src, in_bytes, cudaMemcpyHostToDevice, b.stream)) != cudaSuccess) {
            rc = cuda_fail(e, "cudaMemcpyAsync(H2D)", __FILE__, __LINE__);
            break;
        }
        if (timed) cudaEventRecord(b.ev[1], b.stream);
        if ((rc = enqueue_op(t, dev.device, b, cf, band ? p : nullptr))) break;
        if (timed) cudaEventRecord(b.ev[2], b.stream);
        if ((e = cudaMemcpyAsync(d2h_dst, b.d_out, out_bytes, cudaMemcpyDeviceToHost, b.stream)) != cudaSuccess) {
            rc = cuda_fail(e, "cudaMemcpyAsync(D2H)", __FILE__, __LINE__);
            break;
        }
        if (timed) cudaEventRecord(b.ev[3], b.stream);
        b.owner = p;
        b.copyout_dst = t.out_pinned ? nullptr : dst;
        b.copyout_bytes = out_bytes;
        b.timed = timed;
        p->outstanding++;
    }
    if (rc != RIP_OK && p->rc == RIP_OK) {
        p->rc = rc;
        p->err = rip_last_error_string();
    }
    p->issued = true;
    if (--p->outstanding == 0) finish_part(p);
}

}  // namespace

static void worker_main(DevState *dev)
{
    const bool dev_ok = cudaSetDevice(dev->device) == cudaSuccess;
    for (;;) {
        Part *p = nullptr;
        {
            std::unique_lock<std::mutex> lk(dev->mu);
            if (dev->queue.empty() && !dev->stop) {
                // nothing queued: retire what is in flight (oldest first), then sleep
                lk.unlock();
                for (int k = 0; k < kSets; k++) retire_set(dev->set[(dev->next_set + k) % kSets]);
                lk.lock();
                dev->cv.wait(lk, [&] { return dev->stop || !dev->queue.empty(); });
            }
            if (dev->queue.empty()) {
                if (dev->stop) break;
                continue;
            }
            p = dev->queue.front();
            dev->queue.pop_front();
        }
        if (!dev_ok) {
            p->rc = fail(RIP_ENODEV, "cudaSetDevice(%d) failed in the device worker", dev->device);
            p->err = rip_last_error_string();
            p->issued = true;
            finish_part(p);
            continue;
        }
        issue_part(*dev, p);
    }
    for (int k = 0; k < kSets; k++) retire_set(dev->set[(dev->next_set + k) % kSets]);
}

namespace {

void fill_prof(uint64_t prof_ns[6], const double ms[3])
{
    // cumulative offsets from the start of the call, in ns: [w0, w1, k0, k1, r0, r1]
    const double w = ms[0] * 1e6, k = ms[1] * 1e6, r = ms[2] * 1e6;
    prof_ns[0] = 0;
    prof_ns[1] = (uint64_t)llround(w);
    prof_ns[2] = prof_ns[1];
    prof_ns[3] = (uint64_t)llround(w + k);
    prof_ns[4] = prof_ns[3];
    prof_ns[5] = (uint64_t)llround(w + k + r);
}

// pinned (cudaHostAlloc / cudaHostRegister) or managed memory can be handed to cudaMemcpyAsync directly; anything
// else is pageable and goes through the context's pinned staging buffers
bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

}  // namespace

extern "C" int rip_shard_frames(int n_frames, int n_parts, int index, int *first, int *count)
{
    if (!first || !count || n_frames < 0 || n_parts <= 0 || index < 0 || index >= n_parts)
        return fail(RIP_EINVAL, "rip_shard_frames: bad arguments (%d frames, part %d of %d)", n_frames, index, n_parts);
    const int f0 = (int)((long long)n_frames * index / n_parts), f1 = (int)((long long)n_frames * (index + 1) / n_parts);
    *first = f0;
    *count = f1 - f0;
    return RIP_OK;
}

extern "C" int rip_band_rows(int height, int n_parts, int index, int halo, int *in_row0, int *in_rows, int *out_row0, int *out_rows)
{
    if (!in_row0 || !in_rows || !out_row0 || !out_rows || height <= 0 || n_parts <= 0 || n_parts > height || index < 0 ||
        index >= n_parts || halo < 0)
        return fail(RIP_EINVAL, "rip_band_rows: bad arguments (height %d, part %d of %d, halo %d)", height, index, n_parts, halo);
    const int o0 = (int)((long long)height * index / n_parts), o1 = (int)((long long)height * (index + 1) / n_parts);
    const int i0 = max(0, o0 - halo), i1 = min(height, o1 + halo);
    *out_row0 = o0; *out_rows = o1 - o0; *in_row0 = i0; *in_rows = i1 - i0;
    return RIP_OK;
}

extern "C" int rip_submit(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in, uint8_t *h_out, int width, int height,
                          int n_frames, int flags, rip_ticket **ticket)
{
    if (!ticket) return fail(RIP_EINVAL, "rip_submit: NULL ticket pointer");
    *ticket = nullptr;
    if (!ctx || ctx->devs.empty()) return fail(RIP_EINVAL, "rip_submit: NULL context");
    if (!h_in || !h_out) return fail(RIP_EINVAL, "rip_submit: NULL host buffer");
    if (width <= 0 || height <= 0 || n_frames <= 0)
        return fail(RIP_EINVAL, "rip_submit: width, height and n_frames must be positive (got %d x %d x %d)", width, height, n_frames);
    int cn = 0;
    if (int rc = validate_desc(desc, &cn)) return rc;
    if (desc->in_format == RIP_FMT_NV12 && (height & 1)) return fail(RIP_EINVAL, "NV12 frames need an even height (got %d)", height);
    if (decodes_to_color(desc->in_format))
        if (int rc = check_yuv_shape(desc->in_format, width, height)) return rc;
    const bool banded = (flags & RIP_SUBMIT_BANDED) != 0;
    if (banded) {
        if (decodes_to_color(desc->in_format))
            return fail(RIP_EUNSUPPORTED, "row-band mode does not take %s (it decodes whole frames only)", format_of(desc->in_format)->name);
        if (n_frames != 1) return fail(RIP_EINVAL, "row-band mode takes one frame per call (got %d)", n_frames);
        if (desc->op != RIP_OP_FUSED && desc->op != RIP_OP_EDGE) return fail(RIP_EUNSUPPORTED, "row-band mode supports FUSED and EDGE only");
    }
    std::unique_ptr<rip_ticket> t(new (std::nothrow) rip_ticket());
    if (!t) return fail(RIP_ENOMEM, "rip_submit: out of host memory");
    t->desc = *desc;
    if (desc->weights && (desc->op == RIP_OP_GAUSSIAN || desc->op == RIP_OP_FUSED)) {
        if (desc->ksize < 1 || desc->ksize > RIP_MAX_KSIZE || !(desc->ksize & 1))
            return fail(RIP_EINVAL, "kernel size must be odd and in [1,%d] (got %d)", RIP_MAX_KSIZE, desc->ksize);
        t->weights.assign(desc->weights, desc->weights + desc->ksize * desc->ksize);
        t->desc.weights = t->weights.data();
    }
    t->W = width; t->H = height; t->cn = cn;
    t->in_frame_bytes = frame_bytes(*format_of(desc->in_format), width, height);   // (validate_desc checked the format)
    if (int rc = rip_out_bytes_per_frame(desc, width, height, &t->out_frame_bytes)) return rc;
    t->h_in = h_in; t->h_out = h_out;
    t->in_pinned = is_pinned(h_in);
    t->out_pinned = is_pinned(h_out);
    t->banded = banded;
    t->want_prof = (flags & RIP_SUBMIT_PROFILE) != 0;
    const int nd = (int)ctx->devs.size();
    const int units = banded ? height : n_frames;
    const int used = units < nd ? units : nd;
    const int halo = desc->op == RIP_OP_FUSED ? desc->ksize / 2 + 1 : 1;
    // Row-band mode: a device's band is cut further into `sub` consecutive sub-bands (each with its own halo rows) that go
    // through the device's buffer sets one after the other, so the upload of sub-band i+1 overlaps the kernel of sub-band i
    // and the download of sub-band i-1 -- one 8K frame on one device is otherwise a strictly serial H2D, kernel, D2H.
    int sub = 1;
    if (banded) {
        const size_t band_bytes = (size_t)width * t->cn * ((size_t)height / (size_t)used + 1);
        sub = (int)(band_bytes / ((size_t)12 << 20));
        sub = sub < 1 ? 1 : sub > 4 ? 4 : sub;
        if (height / (used * sub) < 64) sub = 1;
    }
    const int n_parts = used * sub;
    t->n_parts = n_parts;
    t->remaining = n_parts;
    std::vector<Part *> parts;
    for (int i = 0; i < n_parts; i++) {
        Part *p = new Part();
        p->t = t.get();
        p->index = i;
        if (banded) rip_band_rows(height, n_parts, i, halo, &p->in_row0, &p->in_rows, &p->out_row0, &p->out_rows);
        else {
            int fc = 0;
            rip_shard_frames(n_frames, used, i, &p->f0, &fc);
            p->f1 = p->f0 + fc;
        }
        parts.push_back(p);
    }
    rip_ticket *raw = t.release();
    for (int i = 0; i < used; i++) {
        DevState &d = *ctx->devs[i];
        {
            std::lock_guard<std::mutex> lk(d.mu);
            for (int k = 0; k < sub; k++) d.queue.push_back(parts[i * sub + k]);
        }
        d.cv.notify_one();
    }
    *ticket = raw;
    return RIP_OK;
}

extern "C" int rip_ticket_done(rip_ticket *ticket, int *done)
{
    if (!ticket || !done) return fail(RIP_EINVAL, "rip_ticket_done: NULL");
    std::lock_guard<std::mutex> lk(ticket->mu);
    *done = ticket->remaining == 0;
    return RIP_OK;
}

extern "C" int rip_collect(rip_ticket *ticket, uint64_t prof_ns[6])
{
    if (!ticket) return fail(RIP_EINVAL, "rip_collect: NULL ticket");
    int rc;
    {
        std::unique_lock<std::mutex> lk(ticket->mu);
        ticket->cv.wait(lk, [&] { return ticket->remaining == 0; });
        rc = ticket->rc;
        if (rc != RIP_OK) fail(rc, "%s", ticket->err.c_str());
        else if (prof_ns) fill_prof(prof_ns, ticket->prof_ms);
    }
    delete ticket;
    return rc;
}

extern "C" int rip_process_host(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in, uint8_t *h_out, int width,
                                int height, int n_frames, uint64_t prof_ns[6])
{
    rip_ticket *t = nullptr;
    if (int rc = rip_submit(ctx, desc, h_in, h_out, width, height, n_frames, prof_ns ? RIP_SUBMIT_PROFILE : 0, &t)) return rc;
    return rip_collect(t, prof_ns);
}

extern "C" int rip_process_host_banded(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                                       int width, int height, uint64_t prof_ns[6])
{
    rip_ticket *t = nullptr;
    if (int rc = rip_submit(ctx, desc, h_in, h_out, width, height, 1, RIP_SUBMIT_BANDED | (prof_ns ? RIP_SUBMIT_PROFILE : 0), &t)) return rc;
    return rip_collect(t, prof_ns);
}

extern "C" int rip_host_register(void *h_ptr, size_t bytes)
{
    if (!h_ptr || !bytes) return fail(RIP_EINVAL, "rip_host_register: NULL / empty range");
    if (int rc = check_device(0)) return rc;
    RIP_CUDA(cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable));
    return RIP_OK;
}

extern "C" int rip_host_unregister(void *h_ptr)
{
    if (!h_ptr) return RIP_OK;
    RIP_CUDA(cudaHostUnregister(h_ptr));
    return RIP_OK;
}
