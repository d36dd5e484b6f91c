// Controller.cpp -- see Controller.hpp.  Error conventions follow the reference: set-up failures print
// and exit through CheckError or return a NULL handle after printing (RT/src/Controller.cpp:5-11, 122-125,
// 147-175); per-operation failures are logged at ERROR level and the call returns with output_data
// untouched (:461-463).
#include "Controller.hpp"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>

#include "rip_formats.h"

namespace {

rip_platform_rec g_platform{0};
rip_device_rec g_devices[64];

const char *basename_of(const char *path)
{
    const char *s = strrchr(path, '/');
    const char *b = strrchr(path, '\\');
    if (b && (!s || b > s)) s = b;
    return s ? s + 1 : path;
}

}  // namespace

Controller::Controller() : num_platforms(0), num_devices(0), m_image_support(CL_FALSE) {}

void Controller::CheckError(cl_int err, const char *name)
{
    if (err != CL_SUCCESS) {
        std::cerr << "Error: " << name << " (" << err << "): " << rip_last_error_string() << std::endl;
        exit(EXIT_FAILURE);
    }
}

std::vector<cl_platform_id> Controller::GetPlatforms()
{
    int n = 0;
    const int rc = rip_device_count(&n);
    CheckError(rc != RIP_OK ? rc : (n > 0 ? CL_SUCCESS : CL_DEVICE_NOT_FOUND), "rip_device_count (no CUDA device: there is no CPU fallback)");
    num_platforms = 1;
    return {&g_platform};
}

std::vector<cl_device_id> Controller::GetDevices(cl_platform_id platform)
{
    (void)platform;
    int n = 0;
    CheckError(rip_device_count(&n), "rip_device_count");
    std::vector<cl_device_id> out;
    if (m_ordinals.empty()) {
        for (int i = 0; i < n && i < 64; i++) {
            g_devices[i].ordinal = i;
            out.push_back(&g_devices[i]);
        }
    } else {
        for (int o : m_ordinals) {
            if (o < 0 || o >= n || o >= 64) CheckError(CL_INVALID_VALUE, "SetDevices: CUDA ordinal out of range");
            g_devices[o].ordinal = o;
            out.push_back(&g_devices[o]);
        }
    }
    num_devices = (cl_uint)out.size();
    return out;
}

void Controller::SetDevices(const std::vector<int> &ordinals) { m_ordinals = ordinals; }

cl_bool Controller::GetImageSupport() { return CL_FALSE; }
void Controller::SetImageSupport(cl_bool image_support) { m_image_support = image_support; }

cl_context Controller::CreateContext(cl_platform_id platform, std::vector<cl_device_id> devices)
{
    (void)platform;
    rip_context_rec *c = new rip_context_rec();
    c->n_devices = 0;
    for (cl_device_id d : devices)
        if (c->n_devices < 16) c->devices[c->n_devices++] = d->ordinal;
    CheckError(rip_ctx_create(c->devices, c->n_devices, &c->ctx), "rip_ctx_create");
    return c;
}

cl_command_queue Controller::CreateCommandQueue(cl_context context, cl_device_id device)
{
    if (!context || !device) {
        std::cerr << "Failed to create command queue: NULL context or device" << std::endl;
        return NULL;
    }
    rip_queue_rec *q = new rip_queue_rec();
    q->context = context;
    q->ordinal = device->ordinal;
    q->ctx = nullptr;
    if (rip_ctx_create(&q->ordinal, 1, &q->ctx) != RIP_OK) {
        std::cerr << "Failed to create command queue for device " << q->ordinal << ": " << rip_last_error_string() << std::endl;
        delete q;
        return NULL;
    }
    return q;
}

cl_program Controller::CreateProgram(cl_context context, cl_device_id device, const char *filename)
{
    (void)device;
    if (!context || !filename) {
        std::cerr << "Failed to create program: NULL context or file name" << std::endl;
        return NULL;
    }
    // the reference reads and JIT-builds "<name>.cl"; here the name only selects a compiled-in kernel
    rip_module *m = nullptr;
    if (rip_module_load(context->ctx, basename_of(filename), &m) != RIP_OK) {
        std::cerr << "Failed to load kernel image for " << filename << ": " << rip_last_error_string() << std::endl;
        return NULL;
    }
    return m;
}

cl_kernel Controller::CreateKernel(cl_program program, const char *kernel_name)
{
    rip_kernel *k = nullptr;
    CheckError(program ? rip_kernel_get(program, kernel_name, &k) : CL_INVALID_VALUE, "rip_kernel_get");
    return k;
}

void Controller::DisplayPlatformInformation(cl_platform_id platform)
{
    InfoPlatform info(platform);
    info.Display();
}

void Controller::Cleanup(cl_context context, cl_command_queue commandQueue, cl_program program, cl_kernel kernel, cl_sampler sampler,
                         cl_mem *mem_objects, int num_mem_objects)
{
    (void)sampler; (void)mem_objects; (void)num_mem_objects;   // device buffers are cached inside the contexts
    // frames still in flight are collected (their contexts are about to go), pinned containers released
    for (auto &kv : m_pending) rip_collect(kv.second.ticket, nullptr);
    m_pending.clear();
    for (void *p : m_pinned) rip_host_unregister(p);
    m_pinned.clear();
    if (kernel) rip_kernel_release(kernel);
    if (program) rip_module_release(program);
    if (commandQueue) {
        if (commandQueue->ctx) rip_ctx_destroy(commandQueue->ctx);
        delete commandQueue;
    }
    if (context) {
        if (context->ctx) rip_ctx_destroy(context->ctx);
        delete context;
    }
}

std::vector<float> Controller::_GenerateGausianKernel(int kernel_size, float sigma)
{
    std::vector<float> k((size_t)kernel_size * kernel_size);
    CheckError(rip_gauss_weights(kernel_size, sigma, k.data()), "rip_gauss_weights");
    return k;
}

void Controller::_appendProfile(const uint64_t prof_ns[6], std::vector<cl_ulong> *profiling_events)
{
    // [write_start, write_end, kernel_start, kernel_end, read_start, read_end] in ns (RT/src/Controller.cpp:66-74)
    if (!profiling_events) return;
    for (int i = 0; i < 6; i++) profiling_events->push_back(prof_ns[i]);
}

// bytes of one input frame in `fmt` (its row in rip_formats.h), 0 = bad format / shape
static size_t in_frame_bytes(int fmt, int width, int height)
{
    const rip::Format *f = rip::format_of(fmt);
    return f && rip::shape_ok(*f, width, height) ? rip::frame_bytes(*f, width, height) : 0;
}

// Validates the shapes and sizes the result container: resized in place (no zero-filled temporary per call), unless it
// aliases the input.  Returns the output pointer, or nullptr after logging.
static unsigned char *prepare_output(const rip_op_desc &desc, const unsigned char *in, size_t in_bytes, std::vector<unsigned char> *output_data,
                                     int width, int height, int n_frames, Logger &logger, const char *what)
{
    size_t out_frame = 0;
    if (width <= 0 || height <= 0 || n_frames <= 0 || rip_out_bytes_per_frame(&desc, width, height, &out_frame) != RIP_OK) {
        logger.log(std::string(what) + ": bad shape or operation", Logger::LogLevel::ERROR);
        return nullptr;
    }
    const size_t in_frame = in_frame_bytes(desc.in_format, width, height);
    if (in_frame == 0) {
        logger.log(std::string(what) + ": unsupported input format (NV12 needs an even height, NV12_COLOR and I420 an even width and height, "
                   "YUYV and UYVY an even width, Bayer of 8 to 16 bits a width and height of at least 3, packed 10- / 12-bit Bayer a "
                   "width of at least 4 that is a multiple of 4 / 2 and a height of at least 3)", Logger::LogLevel::ERROR);
        return nullptr;
    }
    if (in_bytes != (size_t)-1 && in_bytes < in_frame * (size_t)n_frames) {
        logger.log(std::string(what) + ": input holds fewer bytes than width*height*frames of its format need", Logger::LogLevel::ERROR);
        return nullptr;
    }
    const size_t need = out_frame * (size_t)n_frames;
    const unsigned char *ob = output_data->data(), *oe = ob + output_data->capacity();
    if (ob && in + in_frame * (size_t)n_frames > ob && in < oe) {   // output vector overlaps the input: do not resize under the reader
        logger.log(std::string(what) + ": input and output containers overlap", Logger::LogLevel::ERROR);
        return nullptr;
    }
    output_data->resize(need);   // same observable result as the reference's assignment (RT/src/Controller.cpp:510,605)
    return output_data->data();
}

void Controller::_run(const rip_op_desc &desc, rip_ctx *ctx, std::vector<cl_ulong> *profiling_events, const unsigned char *in,
                      size_t in_bytes, std::vector<unsigned char> *output_data, int width, int height, int n_frames, bool banded,
                      Logger &logger, const char *what)
{
    if (!ctx || !in || !output_data) {
        logger.log(std::string(what) + ": NULL context, input or output", Logger::LogLevel::ERROR);
        return;
    }
    unsigned char *out = prepare_output(desc, in, in_bytes, output_data, width, height, n_frames, logger, what);
    if (!out) return;
    uint64_t prof[6] = {0, 0, 0, 0, 0, 0};
    const int rc = banded ? rip_process_host_banded(ctx, &desc, in, out, width, height, prof)
                          : rip_process_host(ctx, &desc, in, out, width, height, n_frames, prof);
    if (rc != RIP_OK) {
        logger.log(std::string(what) + " failed: " + rip_last_error_string(), Logger::LogLevel::ERROR);
        output_data->clear();
        return;
    }
    _appendProfile(prof, profiling_events);
}

void Controller::PerformCLImageGrayscaling(cl_context *context, cl_command_queue *command_queue, cl_kernel *kernel,
                                           std::vector<cl_ulong> *profiling_events, std::vector<unsigned char> *input_data,
                                           std::vector<unsigned char> *output_data, cl_int &width, cl_int &height, Logger &logger)
{
    (void)context; (void)kernel;
    rip_op_desc d{RIP_OP_GRAY, RIP_FMT_RGBA8, RIP_GRAY_OUT_RGBA, 0, nullptr};
    _run(d, command_queue && *command_queue ? (*command_queue)->ctx : nullptr, profiling_events, input_data ? input_data->data() : nullptr,
         input_data ? input_data->size() : 0, output_data, width, height, 1, false, logger, "PerformCLImageGrayscaling");
}

void Controller::PerformCLImageEdgeDetection(cl_context *context, cl_command_queue *command_queue, cl_kernel *kernel,
                                             std::vector<cl_ulong> *profiling_events, std::vector<unsigned char> *input_data,
                                             std::vector<unsigned char> *output_data, cl_int &width, cl_int &height, Logger &logger)
{
    (void)context; (void)kernel;
    rip_op_desc d{RIP_OP_EDGE, RIP_FMT_RGBA8, 0, 0, nullptr};
    _run(d, command_queue && *command_queue ? (*command_queue)->ctx : nullptr, profiling_events, input_data ? input_data->data() : nullptr,
         input_data ? input_data->size() : 0, output_data, width, height, 1, false, logger, "PerformCLImageEdgeDetection");
}

void Controller::PerformCLGaussianBlur(int &kernel_size, float &kernel_sigma, cl_context *context, cl_command_queue *command_queue,
                                       cl_kernel *kernel, std::vector<cl_ulong> *profiling_events, std::vector<unsigned char> *input_data,
                                       std::vector<unsigned char> *output_data, cl_int &width, cl_int &height, Logger &logger)
{
    (void)context; (void)kernel;
    if (kernel_size < 1 || !(kernel_size & 1) || kernel_size > RIP_MAX_KSIZE) {
        logger.log("PerformCLGaussianBlur: kernel size must be odd and in 1.." + std::to_string(RIP_MAX_KSIZE), Logger::LogLevel::ERROR);
        return;
    }
    const std::vector<float> w = _GenerateGausianKernel(kernel_size, kernel_sigma);   // regenerated per call, like the reference (:659-672)
    rip_op_desc d{RIP_OP_GAUSSIAN, RIP_FMT_RGBA8, 0, kernel_size, w.data()};
    _run(d, command_queue && *command_queue ? (*command_queue)->ctx : nullptr, profiling_events, input_data ? input_data->data() : nullptr,
         input_data ? input_data->size() : 0, output_data, width, height, 1, false, logger, "PerformCLGaussianBlur");
}

void Controller::PerformFused(int &kernel_size, float &kernel_sigma, cl_context *context, cl_command_queue *command_queue, cl_kernel *kernel,
                              std::vector<cl_ulong> *profiling_events, std::vector<unsigned char> *input_data,
                              std::vector<unsigned char> *output_data, cl_int &width, cl_int &height, Logger &logger, int in_format)
{
    (void)context; (void)kernel;
    if (kernel_size < 1 || !(kernel_size & 1) || kernel_size > RIP_MAX_KSIZE) {
        logger.log("PerformFused: kernel size must be odd and in 1.." + std::to_string(RIP_MAX_KSIZE), Logger::LogLevel::ERROR);
        return;
    }
    const std::vector<float> w = _GenerateGausianKernel(kernel_size, kernel_sigma);
    rip_op_desc d{RIP_OP_FUSED, in_format, 0, kernel_size, w.data()};
    _run(d, command_queue && *command_queue ? (*command_queue)->ctx : nullptr, profiling_events, input_data ? input_data->data() : nullptr,
         input_data ? input_data->size() : 0, output_data, width, height, 1, false, logger, "PerformFused");
}

static bool desc_of_method(const std::string &method, int in_format, int kernel_size, const float *w, rip_op_desc *d)
{
    if (method == "GRAYSCALE") *d = rip_op_desc{RIP_OP_GRAY, in_format, in_format == RIP_FMT_RGBA8 ? RIP_GRAY_OUT_RGBA : RIP_GRAY_OUT_U8, 0, nullptr};
    else if (method == "EDGE") *d = rip_op_desc{RIP_OP_EDGE, in_format, 0, 0, nullptr};
    else if (method == "GAUSSIAN") *d = rip_op_desc{RIP_OP_GAUSSIAN, in_format, 0, kernel_size, w};
    else if (method == "FUSED") *d = rip_op_desc{RIP_OP_FUSED, in_format, 0, kernel_size, w};
    else return false;
    return true;
}

void Controller::PerformBatch(const std::string &method, cl_context *context, std::vector<cl_ulong> *profiling_events,
                              const unsigned char *frames, int n_frames, std::vector<unsigned char> *output_data, cl_int &width,
                              cl_int &height, Logger &logger, int in_format, int kernel_size, float kernel_sigma, size_t frames_bytes)
{
    std::vector<float> w;
    if (method == "GAUSSIAN" || method == "FUSED") w = _GenerateGausianKernel(kernel_size, kernel_sigma);
    rip_op_desc d;
    if (!desc_of_method(method, in_format, kernel_size, w.data(), &d)) {
        logger.log("PerformBatch: unknown method " + method, Logger::LogLevel::ERROR);
        return;
    }
    _run(d, context && *context ? (*context)->ctx : nullptr, profiling_events, frames, frames_bytes ? frames_bytes : (size_t)-1, output_data, width, height, n_frames, false,
         logger, "PerformBatch");
}

void Controller::PerformBanded(const std::string &method, cl_context *context, std::vector<cl_ulong> *profiling_events,
                               std::vector<unsigned char> *input_data, std::vector<unsigned char> *output_data, cl_int &width,
                               cl_int &height, Logger &logger, int in_format, int kernel_size, float kernel_sigma)
{
    std::vector<float> w;
    if (method == "FUSED") w = _GenerateGausianKernel(kernel_size, kernel_sigma);
    rip_op_desc d;
    if ((method != "EDGE" && method != "FUSED") || !desc_of_method(method, in_format, kernel_size, w.data(), &d)) {
        logger.log("PerformBanded: method must be EDGE or FUSED", Logger::LogLevel::ERROR);
        return;
    }
    _run(d, context && *context ? (*context)->ctx : nullptr, profiling_events, input_data ? input_data->data() : nullptr,
         input_data ? input_data->size() : 0, output_data, width, height, 1, true, logger, "PerformBanded");
}

// ---- [new] asynchronous per-frame form --------------------------------------------------------------------------------
// The reference's frame loop (RealtimeImageProcessing.cpp:325-418) calls PerformOpenCL once per camera frame and blocks
// three times inside it.  SubmitFrame queues the frame on the context's device worker and returns at once; CollectFrame
// waits for it.  With two or three frames in flight the upload of frame i+1, the kernel of frame i and the download of
// frame i-1 overlap.  input_data must stay untouched and output_data unread until CollectFrame(handle) has returned.
int Controller::SubmitFrame(const std::string &method, cl_command_queue *command_queue, std::vector<unsigned char> *input_data,
                            std::vector<unsigned char> *output_data, cl_int &width, cl_int &height, Logger &logger, int in_format,
                            int kernel_size, float kernel_sigma)
{
    rip_ctx *ctx = command_queue && *command_queue ? (*command_queue)->ctx : nullptr;
    if (!ctx || !input_data || !output_data) {
        logger.log("SubmitFrame: NULL queue, input or output", Logger::LogLevel::ERROR);
        return 0;
    }
    std::vector<float> w;
    if (method == "GAUSSIAN" || method == "FUSED") {
        if (kernel_size < 1 || !(kernel_size & 1) || kernel_size > RIP_MAX_KSIZE) {
            logger.log("SubmitFrame: kernel size must be odd and in 1.." + std::to_string(RIP_MAX_KSIZE), Logger::LogLevel::ERROR);
            return 0;
        }
        w = _GenerateGausianKernel(kernel_size, kernel_sigma);
    }
    rip_op_desc d;
    if (!desc_of_method(method, in_format, kernel_size, w.data(), &d)) {
        logger.log("SubmitFrame: unknown method " + method, Logger::LogLevel::ERROR);
        return 0;
    }
    unsigned char *out = prepare_output(d, input_data->data(), input_data->size(), output_data, width, height, 1, logger, "SubmitFrame");
    if (!out) return 0;
    rip_ticket *t = nullptr;
    if (rip_submit(ctx, &d, input_data->data(), out, width, height, 1, RIP_SUBMIT_PROFILE, &t) != RIP_OK) {   // (copies d and w)
        logger.log(std::string("SubmitFrame failed: ") + rip_last_error_string(), Logger::LogLevel::ERROR);
        output_data->clear();
        return 0;
    }
    const int handle = ++m_next_handle > 0 ? m_next_handle : (m_next_handle = 1);
    m_pending[handle] = Pending{t, output_data};
    return handle;
}

bool Controller::CollectFrame(int handle, std::vector<cl_ulong> *profiling_events, Logger &logger)
{
    auto it = m_pending.find(handle);
    if (it == m_pending.end()) {
        logger.log("CollectFrame: unknown handle " + std::to_string(handle), Logger::LogLevel::ERROR);
        return false;
    }
    const Pending p = it->second;
    m_pending.erase(it);
    uint64_t prof[6] = {0, 0, 0, 0, 0, 0};
    if (rip_collect(p.ticket, prof) != RIP_OK) {
        logger.log(std::string("CollectFrame failed: ") + rip_last_error_string(), Logger::LogLevel::ERROR);
        p.output->clear();
        return false;
    }
    _appendProfile(prof, profiling_events);
    return true;
}

// [new] page-lock a container the caller reuses across calls (the iteration loop hands the same input_data to PerformCL*
// NUMBER_OF_ITERATIONS times), so that the pipeline copies it by DMA without a staging copy.  The container must not
// reallocate while it is pinned; Cleanup() releases whatever is still pinned.
bool Controller::PinHostBuffer(std::vector<unsigned char> *buffer)
{
    if (!buffer || buffer->empty()) return false;
    if (rip_host_register(buffer->data(), buffer->size()) != RIP_OK) return false;
    m_pinned.push_back(buffer->data());
    return true;
}

void Controller::UnpinHostBuffer(std::vector<unsigned char> *buffer)
{
    if (!buffer) return;
    for (size_t i = 0; i < m_pinned.size(); i++)
        if (m_pinned[i] == buffer->data()) {
            rip_host_unregister(m_pinned[i]);
            m_pinned.erase(m_pinned.begin() + i);
            return;
        }
}
