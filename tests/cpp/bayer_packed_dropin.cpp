// bayer_packed_dropin.cpp -- packed 10- and 12-bit Bayer raw frames (RIP_FMT_BAYER_RGGB10P_MIPI ... _GBRG12P_GENICAM)
// through the C++ Controller: the batch call, the fused call and the per-frame submit / collect loop, plus the rejections of
// frames the Controller must not read.  A buffer dequeued from V4L2 (SRGGB10P, SRGGB12P) or libcamera (SRGGB10_CSI2P), or an
// Aravis / GenICam BayerRG10p / BayerRG12p buffer, is handed over exactly like in.raw here, as its bytes.
//
//   bayer_packed_dropin <workdir> <format code> <width> <height> <n_frames>
//
// <workdir>/in.raw holds n_frames frames of the format.  Writes <workdir>/<name>.raw for every result (the test compares them
// with bytes it computes through the oracle) and prints one line per check, then OK or FAILED.
#include <cstdio>
#include <fstream>
#include <iterator>
#include <string>
#include <vector>

#include "Controller.hpp"
#include "Logger.hpp"

static void write_raw(const std::string &path, const std::vector<unsigned char> &v)
{
    std::ofstream f(path, std::ios::binary);
    f.write(reinterpret_cast<const char *>(v.data()), (std::streamsize)v.size());
}

int main(int argc, char **argv)
{
    if (argc < 6) {
        std::fprintf(stderr, "usage: bayer_packed_dropin <workdir> <format code> <width> <height> <n_frames>\n");
        return 2;
    }
    const std::string work = argv[1];
    const int fmt = std::stoi(argv[2]), W = std::stoi(argv[3]), H = std::stoi(argv[4]), N = std::stoi(argv[5]);
    if (fmt < RIP_FMT_BAYER_RGGB10P_MIPI || fmt > RIP_FMT_BAYER_GBRG12P_GENICAM) {
        std::fprintf(stderr, "format %d is not a packed RIP_FMT_BAYER_*P_* format\n", fmt);
        return 2;
    }
    const int bits = (fmt - RIP_FMT_BAYER_RGGB10P_MIPI) % 8 < 4 ? 10 : 12;
    std::ifstream f(work + "/in.raw", std::ios::binary);
    std::vector<unsigned char> in((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    const size_t frame = (size_t)W * H * bits / 8;   // rows of W*5/4 or W*3/2 bytes, no padding
    if (in.size() != frame * N) {
        std::fprintf(stderr, "in.raw holds %zu bytes, %d frames of %dx%d need %zu\n", in.size(), N, W, H, frame * N);
        return 2;
    }
    Logger &logger = Logger::getInstance();
    logger.setLogLevel(Logger::LogLevel::ERROR);
    Controller controller;
    std::vector<cl_platform_id> platforms = controller.GetPlatforms();
    std::vector<cl_device_id> devices = controller.GetDevices(platforms[0]);
    cl_context context = controller.CreateContext(platforms[0], devices);
    cl_command_queue queue = controller.CreateCommandQueue(context, devices[0]);
    int failures = 0;
    auto expect = [&](bool ok, const char *what) {
        std::printf("%s: %s\n", what, ok ? "ok" : "FAILED");
        if (!ok) failures++;
    };
    const int ksize = 5;
    const float sigma = 1.5f;
    std::vector<cl_ulong> events;
    cl_int w = W, h = H;

    // whole batches, sharded over every device of the context
    for (const char *method : {"GRAYSCALE", "GAUSSIAN", "EDGE", "FUSED"}) {
        std::vector<unsigned char> out;
        controller.PerformBatch(method, &context, &events, in.data(), N, &out, w, h, logger, fmt, ksize, sigma, in.size());
        const size_t want = (size_t)W * H * N * (std::string(method) == "GAUSSIAN" ? 4 : 1);
        expect(out.size() == want, (std::string("PerformBatch ") + method + " size").c_str());
        write_raw(work + "/batch_" + method + ".raw", out);
    }

    // the fused call of the camera loop, on the first frame
    {
        std::vector<unsigned char> one(in.begin(), in.begin() + frame), out;
        int ks = ksize;
        float sg = sigma;
        controller.PerformFused(ks, sg, &context, &queue, nullptr, &events, &one, &out, w, h, logger, fmt);
        expect(out.size() == (size_t)W * H, "PerformFused size");
        write_raw(work + "/fused_frame0.raw", out);
    }

    // per frame, three in flight: GAUSSIAN on every frame, results in submission order
    {
        std::vector<std::vector<unsigned char>> ins(N), outs(N);
        std::vector<int> handles(N, 0);
        std::vector<unsigned char> all;
        bool ok = true;
        for (int i = 0; i < N; i++) ins[i].assign(in.begin() + frame * i, in.begin() + frame * (i + 1));
        int next_collect = 0;
        for (int i = 0; i < N; i++) {
            handles[i] = controller.SubmitFrame("GAUSSIAN", &queue, &ins[i], &outs[i], w, h, logger, fmt, ksize, sigma);
            ok = ok && handles[i] != 0;
            if (i - next_collect == 2) ok = controller.CollectFrame(handles[next_collect++], &events, logger) && ok;
        }
        while (next_collect < N) ok = controller.CollectFrame(handles[next_collect++], &events, logger) && ok;
        for (int i = 0; i < N; i++) all.insert(all.end(), outs[i].begin(), outs[i].end());
        expect(ok && all.size() == (size_t)W * H * 4 * N, "SubmitFrame/CollectFrame GAUSSIAN");
        write_raw(work + "/submit_GAUSSIAN.raw", all);
    }

    // rejections: a buffer one byte short of its frames, and frames narrower or shorter than 3
    {
        std::vector<unsigned char> out;
        controller.PerformBatch("GRAYSCALE", &context, &events, in.data(), N, &out, w, h, logger, fmt, ksize, sigma, in.size() - 1);
        expect(out.empty(), "PerformBatch rejects a short buffer");
        std::vector<unsigned char> short_in(in.begin(), in.begin() + frame - 1), out2;
        expect(controller.SubmitFrame("GRAYSCALE", &queue, &short_in, &out2, w, h, logger, fmt) == 0 && out2.empty(),
               "SubmitFrame rejects a short frame");
        cl_int two = 2, two_h = 2, odd = bits == 10 ? 6 : 5;   // a width whose rows are not whole bytes or groups
        std::vector<unsigned char> out3, out4, out5, out6;
        controller.PerformBatch("GAUSSIAN", &context, &events, in.data(), 1, &out3, two, h, logger, fmt, ksize, sigma);
        expect(out3.empty(), "PerformBatch rejects a width of 2");
        controller.PerformBatch("GRAYSCALE", &context, &events, in.data(), 1, &out4, w, two, logger, fmt, ksize, sigma);
        expect(out4.empty(), "PerformBatch rejects a height of 2");
        controller.PerformBatch("EDGE", &context, &events, in.data(), 1, &out6, odd, h, logger, fmt, ksize, sigma);
        expect(out6.empty(), "PerformBatch rejects a width that breaks the packing");
        std::vector<unsigned char> tiny(in.begin(), in.begin() + 8);
        expect(controller.SubmitFrame("EDGE", &queue, &tiny, &out5, two, two_h, logger, fmt) == 0 && out5.empty(),
               "SubmitFrame rejects a 2 x 2 frame");
    }

    controller.Cleanup(0, queue);
    controller.Cleanup(context);
    std::printf("%s\n", failures ? "FAILED" : "OK");
    return failures ? 1 : 0;
}
