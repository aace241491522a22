// qcnn_gpu -- the reference's driver (inference/kernel.cu:74-138: main -> run_all -> testqvrcnn)
// rebuilt on the shim classes.  Same positional CLI:   qcnn_gpu <ori.yuv> <anchor_prefix> <H> <W>
// with the anchor file named <prefix>Q<qp>.yuv (kernel.cu:124), the same report lines
// ("before net:PSNR=", "after quantized net:PSNR=", "time:") appended to log.txt and the PSNR double
// appended to recon_psnr.data (kernel.cu:107-115).  Additions, all optional trailing arguments:
//   --model <printf-template with %d for QP>   (the reference hard-codes D:\...\qvrcnn_nchw_vect_c_8bit_qfp_%d.data)
//   --qp <list>  e.g. 22,27,32,37 (reference loop: 22 only, kernel.cu:122)   --frames <n>
//   --gpus <n>   frame-sharded over n devices, one host thread per device (no communication;
//                the exact int64 SSE partial sums are added on the host)
//   --save-recon <file>
//   --strips <n> every frame is cut into n horizontal strips, strip i on device i mod <gpus> (one host thread per device): the
//                single-very-large-frame partition.  Each GPU uploads only its own rows; the 6 halo rows either side are
//                read by the kernel from the neighbour GPU's memory over NVLink (qv_strip_*), no host synchronisation
//                and no collective between frames
//   --stream     files in, file out through qv_stream_yuv: the sequence is never held in host memory (reader thread,
//                GPU stage and writer thread overlap); PSNR from the exact on-device SSE.  With --strips: the strips read and
//                write their own rows of each frame through qv_strip_stream_yuv_pf, so not even a whole frame is held
//   --psnr-pf    after the report, the per-frame PSNR of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112), one line
//                "PSNR of Frame %d:%f" per frame, then the mean of the per-frame PSNR before and after the net.  Default mode
//                and --gpus: from the host buffers; --stream: qv_stream_yuv_pf; --strips: qv_strip_forward_sse, every strip
//                uploads its rows of the original and the host adds the strips' SSEs; --strips --stream: qv_strip_stream_yuv_pf
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <unistd.h>

#include <cuda_runtime.h>

#include "qvrcnn.cuh"

struct Options {
    std::string model_tmpl = "qvrcnn_nchw_vect_c_8bit_qfp_%d.data";
    std::vector<int> qps{22};
    int frames = 1, gpus = 1, strips = 0;
    std::string save_recon;
    bool stream = false, psnr_pf = false;
};

// --psnr-pf: the lines of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112, format of yuv_data.h) from per-frame SSEs of the
// anchor (before) and of the reconstruction (after), then the means of the per-frame PSNR
static void print_psnr_pf(const std::vector<int64_t> &before, const std::vector<int64_t> &after, size_t fpx)
{
    double mb = 0, ma = 0;
    for (size_t n = 0; n < after.size(); ++n) {
        const double pa = qv_psnr_from_sse(after[n], fpx);
        printf("PSNR of Frame %d:%f\n", (int)n, pa);
        ma += pa;
        mb += qv_psnr_from_sse(before[n], fpx);
    }
    const double k = after.empty() ? 1.0 : (double)after.size();
    printf("mean per-frame PSNR: before net:%f after quantized net:%f\n", mb / k, ma / k);
}

static void report(const char *input_fn, int frame, int height, int width, double psnr1, double psnr2, long long us)
{
    time_t now = time(0);
    FILE *logfile = fopen("log.txt", "a+");
    if (!logfile) printf("write file failed\n");
    else {
        fprintf(logfile, "\nQVRCNN test date:%sdata:%s\nframes:%d\nheight:%d\nwidth:%d\nbefore net:PSNR=%f\nafter quantized net:PSNR=%f\ntime:%lldus\n",
                ctime(&now), input_fn, frame, height, width, psnr1, psnr2, us);
        fclose(logfile);
    }
    logfile = fopen("recon_psnr.data", "ab+");
    if (!logfile) printf("open psnr file failed\n");
    else { fwrite(&psnr2, sizeof(double), 1, logfile); fclose(logfile); }
}

// --strips: image rows [r0[i], r1[i]) of every frame on handle i, on device i mod --gpus; neighbours attached.
static std::vector<qv_net *> make_strips(const char *model_fn, int channel, int height, int width, const Options &opt,
                                         std::vector<int> &r0, std::vector<int> &r1)
{
    const int S = opt.strips, G = opt.gpus;
    auto die = [](const char *what) { printf("%s: %s\n", what, qv_last_error()); exit(1); };
    std::vector<qv_net *> nets(S, nullptr);
    std::vector<qv_strip_desc> desc(S);
    r0.assign(S, 0); r1.assign(S, 0);
    for (int i = 0; i < S; ++i) {
        r0[i] = height / S * i + std::min(i, height % S);
        r1[i] = r0[i] + height / S + (i < height % S ? 1 : 0);
        if (qv_create(i % G, 1, channel, r1[i] - r0[i], width, &nets[i])) die("qv_create");
        const int rc = qv_load_static_para(nets[i], model_fn);
        if (rc == QV_ERR_IO) { printf("cannot open model file.\n"); exit(1); }          // qvrcnn.cu:50-54
        if (rc || qv_strip_setup(nets[i], height, r0[i], r1[i]) || qv_strip_export(nets[i], &desc[i])) die("strip setup");
    }
    for (int i = 0; i < S; ++i) {
        if (i > 0 && qv_strip_attach(nets[i], QV_STRIP_ABOVE, &desc[i - 1])) die("qv_strip_attach");
        if (i + 1 < S && qv_strip_attach(nets[i], QV_STRIP_BELOW, &desc[i + 1])) die("qv_strip_attach");
    }
    return nets;
}

// --save-recon with a streaming mode: created and sized ONCE here; the workers open it without truncation and fill their
// own frame ranges or rows (no truncation race, no stale tail frames of an older, longer file)
static void create_recon_file(const std::string &path, int frame, size_t fpx)
{
    FILE *fr = fopen(path.c_str(), "wb");
    if (!fr || ftruncate(fileno(fr), (off_t)((long long)frame * (long long)(fpx + fpx / 2))) != 0) {
        printf("open file failed. (%s)\n", path.c_str());
        exit(1);
    }
    fclose(fr);
}

// --strips: the frame loop of kernel.cu:91-97 with every frame cut into horizontal strips, one strip per handle.
static void testqvrcnn_strips(const char *ori_fn, const char *input_fn, const char *model_fn, int frame, int channel, int height,
                              int width, const Options &opt)
{
    vrcnn_data test_data(frame, height, width);
    test_data.read_data(ori_fn, input_fn);
    const int S = opt.strips, G = opt.gpus;
    const size_t W = (size_t)width, fpx = (size_t)channel * height * width;
    std::vector<int> r0, r1;
    std::vector<qv_net *> nets = make_strips(model_fn, channel, height, width, opt, r0, r1);
    // One host thread per DEVICE.  A device with a single strip (the layout this mode is for) runs a two-slot pipeline on two
    // streams: the upload of frame k+1 overlaps the compute of frame k, the forwards stay in frame order.  A device that
    // hosts several strips (more strips than GPUs: a test layout) drives all of them on ONE stream, frame by frame, all
    // loads before the forwards: strips on one GPU are ordered by stream order, never by kernels waiting for each other.
    std::vector<std::string> errs(G);
    std::vector<int64_t> sse_b(opt.psnr_pf ? frame : 0, 0), sse_a(opt.psnr_pf ? frame : 0, 0);      // summed over the strips
    std::mutex sse_mu;
    auto t0 = std::chrono::steady_clock::now();
    {
        std::vector<std::thread> th;
        for (int g = 0; g < G; ++g)
            th.emplace_back([&, g] {
                std::vector<int> mine;
                for (int i = g; i < S; i += G) mine.push_back(i);
                if (mine.empty()) return;
                const bool solo = mine.size() == 1;
                cudaStream_t st[2] = {nullptr, nullptr};
                cudaEvent_t ev = nullptr;
                std::vector<uint8_t *> d_out(mine.size() * 2, nullptr), d_ori(opt.psnr_pf ? mine.size() * 2 : 0, nullptr);
                int64_t *d_sse = nullptr;                          // --psnr-pf: [strip j][frame][2]
                bool ok = cudaSetDevice(g) == cudaSuccess && cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess;
                for (int s = 0; s < 2 && ok; ++s) ok = cudaStreamCreateWithFlags(&st[s], cudaStreamNonBlocking) == cudaSuccess;
                for (size_t j = 0; j < mine.size() && ok; ++j)
                    for (int s = 0; s < 2 && ok; ++s)
                        ok = cudaMalloc(&d_out[j * 2 + s], (size_t)(r1[mine[j]] - r0[mine[j]]) * W) == cudaSuccess;
                for (size_t j = 0; j < d_ori.size() && ok; ++j) ok = cudaMalloc(&d_ori[j], (size_t)(r1[mine[j / 2]] - r0[mine[j / 2]]) * W) == cudaSuccess;
                const size_t sse_bytes = mine.size() * (size_t)frame * 2 * sizeof(int64_t);
                if (opt.psnr_pf && ok) ok = cudaMalloc(&d_sse, sse_bytes) == cudaSuccess && cudaMemset(d_sse, 0, sse_bytes) == cudaSuccess;
                if (!ok) errs[g] = "CUDA setup failed";
                for (int k = 0; k < frame && ok; ++k) {
                    const int s = k & 1;
                    cudaStream_t q = solo ? st[s] : st[0];
                    for (size_t j = 0; j < mine.size() && ok; ++j)
                        ok = qv_strip_load(nets[mine[j]], s, test_data.input + (size_t)k * fpx + (size_t)r0[mine[j]] * W, q) == QV_OK;
                    if (ok && solo && k > 0) ok = cudaStreamWaitEvent(q, ev, 0) == cudaSuccess;
                    for (size_t j = 0; j < d_ori.size() / 2 && ok; ++j)      // this strip's rows of the original, same slot scheme
                        ok = cudaMemcpyAsync(d_ori[j * 2 + s], test_data.ori + (size_t)k * fpx + (size_t)r0[mine[j]] * W,
                                             (size_t)(r1[mine[j]] - r0[mine[j]]) * W, cudaMemcpyHostToDevice, q) == cudaSuccess;
                    for (size_t j = 0; j < mine.size() && ok; ++j)
                        ok = (opt.psnr_pf ? qv_strip_forward_sse(nets[mine[j]], s, d_ori[j * 2 + s], d_out[j * 2 + s],
                                                                 d_sse + (j * (size_t)frame + k) * 2, q)
                                          : qv_strip_forward(nets[mine[j]], s, d_out[j * 2 + s], q)) == QV_OK;
                    if (ok && solo) ok = cudaEventRecord(ev, q) == cudaSuccess;
                    for (size_t j = 0; j < mine.size() && ok; ++j) {
                        const int i = mine[j];
                        ok = cudaMemcpyAsync(test_data.recon + (size_t)k * fpx + (size_t)r0[i] * W, d_out[j * 2 + s], (size_t)(r1[i] - r0[i]) * W,
                                             cudaMemcpyDeviceToHost, q) == cudaSuccess;
                    }
                }
                if (!ok && errs[g].empty()) errs[g] = qv_last_error();      // thread-local: copy it here
                for (int s = 0; s < 2; ++s)
                    if (st[s] && qv_synchronize(nets[mine[0]], st[s]) != QV_OK && errs[g].empty()) errs[g] = qv_last_error();
                for (size_t j = 1; j < mine.size(); ++j)
                    if (qv_synchronize(nets[mine[j]], st[0]) != QV_OK && errs[g].empty()) errs[g] = qv_last_error();
                if (d_sse && errs[g].empty()) {
                    std::vector<int64_t> h(mine.size() * (size_t)frame * 2);
                    if (cudaMemcpy(h.data(), d_sse, sse_bytes, cudaMemcpyDeviceToHost) != cudaSuccess) errs[g] = "copy of the SSEs failed";
                    std::lock_guard<std::mutex> l(sse_mu);
                    for (size_t j = 0; j < mine.size(); ++j)
                        for (int k = 0; k < frame; ++k) { sse_b[k] += h[(j * frame + k) * 2]; sse_a[k] += h[(j * frame + k) * 2 + 1]; }
                }
                cudaFree(d_sse);
                for (uint8_t *p : d_ori) cudaFree(p);
                for (uint8_t *p : d_out) cudaFree(p);
                for (int s = 0; s < 2; ++s) if (st[s]) cudaStreamDestroy(st[s]);
                if (ev) cudaEventDestroy(ev);
            });
        for (auto &t : th) t.join();
    }
    auto t1 = std::chrono::steady_clock::now();
    const long long us = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
    for (int g = 0; g < G; ++g)
        if (!errs[g].empty()) { printf("GPU %d: %s\n", g, errs[g].c_str()); exit(1); }
    for (auto *n : nets) qv_destroy(n);
    if (!opt.save_recon.empty()) test_data.save_recon_as(opt.save_recon.c_str());
    const double psnr1 = test_data.psnr(test_data.input), psnr2 = test_data.psnr(test_data.recon);
    printf("\nbefore net:PSNR=%.3f\nafter quantized net:PSNR=%.3f\ntime:%lldus\n", psnr1, psnr2, us);
    printf("throughput:%.1f Mpixel/s (%d frame(s) of %dx%d in %d strip(s) on %d GPU(s), halo rows over peer-mapped memory, copies included)\n",
           (double)frame * fpx / (double)us, frame, width, height, S, G);
    report(input_fn, frame, height, width, psnr1, psnr2, us);
    if (opt.psnr_pf) print_psnr_pf(sse_b, sse_a, fpx);
}

static void testqvrcnn(const char *ori_fn, const char *input_fn, const char *model_fn, int frame, int channel, int height,
                       int width, const Options &opt)
{
    vrcnn_data test_data(frame, height, width);
    test_data.read_data(ori_fn, input_fn);
    const size_t fpx = (size_t)channel * height * width;
    const int G = opt.gpus;
    std::vector<qvrcnn *> nets(G, nullptr);
    for (int g = 0; g < G; ++g) {
        int nf = frame / G + (g < frame % G ? 1 : 0);
        nets[g] = new qvrcnn(g, nf > 0 ? std::min(nf, 8) : 1, channel, height, width);   // GPU_num,NCHW
        nets[g]->load_static_para(model_fn);
    }
    auto t0 = std::chrono::steady_clock::now();
    if (G == 1 && frame == 1) {
        // the reference's own per-frame sequence (kernel.cu:91-97)
        nets[0]->load_data(test_data.input);
        nets[0]->forward_blu();
        cudaMemcpy(test_data.recon, (datatype *)nets[0]->I1.x_rec, fpx, cudaMemcpyDeviceToHost);
    } else {
        std::vector<std::thread> th;
        int f0 = 0;
        for (int g = 0; g < G; ++g) {
            int nf = frame / G + (g < frame % G ? 1 : 0);
            th.emplace_back([&, g, f0, nf] {
                if (nf > 0) nets[g]->forward_frames(test_data.input + (size_t)f0 * fpx, test_data.recon + (size_t)f0 * fpx, nf);
            });
            f0 += nf;
        }
        for (auto &t : th) t.join();
    }
    auto t1 = std::chrono::steady_clock::now();
    long long us = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
    for (auto *n : nets) delete n;
    if (!opt.save_recon.empty()) test_data.save_recon_as(opt.save_recon.c_str());
    double psnr1 = test_data.psnr(test_data.input);
    double psnr2 = test_data.psnr(test_data.recon);
    printf("\nbefore net:PSNR=%.3f\nafter quantized net:PSNR=%.3f\ntime:%lldus\n", psnr1, psnr2, us);
    printf("throughput:%.1f Mpixel/s (%d frame(s) of %dx%d on %d GPU(s), host buffers, copies included)\n",
           (double)frame * fpx / (double)us, frame, width, height, G);
    report(input_fn, frame, height, width, psnr1, psnr2, us);
    if (opt.psnr_pf) {
        std::vector<int64_t> b(frame), a(frame);
        for (int n = 0; n < frame; ++n) {
            qv_psnr(test_data.input + (size_t)n * fpx, test_data.ori + (size_t)n * fpx, fpx, &b[n]);
            qv_psnr(test_data.recon + (size_t)n * fpx, test_data.ori + (size_t)n * fpx, fpx, &a[n]);
        }
        print_psnr_pf(b, a, fpx);
    }
}

// --stream: the same report from the streaming pipeline.  Each GPU takes a contiguous frame range and fills its own part
// of the reconstruction file; the SSE partial sums are exact integers, so their sum is the sequential result.
static void testqvrcnn_stream(const char *ori_fn, const char *input_fn, const char *model_fn, int frame, int channel, int height,
                              int width, const Options &opt)
{
    const int G = opt.gpus;
    const size_t fpx = (size_t)channel * height * width;
    std::vector<qv_net *> nets(G, nullptr);
    for (int g = 0; g < G; ++g) {
        if (qv_create(g, std::min(std::max(frame / G, 1), 8), channel, height, width, &nets[g]) || qv_load_static_para(nets[g], model_fn)) {
            printf("%s\n", qv_last_error());
            exit(1);
        }
    }
    std::vector<int64_t> pf_b(frame, 0), pf_a(frame, 0);              // per frame; GPU g fills its own frame range
    std::vector<int> rcs(G, 0);
    std::vector<std::string> errs(G);
    if (!opt.save_recon.empty()) create_recon_file(opt.save_recon, frame, fpx);
    auto t0 = std::chrono::steady_clock::now();
    {
        std::vector<std::thread> th;
        int f0 = 0;
        for (int g = 0; g < G; ++g) {
            const int nf = frame / G + (g < frame % G ? 1 : 0);
            th.emplace_back([&, g, f0, nf] {
                rcs[g] = qv_stream_yuv_pf(nets[g], input_fn, ori_fn, opt.save_recon.empty() ? nullptr : opt.save_recon.c_str(), f0, nf,
                                          pf_b.data() + f0, pf_a.data() + f0);
                if (rcs[g]) errs[g] = qv_last_error();                      // thread-local: copy it in this thread
            });
            f0 += nf;
        }
        for (auto &t : th) t.join();
    }
    auto t1 = std::chrono::steady_clock::now();
    const long long us = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
    long long b = 0, a = 0;
    for (int g = 0; g < G; ++g) {
        if (rcs[g]) { printf("%s\n", errs[g].c_str()); exit(1); }
        qv_destroy(nets[g]);
    }
    for (int n = 0; n < frame; ++n) { b += pf_b[n]; a += pf_a[n]; }
    const double psnr1 = qv_psnr_from_sse(b, (size_t)frame * fpx), psnr2 = qv_psnr_from_sse(a, (size_t)frame * fpx);
    printf("\nbefore net:PSNR=%.3f\nafter quantized net:PSNR=%.3f\ntime:%lldus\n", psnr1, psnr2, us);
    printf("throughput:%.1f Mpixel/s (%d frame(s) of %dx%d on %d GPU(s), streamed from and to files)\n",
           (double)frame * fpx / (double)us, frame, width, height, G);
    report(input_fn, frame, height, width, psnr1, psnr2, us);
    if (opt.psnr_pf) print_psnr_pf(pf_b, pf_a, fpx);
}

// --strips --stream: the --strips partition fed from and to files through qv_strip_stream_yuv_pf -- every handle reads and
// writes only its own rows of each frame, so neither the sequence nor a whole frame is ever held in host memory.
static void testqvrcnn_strips_stream(const char *ori_fn, const char *input_fn, const char *model_fn, int frame, int channel,
                                     int height, int width, const Options &opt)
{
    const int S = opt.strips, G = opt.gpus;
    const size_t fpx = (size_t)channel * height * width;
    std::vector<int> r0, r1;
    std::vector<qv_net *> nets = make_strips(model_fn, channel, height, width, opt, r0, r1);
    if (!opt.save_recon.empty()) create_recon_file(opt.save_recon, frame, fpx);
    std::vector<int64_t> pf_b(frame, 0), pf_a(frame, 0);              // per frame, summed over the strips
    auto t0 = std::chrono::steady_clock::now();
    const int rc = qv_strip_stream_yuv_pf(nets.data(), S, input_fn, ori_fn, opt.save_recon.empty() ? nullptr : opt.save_recon.c_str(),
                                          0, frame, pf_b.data(), pf_a.data());
    auto t1 = std::chrono::steady_clock::now();
    if (rc) { printf("%s\n", qv_last_error()); exit(1); }
    const long long us = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
    for (auto *n : nets) qv_destroy(n);
    long long b = 0, a = 0;
    for (int n = 0; n < frame; ++n) { b += pf_b[n]; a += pf_a[n]; }
    const double psnr1 = qv_psnr_from_sse(b, (size_t)frame * fpx), psnr2 = qv_psnr_from_sse(a, (size_t)frame * fpx);
    printf("\nbefore net:PSNR=%.3f\nafter quantized net:PSNR=%.3f\ntime:%lldus\n", psnr1, psnr2, us);
    printf("throughput:%.1f Mpixel/s (%d frame(s) of %dx%d in %d strip(s) on %d GPU(s), halo rows over peer-mapped memory, "
           "streamed from and to files)\n", (double)frame * fpx / (double)us, frame, width, height, S, G);
    report(input_fn, frame, height, width, psnr1, psnr2, us);
    if (opt.psnr_pf) print_psnr_pf(pf_b, pf_a, fpx);
}

static int run_all(const char *oriname, const char *inputname, int height, int width, const Options &opt)
{
    for (int qp : opt.qps) {
        char input_fn[512], model_fn[512];
        snprintf(input_fn, sizeof(input_fn), "%sQ%d.yuv", inputname, qp);           // kernel.cu:124
        snprintf(model_fn, sizeof(model_fn), opt.model_tmpl.c_str(), qp);           // kernel.cu:125
        if (opt.strips > 0 && opt.stream) testqvrcnn_strips_stream(oriname, input_fn, model_fn, opt.frames, 1, height, width, opt);
        else if (opt.strips > 0) testqvrcnn_strips(oriname, input_fn, model_fn, opt.frames, 1, height, width, opt);
        else if (opt.stream) testqvrcnn_stream(oriname, input_fn, model_fn, opt.frames, 1, height, width, opt);
        else testqvrcnn(oriname, input_fn, model_fn, opt.frames, 1, height, width, opt);
    }
    return 0;
}

int main(int argc, char **argv)
{
    if (argc < 5) {
        fprintf(stderr, "usage: %s <ori.yuv> <anchor_prefix> <H> <W> [--model tmpl%%d] [--qp 22,27,..] [--frames n] [--gpus n] [--save-recon f] [--stream] [--strips n] [--psnr-pf]\n", argv[0]);
        return 2;
    }
    Options opt;
    for (int i = 5; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "--model" && i + 1 < argc) opt.model_tmpl = argv[++i];
        else if (a == "--frames" && i + 1 < argc) opt.frames = atoi(argv[++i]);
        else if (a == "--gpus" && i + 1 < argc) opt.gpus = atoi(argv[++i]);
        else if (a == "--save-recon" && i + 1 < argc) opt.save_recon = argv[++i];
        else if (a == "--strips" && i + 1 < argc) opt.strips = atoi(argv[++i]);
        else if (a == "--stream") opt.stream = true;
        else if (a == "--psnr-pf") opt.psnr_pf = true;
        else if (a == "--qp" && i + 1 < argc) {
            opt.qps.clear();
            for (char *t = strtok(argv[++i], ","); t; t = strtok(nullptr, ",")) opt.qps.push_back(atoi(t));
        } else { fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    if (opt.frames < 1 || opt.gpus < 1 || opt.strips < 0) { fprintf(stderr, "bad --frames/--gpus/--strips\n"); return 2; }
    return run_all(argv[1], argv[2], atoi(argv[3]), atoi(argv[4]), opt);
}
