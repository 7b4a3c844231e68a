// kpn_gpu::fast_fir_multi in a threaded graph: 6 channels, chunk by chunk; each channel's outputs must be a bitwise prefix
// of lrc_fastfir_run over the channel's whole input (flush = 1), for a plan on each overlap-save kernel.
#include <cstdio>
#include <random>
#include "gpu_blocks.hpp"
using namespace kpn;
using kpn_gpu::cf32;

#define CHECK(c) do { if (!(c)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

int main()
{
    kpn_gpu::Gpu gpu(0);
    std::mt19937 rng(3);
    std::normal_distribution<float> nd;
    const size_t n_ch = 6;
    // (nh, nfft, chunk, chunks): nfft-point blocks of fastfir_kernel, and 16384-point blocks
    const size_t cases[][4] = {{300, 0, 5000, 7}, {4096, 0, 20000, 5}};
    for (const auto &cs : cases) {
        const size_t nh = cs[0], nfft = cs[1], chunk = cs[2], n_chunks = cs[3], n = chunk * n_chunks;
        std::vector<cf32> h(nh);
        for (auto &v : h) v = cf32(nd(rng), nd(rng)) / 64.f;
        std::vector<Receiver<std::vector<cf32>>> ins; std::vector<Sender<std::vector<cf32>>> outs;
        std::vector<Sender<std::vector<cf32>>> src; std::vector<Receiver<std::vector<cf32>>> sink;
        for (size_t c = 0; c < n_ch; ++c) {
            auto [a, b] = channel<std::vector<cf32>>(); src.push_back(std::move(a)); ins.push_back(std::move(b));
            auto [d, e] = channel<std::vector<cf32>>(); outs.push_back(std::move(d)); sink.push_back(std::move(e));
        }
        std::thread t = spawn([&gpu, i = std::move(ins), o = std::move(outs), h, nfft, chunk]() mutable {
            kpn_gpu::fast_fir_multi(gpu, std::move(i), std::move(o), h, nfft, chunk); });
        std::vector<std::vector<cf32>> x(n_ch, std::vector<cf32>(n));
        for (auto &ch : x) for (auto &s : ch) s = cf32(nd(rng), nd(rng));
        for (size_t k = 0; k < n_chunks; ++k)
            for (size_t c = 0; c < n_ch; ++c) src[c].send(std::vector<cf32>(x[c].begin() + k * chunk, x[c].begin() + (k + 1) * chunk));
        for (auto &s : src) s.drop();
        t.join();

        // the one-shot reference, and the streamed count: every complete compute block of the n samples
        lrc_fastfir *ff = nullptr;
        kpn_gpu::check(lrc_fastfir_create(gpu.ctx, (const float *)h.data(), nh, nfft, &ff), "lrc_fastfir_create");
        const size_t nc = (nh > 1024 || lrc_fastfir_nfft(ff) >= 8192) ? 16384 : lrc_fastfir_nfft(ff), good = nc - nh + 1;
        const size_t want = n >= nc ? ((n - nc) / good + 1) * good : 0;
        const size_t total = lrc_fastfir_out_len(ff, n, 1);
        CHECK(want > 0 && want <= total);
        void *d_in = nullptr, *d_out = nullptr;
        kpn_gpu::cuda_check(cudaMalloc(&d_in, n * sizeof(cf32)), "cudaMalloc");
        kpn_gpu::cuda_check(cudaMalloc(&d_out, total * sizeof(cf32)), "cudaMalloc");
        std::vector<cf32> ref(total);
        for (size_t c = 0; c < n_ch; ++c) {
            std::vector<cf32> y;
            size_t msgs = 0;
            while (auto p = sink[c].try_recv()) { y.insert(y.end(), p->begin(), p->end()); ++msgs; CHECK(p->size() % good == 0); }
            CHECK(msgs > 1);                                               // outputs came while the stream ran
            CHECK(y.size() == want);
            kpn_gpu::cuda_check(cudaMemcpy(d_in, x[c].data(), n * sizeof(cf32), cudaMemcpyHostToDevice), "H2D");
            size_t no = 0;
            kpn_gpu::check(lrc_fastfir_run(ff, (const float *)d_in, n, (float *)d_out, 1, &no, nullptr), "lrc_fastfir_run");
            kpn_gpu::check(lrc_ctx_sync(gpu.ctx), "lrc_ctx_sync");         // the context's stream does not block with cudaMemcpy
            kpn_gpu::cuda_check(cudaMemcpy(ref.data(), d_out, total * sizeof(cf32), cudaMemcpyDeviceToHost), "D2H");
            CHECK(no == total);
            CHECK(std::memcmp(y.data(), ref.data(), want * sizeof(cf32)) == 0);   // bitwise prefix of the one-shot
        }
        cudaFree(d_in); cudaFree(d_out);
        lrc_fastfir_destroy(ff);
    }
    std::printf("kpn fastfir stream OK\n");
    return 0;
}
