// The reference's applications wired as KPN graphs on GPU blocks, fed from its wire formats (SURVEY 8f rank 4):
//
//   ook   <capture.iq> <n_blocks> <expected.txt>
//         iq_file_source_u8 (raw rtl_sdr capture, 512-sample blocks as read_async delivers them, bitfount.rs:16-34)
//           -> batch (n_blocks messages -> one capture) -> kpn_gpu::ook_decode
//           -> split_protocols -> protocol A (36 bits): fork -> binconv([4,8,4,12,8]) and binconv([4,8,2,10,12])
//                                 protocol B (24 bits): applicator(|x| {x.push(0); x})          (ratpak.rs:60-123)
//         every field tuple must equal the expected file's (written by tests/test_gpu_kpn.py from the bits the synthetic
//         capture was built to carry AND from the CPU oracle's decode of the same capture).
//   ook_stream <capture.iq> <k> <expected.txt>
//         the same graph as a live receiver runs it: iq_file_source_u8 -> batch(k) (the last message holds what is left)
//           -> kpn_gpu::ook_decode_stream (state carried on the device from message to message) -> split_protocols -> ...
//         k is meant not to divide a burst's length: packets cross message boundaries.  The expected file is the `ook`
//         mode's for the whole capture.
//   psd   <file.wav> <rate> <chunk> <k_avg> <expected.f32>
//         wav_source_complex_chunks (wavio.rs:30-46 as Vec chunks) -> kpn_gpu::chain_psd (FIR64/10 -> Hann FFT1024 -> |X|^2)
//         rows within 1e-4 x RMS of the expected rows (oracle FIR + f64 PSD, per chunk).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include "gpu_blocks.hpp"
#include "sources.hpp"
using namespace kpn;
using kpn_gpu::cf32;

#define CHECK(c) do { if (!(c)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

// n_blocks chunk messages -> one batch message (what kpn_gpu::ook_decode consumes); a trailing partial batch is dropped
static void batch(Receiver<std::vector<uint8_t>> u, Sender<std::vector<uint8_t>> v, size_t n_blocks)
{
    for (;;) {
        std::vector<uint8_t> cap;
        for (size_t k = 0; k < n_blocks; ++k) {
            std::vector<uint8_t> x = u.recv();
            cap.insert(cap.end(), x.begin(), x.end());
        }
        v.send(std::move(cap));
    }
}

// like batch, but the end of the input sends what was collected: a live stream has no whole number of messages
static void batch_flush(Receiver<std::vector<uint8_t>> u, Sender<std::vector<uint8_t>> v, size_t n_blocks)
{
    for (;;) {
        std::vector<uint8_t> cap;
        try {
            for (size_t k = 0; k < n_blocks; ++k) {
                std::vector<uint8_t> x = u.recv();
                cap.insert(cap.end(), x.begin(), x.end());
            }
        } catch (const PortClosed &) {
            if (!cap.empty()) v.send(std::move(cap));
            throw;
        }
        v.send(std::move(cap));
    }
}

static int app_ook(int argc, char **argv, bool streaming)
{
    if (argc < 5) { std::printf("usage: ook|ook_stream capture.iq n_blocks|k expected.txt\n"); return 2; }
    const std::string cap = argv[2], expf = argv[4];
    const size_t n_blocks = (size_t)std::atol(argv[3]);
    kpn_gpu::Gpu gpu(0);
    auto [s0, r0] = channel<std::vector<uint8_t>>();
    auto [s1, r1] = channel<std::vector<uint8_t>>();
    auto [s2, r2] = channel<kpn_gpu::OokPacket>();
    auto [sa, ra] = channel<std::vector<size_t>>();
    auto [sb, rb] = channel<std::vector<size_t>>();
    auto [sa1, ra1] = channel<std::vector<size_t>>();
    auto [sa2, ra2] = channel<std::vector<size_t>>();
    auto [sf1, rf1] = channel<std::vector<size_t>>();
    auto [sf2, rf2] = channel<std::vector<size_t>>();
    auto [sfb, rfb] = channel<std::vector<size_t>>();
    std::thread t0 = spawn([s = std::move(s0), cap]() mutable { iq_file_source_u8(std::move(s), cap, 512); });
    std::thread t1 = spawn([r = std::move(r0), s = std::move(s1), n_blocks, streaming]() mutable {
        if (streaming) batch_flush(std::move(r), std::move(s), n_blocks); else batch(std::move(r), std::move(s), n_blocks); });
    std::thread t2 = spawn([&gpu, r = std::move(r1), s = std::move(s2), n_blocks, streaming]() mutable {
        if (streaming) kpn_gpu::ook_decode_stream(gpu, std::move(r), std::move(s), 1, 256000);
        else kpn_gpu::ook_decode(gpu, std::move(r), std::move(s), 1, n_blocks, 256000); });
    std::thread t3 = spawn([r = std::move(r2), a = std::move(sa), b = std::move(sb)]() mutable {
        kpn_gpu::split_protocols(std::move(r), std::move(a), std::move(b)); });
    // ratpak.rs:98-101: the 36-bit packets fork to BOTH field layouts; :112-119
    std::thread t4 = spawn([r = std::move(ra), a = std::move(sa1), b = std::move(sa2)]() mutable {
        std::vector<Sender<std::vector<size_t>>> outs; outs.push_back(std::move(a)); outs.push_back(std::move(b));
        fork(std::move(r), std::move(outs)); });
    std::thread t5 = spawn([r = std::move(ra1), s = std::move(sf1)]() mutable { binconv(std::move(r), std::move(s), {4, 8, 4, 12, 8}); });
    std::thread t6 = spawn([r = std::move(ra2), s = std::move(sf2)]() mutable { binconv(std::move(r), std::move(s), {4, 8, 2, 10, 12}); });
    // ratpak.rs:120-123: the 24-bit packets get a trailing 0
    std::thread t7 = spawn([r = std::move(rb), s = std::move(sfb)]() mutable {
        applicator(std::move(r), std::move(s), [](std::vector<size_t> x) { x.push_back(0); return x; }); });
    for (std::thread *t : {&t0, &t1, &t2, &t3, &t4, &t5, &t6, &t7}) t->join();
    // expected: lines "A f0 .. f4" (36-bit packets, first layout), "C f0 .. f4" (same packets, second layout),
    // "B b0 .. b23 0" (24-bit packets with the appended 0), each kind in emission order
    std::vector<std::vector<size_t>> want[3];
    std::ifstream in(expf);
    std::string line;
    while (std::getline(in, line)) {
        std::istringstream ls(line);
        char p; ls >> p;
        std::vector<size_t> f; size_t v;
        while (ls >> v) f.push_back(v);
        want[p == 'A' ? 0 : (p == 'C' ? 1 : 2)].push_back(f);
    }
    size_t n_got = 0;
    Receiver<std::vector<size_t>> *rxs[3] = {&rf1, &rf2, &rfb};
    for (int p = 0; p < 3; ++p) {
        for (const auto &w : want[p]) {
            auto got = rxs[p]->try_recv();
            CHECK(got.has_value());
            CHECK(*got == w);
            ++n_got;
        }
        CHECK(!rxs[p]->try_recv().has_value());
    }
    CHECK(n_got >= 1);
    std::printf("kpn app %s OK (%zu packets)\n", streaming ? "ook_stream" : "ook", n_got);
    return 0;
}

static int app_psd(int argc, char **argv)
{
    if (argc < 7) { std::printf("usage: psd file.wav rate chunk k_avg expected.f32\n"); return 2; }
    const std::string wav = argv[2], expf = argv[6];
    const uint32_t rate = (uint32_t)std::atol(argv[3]);
    const size_t chunk = (size_t)std::atol(argv[4]), k_avg = (size_t)std::atol(argv[5]), nfft = 1024;
    kpn_gpu::Gpu gpu(0);
    std::vector<float> taps(64);
    {   // the corrected dsputils::lpf(64, 0.04) (kpn/dsputils.hpp is the product's designer; the driver used the same)
        std::ifstream tf(std::string(argv[6]) + ".taps", std::ios::binary);
        tf.read(reinterpret_cast<char *>(taps.data()), 64 * sizeof(float));
        CHECK(tf.gcount() == (std::streamsize)(64 * sizeof(float)));
    }
    auto [s0, r0] = channel<std::vector<cf32>>();
    auto [s1, r1] = channel<std::vector<float>>();
    std::thread t0 = spawn([s = std::move(s0), wav, rate, chunk]() mutable { wav_source_complex_chunks(std::move(s), wav, rate, chunk); });
    std::thread t1 = spawn([&gpu, r = std::move(r0), s = std::move(s1), taps, k_avg]() mutable {
        kpn_gpu::chain_psd(gpu, std::move(r), std::move(s), taps, 10, 1024, k_avg); });
    t0.join(); t1.join();
    std::ifstream ef2(expf, std::ios::binary | std::ios::ate);
    const size_t n_f = (size_t)ef2.tellg() / sizeof(float);
    ef2.seekg(0);
    std::vector<float> exp_rows(n_f);
    ef2.read(reinterpret_cast<char *>(exp_rows.data()), (std::streamsize)(n_f * sizeof(float)));
    CHECK(n_f % nfft == 0 && n_f >= nfft);
    double rms = 0;
    for (float v : exp_rows) rms += (double)v * v;
    rms = std::sqrt(rms / (double)n_f);
    size_t rows = 0;
    double worst = 0;
    while (auto row = r1.try_recv()) {
        CHECK(row->size() == nfft && (rows + 1) * nfft <= n_f);
        for (size_t b = 0; b < nfft; ++b) worst = std::max(worst, std::fabs((double)(*row)[b] - (double)exp_rows[rows * nfft + b]));
        ++rows;
    }
    CHECK(rows * nfft == n_f);
    CHECK(worst <= 1e-4 * rms);
    std::printf("kpn app psd OK (%zu rows, max err %.2e x rms)\n", rows, worst / rms);
    return 0;
}

int main(int argc, char **argv)
{
    if (argc >= 2 && !std::strcmp(argv[1], "ook")) return app_ook(argc, argv, false);
    if (argc >= 2 && !std::strcmp(argv[1], "ook_stream")) return app_ook(argc, argv, true);
    if (argc >= 2 && !std::strcmp(argv[1], "psd")) return app_psd(argc, argv);
    std::printf("usage: test_gpu_apps ook|ook_stream|psd ...\n");
    return 2;
}
