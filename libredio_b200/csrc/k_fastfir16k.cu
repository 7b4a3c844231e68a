// k_fastfir16k.cu -- overlap-save in 16384-point blocks: the compute block lrc_fastfir_create picks for every plan with
// nh > 1024 or nfft >= 8192, whatever output length the plan's nfft fixes (the config-5 shape among them).
//
// Why: with nh = 4096 an 8192-point block keeps 4097 of 8192 outputs (50 %), a 16384-point block keeps 12289 of 16384
// (75 %): 1.39x fewer butterflies per output sample (kiss_fastfir.c:81-93 picks the block size by a cost model of
// its own; the result is the same convolution whatever the block size).
//
//   16384 = 16 x 1024,  n = 1024 n1 + n2,  k = k1 + 16 k2
//   P1   column n2: DFT16 over n1 straight from global memory, times W_16384^(n2 k1), into shared row k1
//   P2   warp k1 owns row k1: 1024 points as 32 x 32 in registers (the row buffer itself is the exchange tile),
//        .* H[k1 + 16 k2], inverse transform, back into the row
//   P1'  column n2: times conj(W^(n2 k1)), IDFT16 over k1, outputs 1024 n1 + n2 < ngood to global memory; fused per
//        thread with P1 of the CTA's next block (its loads are in flight during the inverse butterflies) -- no barrier
//        between the two blocks' P1 phases because a column is private to its thread in both.
// Two CTA barriers per block.
//
// Shared-memory layout (round 2).  ncu on the first version (profiles/r2_ff16k_v1_ncu_keys.txt): the FP32 pipe (packed
// FADD2/FFMA2, 2 cycles each) and the shared-memory pipe both need ~12.5 k cycles per block and the top stall was
// mio_throttle (2.4 per issue) -- the LSU instruction queue full of 64-bit shared accesses arriving in bursts of 32.
// So every shared access that can be is now 128 bits wide (half the LSU instructions for the same bytes):
//   row k1, element n2 = l + 32 e  lives at  l * 34 + e   (a 32-entry slab per lane l, padded to 34 so that slabs
//   start 16 bytes apart modulo 128: LDS.128/STS.128 of 8 consecutive lanes hit 8 distinct bank groups)
//   - P2's lane l reads/writes its 32 points x[l + 32 e] as 16 LDS.128 / STS.128; the transposing reads of the two
//     exchanges stay 64-bit (column reads, conflict-free)
//   - a P1 thread (lane l, warp j) owns the column PAIR n2 = l + 64 j and n2 + 32, i.e. e = 2 j and 2 j + 1: adjacent
//     entries of slab l, one STS.128 / LDS.128 per row.  The pair's second twiddle is W_512^k1 (a literal) times the first.
//   - twiddle tables are stored per thread / per lane contiguously (pitch 18 / 34 entries) and read as LDS.128;
//     the inverse uses the same tables conjugated in the multiply; H is stored so that a lane's two consecutive
//     bins are one coalesced LDG.128.
// Shared memory: 16 rows x 1088 complex (136 KB) + 512 x 18 P1 twiddles (72 KB) + 32 x 34 warp-transform twiddles
// (8.5 KB) = 216.5 KB, one 512-thread CTA per SM.
//
// STREAM = true (lrc_fastfir_stream_push): a work item is (channel, block) of many channels (fastfir.cuh), the fused
// P1' / next P1 and the L2 prefetch run across channel boundaries as they do across blocks.  Blocks that start past
// the carried history read the chunk alone (CTA-uniform branch); only the first blocks of a channel's push start inside
// it, and those are loaded at the head of their own iteration rather than fused (no registers for a second source).
// STREAM = false compiles to the instructions of the batch kernel before the stream form existed.
#include "fastfir.cuh"
#include "fft_core.cuh"

using namespace lrfft;

namespace ff16k {
constexpr int N = 16384, NPAIR = 512, ROWS = 16;
constexpr int NT = NPAIR;                        // one column pair per thread, one row per warp
static_assert(NT / 32 == ROWS, "one row per warp");
constexpr int LP = 34;                          // entries per lane slab (32 used)
constexpr int RP = 32 * LP;                     // entries per row
constexpr int DATA_CPX = ROWS * RP;
constexpr int T1P = 18;                         // P1 twiddles per thread: q = 0..15 (+2 pad)
constexpr int TW1_CPX = NPAIR * T1P;
constexpr int TWW_CPX = 32 * LP;                // [lane][r] : W_1024^(lane r)
constexpr int SMEM_BYTES = (DATA_CPX + TW1_CPX + TWW_CPX) * 8;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");

// exp(-2 pi j q / 512), q < 16 (compile-time index after unrolling): W_16384^(32 q)
__device__ __forceinline__ float2 w512(int q)
{
    constexpr float C[16] = {1.00000000000000000000f, 0.99992470183914450299f, 0.99969881869620424997f,
                             0.99932238458834954375f, 0.99879545620517240501f, 0.99811811290014917919f,
                             0.99729045667869020697f, 0.99631261218277800129f, 0.99518472667219692873f,
                             0.99390697000235606051f, 0.99247953459870996706f, 0.99090263542778000971f,
                             0.98917650996478101444f, 0.98730141815785843473f, 0.98527764238894122162f,
                             0.98310548743121628501f};
    constexpr float S[16] = {0.00000000000000000000f, 0.01227153828571992539f, 0.02454122852291228812f,
                             0.03680722294135883171f, 0.04906767432741801493f, 0.06132073630220857829f,
                             0.07356456359966742631f, 0.08579731234443989385f, 0.09801714032956060363f,
                             0.11022220729388305938f, 0.12241067519921619566f, 0.13458070850712616773f,
                             0.14673047445536174793f, 0.15885814333386144570f, 0.17096188876030121717f,
                             0.18303988795514095078f};
    return make_float2(C[q], -S[q]);
}

__device__ __forceinline__ float2 lo(float4 x) { return make_float2(x.x, x.y); }
__device__ __forceinline__ float2 hi(float4 x) { return make_float2(x.z, x.w); }
__device__ __forceinline__ float4 pack(float2 a, float2 b) { return make_float4(a.x, a.y, b.x, b.y); }
__device__ __forceinline__ float2 ldg_nc_f2(const float2 *p)
{
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}

// one 1024-point transform by the calling warp, in place in its lane slabs: on entry and exit v[e] = x[lane + 32 e]
// (entry) / X[lane + 32 e] (exit).  `row`: the warp's RP-entry buffer, free to be overwritten; tww: [lane][r] twiddles.
template <bool INV>
__device__ __forceinline__ void warp_fft1024(float2 *v, float2 *row, const float2 *tww, int lane)
{
    RegFFT<32, INV>::run(v);
    const float4 *tw4 = reinterpret_cast<const float4 *>(tww + lane * LP);
    float4 *slab4 = reinterpret_cast<float4 *>(row + lane * LP);
    __syncwarp();                                        // every lane is done reading the tile (previous exchange)
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const float4 w = tw4[i];
        const float2 a = i ? (INV ? cmul_conjb(v[2 * i], lo(w)) : cmulf(v[2 * i], lo(w))) : v[0];
        const float2 b = INV ? cmul_conjb(v[2 * i + 1], hi(w)) : cmulf(v[2 * i + 1], hi(w));
        slab4[i] = pack(a, b);                           // tile[n2' = lane][k1' = 2 i, 2 i + 1]
    }
    __syncwarp();
    const float2 *col = row + lane;                      // tile[e][k1' = lane]
#pragma unroll
    for (int e = 0; e < 32; ++e) v[e] = col[e * LP];
    RegFFT<32, INV>::run(v);
}
}  // namespace ff16k

// Measured and rejected for the P1 phase (whose global loads cannot be held in registers across P2 at 128 registers/thread):
//   - staging the next block's first column in shared memory with cp.async during P2 (P1 twiddles factorised into two
//     small tables to make room): 121 Gsamples/s against 140 -- 8192 LDGSTS per CTA sit in the LSU queue in front of the
//     barrier (lg_throttle 0.12 -> 0.79, barrier 0.63 -> 1.07 per issue), profiles/r2_ff16k_staged_ncu_phases.txt;
//   - a CTA-uniform fast path with unpredicated loads: 133 against 140;
//   - 256 threads with two column pairs and two rows each at 255 registers, room to request a whole pair of the next block
//     before P2 and the other at the head of the P1 phase, with half the warps to hide everything else: timed against
//     512 threads in tools/runs/r2c.sh, whose 512-thread captures are profiles/r2_r2c_ff16k_512_ncu_keys.txt and
//     r2_r2c_ff16k_512_ncu_phases.txt.
// A TMA tensor copy would take the loads off the LSU, but block starts (multiples of ngood = 12289 samples) are only
// 8-byte aligned every other block.
template <bool STREAM>
__global__ void __launch_bounds__(ff16k::NT, 1)
fastfir16k_kernel(const float2 *__restrict__ in, size_t n_in, float2 *__restrict__ out, size_t n_blocks_full,
                  size_t n_blocks, size_t ngood, size_t flush_keep, const float2 *__restrict__ tw /* W_16384^k */,
                  const float2 *__restrict__ tw1k /* W_1024^k */, const float4 *__restrict__ Hq, FfStreamArgs sa)
{
    using namespace ff16k;
    extern __shared__ __align__(16) float2 ff16k_smem[];
    float2 *sd = ff16k_smem;                         // [16][RP]
    float2 *tw1 = sd + DATA_CPX;                     // [512 pairs][T1P]
    float2 *tww = tw1 + TW1_CPX;                     // [32][LP]
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int i = t; i < TW1_CPX; i += NT) {
        const int pr = i / T1P, q = i % T1P;
        const int col = (pr & 31) + 64 * (pr >> 5);
        tw1[i] = q < 16 ? __ldg(tw + col * q) : make_float2(0.f, 0.f);        // 991 * 15 < 16384
    }
    for (int i = t; i < TWW_CPX; i += NT) {
        const int ln = i / LP, r = i % LP;
        tww[i] = r < 32 ? __ldg(tw1k + ln * r) : make_float2(0.f, 0.f);       // 31 * 31 < 1024
    }
    __syncthreads();

    // this thread's pair: pair index t = lane + 32 warp, columns ca = lane + 64 warp and ca + 32,
    // cells (row q) at sd[q RP + lane LP + 2 warp] (.lo = column ca, .hi = column ca + 32)
    auto twp_of = [&]() { return reinterpret_cast<const float4 *>(tw1 + t * T1P); };
    auto cell_of = [&]() { return reinterpret_cast<float4 *>(sd + lane * LP + 2 * warp); };

    // the 2 x 16 inputs of the column pair of block `blk`; volatile loads: they stay where they are written
    auto p1_load = [&](size_t blk, int ca, float2 *va, float2 *vb) {
        const size_t s0 = blk * ngood;
        const float2 *src = in + s0 + ca;
        if (n_in - s0 >= (size_t)N) {                            // every block but a ragged last one (CTA-uniform)
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                va[r] = ldg_nc_f2(src + 1024 * r);
                vb[r] = ldg_nc_f2(src + 1024 * r + 32);
            }
        } else {
            const int avail = (int)(n_in - s0);
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                va[r] = ca + 1024 * r < avail ? ldg_nc_f2(src + 1024 * r) : make_float2(0.f, 0.f);
                vb[r] = ca + 32 + 1024 * r < avail ? ldg_nc_f2(src + 1024 * r + 32) : make_float2(0.f, 0.f);
            }
        }
    };
    // STREAM: the 16 inputs of column `col` of block bc of channel c (bounds as lim = bound - col against 1024 r literals,
    // so that no column index is held across the loop)
    auto s_load = [&](size_t c, size_t bc, int col, float2 *u) {
        const size_t s0 = bc * ngood;
        const float2 *row = in + c * sa.in_stride;
        const bool whole = n_in - s0 >= (size_t)N;
        const int lim = (whole ? N : (int)(n_in - s0)) - col;
        if (s0 >= sa.held) {                                    // the block lies in the chunk (CTA-uniform)
            const float2 *src = row + (s0 - sa.held) + col;
#pragma unroll
            for (int r = 0; r < 16; ++r)
                u[r] = (whole || 1024 * r < lim) ? ldg_nc_f2(src + 1024 * r) : make_float2(0.f, 0.f);
        } else {                                                // straddles the carried history (held < N)
            const int hlim = (int)(sa.held - s0) - col;
            const float2 *csrc = sa.carry + c * sa.carry_pitch + s0 + col;
            // row + (1024 r - hlim): integer arithmetic, the address is only formed for 1024 r >= hlim
            const uintptr_t xsrc = reinterpret_cast<uintptr_t>(row) - (intptr_t)hlim * (intptr_t)sizeof(float2);
#pragma unroll
            for (int r = 0; r < 16; ++r)
                u[r] = 1024 * r < lim ? ldg_nc_f2(1024 * r < hlim ? csrc + 1024 * r
                                                                  : reinterpret_cast<const float2 *>(xsrc) + 1024 * r)
                                      : make_float2(0.f, 0.f);          // hlim <= lim
        }
    };
    // forward butterflies of the column pair; results into the pair's 16 shared cells
    auto p1_forward = [&](float2 *va, float2 *vb) {
        const float4 *twp = twp_of();
        float4 *cell = cell_of();
        RegFFT<16, false>::run(va);
        RegFFT<16, false>::run(vb);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 w = twp[i];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int q = 2 * i + h;
                const float2 wq = h ? hi(w) : lo(w);
                const float2 a = q ? cmulf(va[q], wq) : va[0];
                const float2 b = q ? cmulf(cmulf(vb[q], w512(q)), wq) : vb[0];
                cell[q * (RP / 2)] = pack(a, b);
            }
        }
    };
    // inverse side of a pair, part 1: cells -> registers, conjugated twiddles
    auto p1_unload = [&](float2 *ua, float2 *ub) {
        const float4 *twp = twp_of();
        const float4 *cell = cell_of();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 w = twp[i];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int q = 2 * i + h;
                const float2 wq = h ? hi(w) : lo(w);
                const float4 x = cell[q * (RP / 2)];
                ua[q] = q ? cmul_conjb(lo(x), wq) : lo(x);
                ub[q] = q ? cmul_conjb(cmul_conjb(hi(x), w512(q)), wq) : hi(x);
            }
        }
    };
    // part 2: IDFT16 of one column, outputs 1024 r + col < keep to global memory
    auto p1_emit = [&](float2 *u, float2 *dst, int col, int keep) {
        RegFFT<16, true>::run(u);
        const int cnt = keep > col ? ((keep - 1 - col) >> 10) + 1 : 0;
#pragma unroll
        for (int r = 0; r < 16; ++r)
            if (r < cnt) __stcs(dst + 1024 * r, u[r]);
    };

    size_t b = blockIdx.x;
    // STREAM: item b is block bc of channel c, tracked without a division per item (CTA-uniform integer arithmetic)
    // A straddling block is loaded at the head of its own iteration instead of in the fused phase, where the 128
    // registers have no room for the second source.
    size_t c = 0, bc = b;
    bool loaded = false;                                        // STREAM: item b's P1 forward is done
    if constexpr (STREAM) {
        while (bc >= sa.nblk) { bc -= sa.nblk; ++c; }
    } else if (b < n_blocks) {
        float2 va[16], vb[16];
        p1_load(b, lane + 64 * warp, va, vb);
        p1_forward(va, vb);
    }
    for (; b < n_blocks; b += gridDim.x) {
        if constexpr (STREAM) {
            if (!loaded) {
                float2 va[16], vb[16];
                s_load(c, bc, lane + 64 * warp, va);
                s_load(c, bc, lane + 64 * warp + 32, vb);
                p1_forward(va, vb);
            }
        }
        const size_t nb = b + gridDim.x;
        const bool more = nb < n_blocks;
        size_t nc = c + sa.step_c, nbc = bc + sa.step_b;           // STREAM: item nb
        if (nbc >= sa.nblk) { nbc -= sa.nblk; ++nc; }
        // the next block's input (1024 lines) is asked into L2 now; its P1 loads come later
        if constexpr (STREAM) {
            if (more) {                                          // the chunk part of the next item
                const size_t s0 = nbc * ngood, from = s0 > sa.held ? s0 : sa.held;
                const char *nsrc = reinterpret_cast<const char *>(in + nc * sa.in_stride + (from - sa.held));
                const size_t lim = (n_in - from) * 8;
#pragma unroll
                for (int k = 0; k < 1024 / NT; ++k) {
                    const size_t off = (size_t)(t + NT * k) * 128;
                    if (off < lim) asm volatile("prefetch.global.L2 [%0];" :: "l"(nsrc + off));
                }
            }
        } else if (more) {
            const char *nsrc = reinterpret_cast<const char *>(in + nb * ngood);
#pragma unroll
            for (int k = 0; k < 1024 / NT; ++k) {
                const size_t off = (size_t)(t + NT * k) * 128;
                if (nb * ngood * 8 + off < n_in * 8) asm volatile("prefetch.global.L2 [%0];" :: "l"(nsrc + off));
            }
        }
        __syncthreads();
        // ---- P2: warp k1 transforms row k1, multiplies by its slice of H, transforms back ----------------------
        {
            const int k1 = warp;
            float2 *row = sd + RP * k1;
            float4 *slab4 = reinterpret_cast<float4 *>(row + lane * LP);
            float2 v[32];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float4 x = slab4[i];
                v[2 * i] = lo(x);
                v[2 * i + 1] = hi(x);
            }
            warp_fft1024<false>(v, row, tww, lane);              // X[k1 + 16 (lane + 32 e)]
            const float4 *hq = Hq + (size_t)k1 * 512 + lane;
#pragma unroll
            for (int i = 0; i < 16; ++i) {                       // C_MUL  kiss_fastfir.c:180-184
                const float4 h = __ldg(hq + 32 * i);
                v[2 * i] = cmulf(v[2 * i], lo(h));
                v[2 * i + 1] = cmulf(v[2 * i + 1], hi(h));
            }
            warp_fft1024<true>(v, row, tww, lane);
            __syncwarp();                                        // the tile reads of the last exchange are done
#pragma unroll
            for (int i = 0; i < 16; ++i) slab4[i] = pack(v[2 * i], v[2 * i + 1]);
        }
        __syncthreads();
        // ---- P1 inverse of this block fused with P1 forward of the CTA's next block -----------------------
        // 128 registers: ua, ub, nxa, nxb are 32 each, so a column of the next block is requested only once a
        // column of this block has left
        const int ca = lane + 64 * warp;
        int keep;
        float2 *dstg;
        bool fuse = more;
        const float2 *src;
        bool whole;
        int avail;
        if constexpr (STREAM) {
            keep = (int)((bc < n_blocks_full) ? ngood : flush_keep);
            dstg = out + c * sa.out_stride + bc * ngood;
            const size_t s0 = nbc * ngood;
            fuse = more && s0 >= sa.held;                        // the next item lies in the chunk
            src = fuse ? in + nc * sa.in_stride + (s0 - sa.held) + ca : in;
            whole = fuse && n_in - s0 >= (size_t)N;
            avail = fuse ? (whole ? N : (int)(n_in - s0)) : 0;
        } else {
            keep = (int)((b < n_blocks_full) ? ngood : flush_keep);
            dstg = out + b * ngood;
            src = in + nb * ngood + ca;
            // (one predicated form for whole and ragged blocks: splitting it into a CTA-uniform fast path with
            // unpredicated loads measured 5 % SLOWER, 133 vs 140 Gsamples/s -- the phase waits on memory, not on issue)
            whole = more && n_in - nb * ngood >= (size_t)N;
            avail = more ? (whole ? N : (int)(n_in - nb * ngood)) : 0;
        }
        float2 ua[16], ub[16], nxa[16], nxb[16];
        p1_unload(ua, ub);
        p1_emit(ua, dstg + ca, ca, keep);
        asm volatile("" ::: "memory");
#pragma unroll
        for (int r = 0; r < 16; ++r) nxa[r] = (whole || ca + 1024 * r < avail) ? ldg_nc_f2(src + 1024 * r) : make_float2(0.f, 0.f);
        p1_emit(ub, dstg + ca + 32, ca + 32, keep);
        asm volatile("" ::: "memory");
#pragma unroll
        for (int r = 0; r < 16; ++r)
            nxb[r] = (whole || ca + 32 + 1024 * r < avail) ? ldg_nc_f2(src + 1024 * r + 32) : make_float2(0.f, 0.f);
        if (fuse) p1_forward(nxa, nxb);
        c = nc;
        bc = nbc;
        loaded = fuse;
    }
}

// H (natural order, already scaled by 1/nfft) -> Hq[k1][i][lane][c] = H[k1 + 16 (lane + 32 (2 i + c))]: what warp k1's
// lane holds in registers 2 i, 2 i + 1 after the forward transform, as one 16-byte word; a warp's load is 512 contiguous bytes
void lrc_fastfir16k_permute_H(const float2 *H, float2 *Hq)
{
    for (int k1 = 0; k1 < 16; ++k1)
        for (int i = 0; i < 16; ++i)
            for (int lane = 0; lane < 32; ++lane)
                for (int c = 0; c < 2; ++c)
                    Hq[((k1 * 16 + i) * 32 + lane) * 2 + c] = H[k1 + 16 * (lane + 32 * (2 * i + c))];
}

int lrc_fastfir16k_prepare(void)
{
    LRC_CUDA(cudaFuncSetAttribute(fastfir16k_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff16k::SMEM_BYTES));
    LRC_CUDA(cudaFuncSetAttribute(fastfir16k_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff16k::SMEM_BYTES));
    return LRC_OK;
}

// nblk: the work items (blocks of the one batch channel, or channels x blocks per channel of a stream push)
int lrc_fastfir16k_launch(int n_sm, const float2 *in, size_t n_in, float2 *out, size_t full, size_t nblk, size_t ngood,
                          size_t keep, const float2 *d_tw16k, const float2 *d_tw1k, const float2 *d_Hq,
                          const FfStreamArgs *sa, cudaStream_t s)
{
    size_t blocks = (size_t)n_sm;                    // one CTA per SM (216.5 KB of shared memory)
    if (blocks > nblk) blocks = nblk;
    FfStreamArgs a{};
    if (sa) {
        a = *sa;
        a.step_c = blocks / a.nblk;
        a.step_b = blocks % a.nblk;
    }
    auto kern = sa ? fastfir16k_kernel<true> : fastfir16k_kernel<false>;
    kern<<<(unsigned)blocks, ff16k::NT, ff16k::SMEM_BYTES, s>>>(in, n_in, out, full, nblk, ngood, keep, d_tw16k, d_tw1k,
                                                             reinterpret_cast<const float4 *>(d_Hq), a);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}
