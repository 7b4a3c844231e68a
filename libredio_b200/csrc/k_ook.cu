// k_ook.cu -- 433 MHz OOK packet decode, bit-exact with the reference chain of src/ratpak.rs:60-111:
//
//   rtlsdr::data_to_samples (rtlsdr.rs:160)  -> |x| = hypot (ratpak.rs:64-68)
//   -> bitfount::trigger (bitfount.rs:36-85)  -> bitfount::discretize (:87-96)
//   -> kpn::rle (kpn.rs:17-29) -> kpn::dle (:32-38) -> pulse-pair matchers (ratpak.rs:88-97)
//   -> kpn::shaper_optional 36 / 24 (kpn.rs:266-275)
//
// The reference runs this as eight threads exchanging one message per SAMPLE.  Here it is a handful of kernels
// over all streams at once; every float operation that feeds a comparison is the same IEEE operation in
// the same order as the reference (explicit __f*_rn / __d*_rn intrinsics, never contracted):
//
//   K-A  ook_block_tma_kernel: per 512-sample block, envelope of every sample, the strictly sequential f32
//                              block sum `s` (bitfount.rs:48) and the block max (order-free, exact)
//   K-B  ook_trigger_kernel  : the trigger state machine (:46-81) per stream: a walker warp runs the dependent chain
//                              (threshold, counter) and leaves collect / send bit masks, a keeper warp steps from send
//                              to send (burst index, buffer length, OOM guard), helper warps stage the sums and expand
//                              the masks into per-block tags (the burst a block is collected into, -1 = none)
//   K-B2 ook_burst_kernel    : per sent burst its maximum (fold of the tagged blocks' maxima), max/2 (discretize
//                              :90-91) and that threshold as a rank among the distinct envelope values
//   K-C  ook_slice_kernel + ook_scan_kernel + ook_scatter_kernel: the slicer + rle.  Every (stream, 32 blocks) is sliced
//                              independently against the burst's rank threshold into stored bit masks, a per-stream scan over
//                              per-block summaries places every block in the bit stream and the transition list, every block
//                              writes the positions where the continuous bit stream changes value in place (rle: runs span
//                              burst boundaries, the last run is never flushed).  A collected block whose maximum does not
//                              exceed the burst's max/2 is not read (512 zeros)
//   K-D  ook_match_kernel    : per stream: run lengths -> seconds (dle, IEEE f32 division) -> matcher A and B ->
//                              shaper_optional -> packed packets
//
// Two plans run these kernels.  lrc_ook decodes finite captures, every stream from the reference's initial state.
// lrc_ook_stream decodes endless streams pushed a few blocks at a time: K-B, K-B2, K-C and K-D take a per-stream
// OokSeam (null for lrc_ook) with what the reference's blocks hold between two messages, and ook_carry_kernel keeps the
// blocks of the burst still open at the end of a push, which the slicer reads in place, in front of the push's blocks, when
// that burst is sent.  The packets after any push are those of the reference on everything pushed so far.
//
// Measured and rejected (round 2, one B200 at its 1 kW power cap; whole chain, tools/bench_kernels.py --only ook; every form
// produced the same bits):
//   - K-A as the round-1 ook_block_kernel: a triangular envelope table (32896 sorted pairs, rows padded) and cp.async slabs,
//     13.6 issued instructions per sample, 5.5 of them table index work and ~4 slab bookkeeping
//     (profiles/r1_s3_ookA3_ncu_keys.txt): 0.893 ms against 0.825 for the TMA kernel with the folded table (tools/runs/r2n.sh);
//   - K-A with the table skew k2 + (k2 >> 5) as mad.hi by 2^27 + 1, to move it from the ALU pipe (LEA.HI) to the FMA pipe:
//     IMAD.HI adds into a 64-bit register pair whose low half has to be zeroed for every use, one more instruction per sample
//     in a kernel bound by issue slots (81 % busy): 0.913 ms, and 1.001 ms with 8 warps x 4 stages (tools/runs/r2n.sh);
//   - K-C as ook_rle_kernel, one warp per stream walking its collected blocks in order: with quiet blocks skipped the split
//     form won at every size, whole chain in ms, one warp / split: 4096 streams 0.596 / 0.571, 3072 0.493 / 0.452,
//     2048 0.391 / 0.335, 1024 0.292 / 0.220, 512 (one GPU's share of 4096 over eight) 0.253 / 0.163
//     (profiles/r2_bb_ook_forms.txt).
#include "common.cuh"
#include "unpack.cuh"
#include <cuda.h>
#include <algorithm>
#include <vector>

static const int OOK_BLOCK = 512;            // bitfount.rs:38
static const int OOK_TRIGGER_DURATION = 50;  // bitfount.rs:40

// |i2f(b0) + j i2f(b1)| = (float)sqrt((double)re*re + (double)im*im)  -- SURVEY 8c definition of
// num::Complex::norm (hypot).  Both products are exact in f64, so this is one rounded add, one
// correctly rounded sqrt and one narrowing, exactly as oracle/restated.c orc_norm.
__device__ __forceinline__ float lr_envelope(uint32_t b0, uint32_t b1)
{
    const double re = (double)lr_i2f(b0), im = (double)lr_i2f(b1);
    const double s = __dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im));
    return __double2float_rn(__dsqrt_rn(s));
}

// The envelope depends on the two bytes only and is symmetric in them (the f64 add commutes), so the block-sum
// kernel reads it from a table of the 32896 sorted pairs {lo <= hi} (the folded table below, 135.7 KB) held in shared
// memory.  The table is filled ON THE DEVICE by lr_envelope above when the plan is created; the u8 domain being
// finite, table == formula for all 65536 pairs is a proof of equivalence, checked exhaustively by
// tests/test_gpu_ook_fastfir.py::test_envelope_exhaustive_65536_pairs_bit_exact (formula vs CPU) and by the
// bit-exact block sums of every OOK test (table vs CPU).
// The lookup is most of the block-sum kernel's instructions, and byte extraction, max/min, index and address arithmetic run on
// the ALU pipe at half the FMA pipe's rate, so the folded table is laid out for a lookup with no byte extraction and no
// per-byte max/min:
//   * a 32-bit word holds two samples {b0, b1} {b2, b3}; ONE PRMT swaps the bytes of both halfwords and ONE
//     VIMNMX.U16x2 (__vmaxu2) takes the per-halfword maximum  max(b0 | b1 << 8, b1 | b0 << 8) = hi << 8 | lo,
//     the sorted pair as a 16-bit key -- two ALU instructions for two samples;
//   * the triangle {lo <= hi} is folded into the 129 x 256 rectangle of rows 127..255: rows hi >= 128 stay where they
//     are (columns 0..hi), a row hi <= 127 goes to row 254 - hi, columns 255 - lo (the free columns hi' + 1 .. 255 of
//     that row): key2 = max(key, 65279 - key), one integer multiply-add (FMA pipe) and one signed max;
//   * rows are skewed 8 banks apart: index = key2 + (key2 >> 5) = 264 row + col + col / 32 (one LEA.HI), injective
//     because col + col / 32 <= 262 < 264.  (With a pitch of 256 every row starts in the same bank, and the pairs of a
//     noise floor -- a few codes around 127 / 127, in neighbouring rows -- pile a warp's 32 lookups onto a handful of banks.)
// 3.5 ALU-pipe instructions per sample (5.5 for the round-1 triangular table, see the rejected forms above).
constexpr uint32_t OOK_FOLD_C = 65279u;                                  // 254 * 256 + 255
__host__ __device__ __forceinline__ uint32_t ook_fold_index(uint32_t key)   // key = hi << 8 | lo, lo <= hi
{
    const int alt = (int)OOK_FOLD_C - (int)key;                          // negative for hi = 255: loses the signed max
    const uint32_t k2 = (uint32_t)(alt > (int)key ? alt : (int)key);
    return k2 + (k2 >> 5);
}
constexpr uint32_t OOK_FOLD_MIN = 32640u + (32640u >> 5);                // smallest index in use (key2 >= 32640)
constexpr uint32_t OOK_FOLD_MAX = 65535u + (65535u >> 5);
constexpr int OOK_FLUT_N = (int)((OOK_FOLD_MAX - OOK_FOLD_MIN + 1 + 3) / 4 * 4);   // 33924 floats
constexpr int OOK_FLUT_BYTES = OOK_FLUT_N * 4;

__global__ void ook_build_flut_kernel(float *__restrict__ flut)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 65536u) return;
    const uint32_t hi = i >> 8, lo = i & 0xffu;
    if (lo <= hi) flut[ook_fold_index(i) - OOK_FOLD_MIN] = lr_envelope(hi, lo);
}

struct lrc_ook {
    lrc_ctx *ctx;
    size_t   n_streams, n_blocks, max_runs, max_packets, max_bursts;
    unsigned sample_rate;
    uint32_t guard_samples;           // bitfount.rs:52 1000 * trigger_duration * block_size (LRC_OOK_TEST_GUARD_BLOCKS: a test hook)
    DevBuf<float>    d_sum, d_max;    // [n_streams][n_blocks]
    DevBuf<int32_t>  d_tag;           // [n_streams][n_blocks] burst index the block is collected into, -1 = none
    DevBuf<float>    d_half;          // [n_streams][max_bursts]  max/2 of the burst
    DevBuf<uint8_t>  d_bflags;        // [n_streams][max_bursts]  bit0 = emitted, bit1 = leading 0.0 sample
    DevBuf<uint32_t> d_bend;          // [n_streams][max_bursts]  last block that can belong to the burst (the one that sent / dropped it)
    DevBuf<uint32_t> d_nbursts;       // [n_streams]
    DevBuf<uint32_t> d_trans;         // [n_streams][max_runs] positions where the bit stream changes value
    DevBuf<uint32_t> d_ntrans;        // [n_streams]  (may exceed max_runs: overflow is detected on fetch)
    DevBuf<uint32_t> d_nbits;         // [n_streams]  length of the flattened bit stream
    DevBuf<unsigned long long> d_packets;   // [n_streams][2][max_packets] packets packed MSB-first
    DevBuf<uint32_t> d_npackets;      // [n_streams][2]
    DevBuf<uint32_t> d_runs_dbg;      // [n_streams][max_runs] (value << 31 | length), filled by K-D
    DevBuf<float>    d_flut;          // folded envelope table, OOK_FLUT_N floats (the block-sum kernel's)
    void     *encode_tiled;           // cuTensorMapEncodeTiled (driver entry point, fetched once)
    DevBuf<uint16_t> d_mask;          // [n_streams][n_blocks][32] slicer output of collected blocks, 512 bits each (K-C)
    DevBuf<uint32_t> d_hrank;         // [n_streams][max_bursts] rank threshold of a sent burst (K-C)
    DevBuf<uint32_t> d_next;          // [1] next (stream, group) the slice kernel hands out
    DevBuf<uint32_t> d_bsum;          // [n_streams][n_blocks] {inner transitions, first bit, last bit} of a collected block
    DevBuf<uint4>    d_binfo;         // [n_streams][n_blocks] place of a collected block in the bit stream and the transition list
    DevBuf<uint16_t> d_rank;          // [65536] rank of the pair's envelope among the distinct envelope values
    DevBuf<float>    d_uniq;          // [n_uniq] the distinct envelope values, ascending
    uint32_t  n_uniq;
    size_t    cpitch;                 // carry slots per stream in front of the blocks of d_mask / d_bsum / d_binfo (0: batch plan)
};

// ---- streaming (lrc_ook_stream) -------------------------------------------------------------------------------------------
// Everything one stream holds between two pushes: the state of the reference's blocks as they stand between two messages.  The
// kernels take a pointer to an array of these that is null on the batch path (initial state, nothing carried).
struct OokSeam {
    // K-B walker (bitfount.rs:41-44, :46-70): threshold, counter (clamped at -1: every counter below 0 walks the same way), and the
    // two look-ahead predicates of the walk; keeper (:43, :52-54, :73-81): buffer length in samples, buffer starts with the 0.0
    float    threshold;
    int32_t  trig;
    uint32_t buf_len;
    uint8_t  fired, low2, lead0, pad0;
    // the open burst: collected blocks held in the carry region, and their running maximum (discretize :90 is order-free)
    uint32_t n_carry;
    float    run_max;
    // K-C2: value of the last bit emitted, whether any bit was
    uint32_t prev, any;
    // K-D: the open run of rle (kpn.rs:17-29), the matchers' state (ratpak.rs:88-97, kpn.rs:266-275) per protocol
    unsigned long long run_len;
    uint32_t run_val;
    uint32_t m_pending[2], m_n[2], m_count[2];
    float    m_d[2];
    unsigned long long m_acc[2];
    uint32_t err;                     // OOK_ERR_* bits, sticky until reset
};
constexpr uint32_t OOK_ERR_CARRY = 1u, OOK_ERR_RUNS = 2u, OOK_ERR_BURSTS = 4u;
constexpr int32_t OOK_TAG_OPEN = -2;  // stream plans: a block collected into the burst still open at the end of the push

static OokSeam ook_seam_initial()
{
    OokSeam z;
    memset(&z, 0, sizeof(z));
    z.buf_len = 1; z.low2 = 1; z.lead0 = 1;   // sample_buffer = vec!(0.0) (:43); 0 - 1 < 0 on the first block
    return z;
}

// the carry region [stream][cpitch] in front of a push's blocks [stream][n_blocks] form one virtual row per stream, read in place
struct OokCarry {
    size_t          cpitch;           // slots per stream (a multiple of 32: a group of 32 is all carry or all push)
    const uint8_t  *bytes;            // [stream][cpitch][1024]
    const float    *bmax;             // [stream][cpitch] block maxima
    const uint32_t *live;             // [stream] carried blocks that belong to a burst sent in this push (0 otherwise)
};

// ---------------------------------------------------------------------------------------------
// K-A: envelope, sequential block sum, block max.  One warp handles 32 consecutive blocks of one
// stream and lane b owns block b: its 512 envelopes must be added one after the other (bitfount.rs:48),
// so the lane walks its own 1024 bytes, through the folded table above.  The bytes reach it through shared
// memory, staged by the TMA engine: the capture is described to it as a 3-D byte tensor
// [stream][block][1024 B]; ONE cp.async.bulk.tensor per slab (issued by lane 0) brings the box
// {64 B, 32 blocks, 1 stream} into a 2 KB stage with the 64-byte hardware swizzle, i.e. 16-byte chunk c of
// row r lands at chunk c ^ ((r >> 1) & 3).  Lane r then reads its row with four LDS.128 and the eight lanes of
// a quarter-warp phase hit eight distinct bank groups (4 r + (c ^ f(r)) mod 8 takes all values 0..7) -- the
// transposition costs no padding, no per-lane address arithmetic and no LDGSTS instructions.  Blocks past the
// end of the capture are zero-filled by the TMA (out-of-bounds rows of the box).  No envelope is ever written
// back to shared memory.
// Every warp runs its own ring of KA2_STAGES stages with one mbarrier per stage and treats all its (group, slab)
// pairs as one flat sequence, so the prefetch runs across group boundaries.
// ---------------------------------------------------------------------------------------------
constexpr int KA2_SLAB_BYTES = 64;
constexpr int KA2_STAGE_BYTES = 32 * KA2_SLAB_BYTES;
constexpr int KA2_SLABS = OOK_BLOCK * 2 / KA2_SLAB_BYTES;     // 16 slabs per block row
constexpr int KA2_WARPS = 16, KA2_STAGES = 2;
constexpr int KA2_STG_OFF = (OOK_FLUT_BYTES + 1023) / 1024 * 1024;
constexpr int KA2_BAR_OFF = KA2_STG_OFF + KA2_WARPS * KA2_STAGES * KA2_STAGE_BYTES;
constexpr int KA2_SMEM_BYTES = KA2_BAR_OFF + KA2_WARPS * KA2_STAGES * 8 + 1024;     // + slack to align the base to 1024
static_assert(KA2_SMEM_BYTES <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ void tma_load_box3(uint32_t dst_s, const CUtensorMap *tm, int c0, int c1, int c2, uint32_t bar_s)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"(dst_s), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar_s) : "memory");
}

// envelope of one sorted 16-bit key through the folded table; flut_adj = shared address of the table minus
// 4 OOK_FOLD_MIN.  The negation runs on the FMA pipe (IMAD.MOV), the fused add-max (VIADDMNMX), the skew (LEA.HI) and
// the address LEA on the ALU pipe.
__device__ __forceinline__ float flut_envelope(uint32_t flut_adj, uint32_t key)
{
    int alt;
    asm("mad.lo.s32 %0, %1, -1, 65279;" : "=r"(alt) : "r"((int)key));
    const uint32_t k2 = (uint32_t)max(alt, (int)key);
    const uint32_t idx = k2 + (k2 >> 5);
    float e;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(e) : "r"(flut_adj + 4u * idx));
    return e;
}

__global__ void __launch_bounds__(KA2_WARPS * 32, 1)
ook_block_tma_kernel(const __grid_constant__ CUtensorMap tmap, size_t n_streams, size_t n_blocks,
                     const float *__restrict__ g_flut, float *__restrict__ d_sum, float *__restrict__ d_max)
{
    extern __shared__ __align__(1024) uint8_t ka2_smem[];
    // the 64-byte swizzle pattern is a function of the shared ADDRESS: stages must sit on 512-byte boundaries
    const uint32_t base_s = (smem_u32(ka2_smem) + 1023u) & ~1023u;
    uint8_t *base = ka2_smem + (base_s - smem_u32(ka2_smem));
    float *flut = reinterpret_cast<float *>(base);
    for (int i = threadIdx.x; i < OOK_FLUT_N / 4; i += blockDim.x)
        reinterpret_cast<float4 *>(flut)[i] = __ldg(reinterpret_cast<const float4 *>(g_flut) + i);
    // warp index through a shuffle: the compiler then knows it (and every stage, barrier and box coordinate derived
    // from it) is warp-uniform and keeps the TMA operands in uniform registers
    const int lane = threadIdx.x & 31, warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const uint32_t stg_s = base_s + KA2_STG_OFF + warp * (KA2_STAGES * KA2_STAGE_BYTES);
    const uint32_t bar_s = base_s + KA2_BAR_OFF + warp * (KA2_STAGES * 8);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < KA2_STAGES; ++s)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar_s + 8 * s), "r"(1));
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t flut_adj = base_s - 4u * OOK_FOLD_MIN;
    const size_t groups_per_stream = (n_blocks + 31) / 32;
    const size_t n_groups = groups_per_stream * n_streams;
    const size_t warps_total = (size_t)gridDim.x * KA2_WARPS;
    size_t grp = (size_t)blockIdx.x * KA2_WARPS + warp;
    if (grp >= n_groups) return;
    // lane's read offsets inside a stage: row = lane, chunk q at (q ^ ((lane >> 1) & 3))
    const uint32_t row_s = stg_s + lane * KA2_SLAB_BYTES;
    const uint32_t f16 = ((uint32_t)(lane >> 1) & 3u) << 4;
    // stage = slab % KA2_STAGES and parity = (slab / KA2_STAGES) & 1 come from the slab counter alone: a group has 16 slabs, a
    // multiple of 2 KA2_STAGES, so every group starts with all barriers back in phase 0
    static_assert(KA2_SLABS % (2 * KA2_STAGES) == 0, "phase bookkeeping");
    auto issue = [&](int st, int b0, int slab) {                 // lane 0
        const uint32_t bar = bar_s + 8 * (slab % KA2_STAGES);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(KA2_STAGE_BYTES) : "memory");
        tma_load_box3(stg_s + (slab % KA2_STAGES) * KA2_STAGE_BYTES, &tmap, slab * KA2_SLAB_BYTES, b0, st, bar);
    };
    int st = (int)(grp / groups_per_stream), b0 = (int)(grp % groups_per_stream) * 32;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < KA2_STAGES - 1; ++k) issue(st, b0, k);
    }
    while (true) {
        const size_t grp_n = grp + warps_total;
        const bool has_n = grp_n < n_groups;
        const int st_n = (int)(grp_n / groups_per_stream), b0_n = (int)(grp_n % groups_per_stream) * 32;
        float s = 0.0f, mx = 0.0f;
#pragma unroll 1
        for (int so = 0; so < KA2_SLABS; so += KA2_STAGES) {
            const uint32_t parity = (uint32_t)(so / KA2_STAGES) & 1u;
#pragma unroll
            for (int h = 0; h < KA2_STAGES; ++h) {
                const int slab = so + h;
                // the stage this issue overwrites was read one slab ago (closed by its __syncwarp)
                {
                    const int nx = slab + KA2_STAGES - 1;
                    const bool wrap = nx >= KA2_SLABS;           // the prefetch runs into the warp's next group
                    if (lane == 0 && (!wrap || has_n)) issue(wrap ? st_n : st, wrap ? b0_n : b0, wrap ? nx - KA2_SLABS : nx);
                }
                asm volatile(
                    "{\n"
                    ".reg .pred p;\n"
                    "WAITA_%=:\n"
                    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                    "@p bra DONEA_%=;\n"
                    "bra WAITA_%=;\n"
                    "DONEA_%=:\n"
                    "}\n" :: "r"(bar_s + 8 * h), "r"(parity) : "memory");
                const uint32_t rs = row_s + h * KA2_STAGE_BYTES;
#pragma unroll
                for (int q = 0; q < KA2_SLAB_BYTES / 16; ++q) {
                    uint4 v;
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(rs + (((uint32_t)q << 4) ^ f16)));
                    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        // both samples of the word at once: per halfword max(b0 | b1 << 8, b1 | b0 << 8) = hi << 8 | lo
                        const uint32_t K = __vmaxu2(w[k], __byte_perm(w[k], 0, 0x2301));
                        const float e0 = flut_envelope(flut_adj, K & 0xffffu);
                        const float e1 = flut_envelope(flut_adj, __umulhi(K, 65536u));    // K >> 16 on the FMA pipe
                        s = __fadd_rn(s, e0);                    // samples.iter().sum(): left to right from 0.0
                        s = __fadd_rn(s, e1);
                        mx = fmaxf(mx, fmaxf(e0, e1));
                    }
                }
                __syncwarp();                                    // every lane is done with the stage
            }
        }
        if ((size_t)b0 + lane < n_blocks) {
            d_sum[(size_t)st * n_blocks + b0 + lane] = s;
            d_max[(size_t)st * n_blocks + b0 + lane] = mx;
        }
        if (!has_n) break;
        grp = grp_n; st = st_n; b0 = b0_n;
    }
}

// ---------------------------------------------------------------------------------------------
// K-B: trigger state machine (bitfount.rs:41-81, statement by statement), 32 streams per CTA
//
// The walk along a stream is one dependent chain (threshold -> compare -> counter -> threshold ...): its length in
// cycles IS the kernel's duration, whatever the number of streams.  Round 1 had every thread stage its tile, divide its
// sums by 1000, walk, and write its tags back: ~2500 dependent-issue slots per 32-block tile on a warp that has an SM
// sub-partition to itself (133 us for 500 blocks, 490 cycles per block).  Now a CTA is 14 warps in three roles, a
// tile of 32 blocks apart from each other and one __syncthreads per tile:
//   helpers (12 warps), iteration i: wait for the cp.async copies of the sums of tile i+1 (issued two iterations ago),
//                          q = s / 1000 (:63) for tile i+1, tags of tile i-2 out to global memory (expanded from the
//                          masks, coalesced), cp.async of tile i+3
//   walker,  iteration i : tile i from shared memory, eight blocks ahead into registers, the chain's statements as
//                          selects (32 streams are in 32 different states: as branches every `if` would run both
//                          sides one after the other); leaves the masks {counter > 1}, {counter == 0} of the tile
//   keeper,  iteration i : tile i-1: burst index, buffer length and flags from the masks, send by send
// A burst that is dropped (the OOM guard :52-54, or still open when the capture ends) keeps bit 0 of its flag clear and
// has its blocks un-tagged once all tags are in global memory.
// ---------------------------------------------------------------------------------------------
constexpr int KB_STREAMS = 32;                // streams per CTA = lanes of the walker warp (and of the keeper warp)
constexpr int KB_HELPERS = 384;               // helper threads (twelve warps: with three, then six, they -- not the chain -- set the pace)
constexpr int KB_THREADS = 2 * KB_STREAMS + KB_HELPERS;
constexpr int KB_TILE = 32;                   // blocks per staged tile
constexpr int KB_LD = KB_TILE + 1;            // conflict-free both ways: helpers move rows, the walker reads columns

// STREAM (stream plans): the walker and the keeper start from the stream's OokSeam and store it back after the last block, and the
// burst still open at the end is tagged OOK_TAG_OPEN (for ook_carry_kernel) instead of un-tagged.
template <bool STREAM>
__global__ void __launch_bounds__(KB_THREADS)
ook_trigger_kernel(const float *__restrict__ d_sum, size_t n_streams, size_t n_blocks, size_t max_bursts, uint32_t guard_samples,
                   int32_t *__restrict__ d_tag, uint32_t *__restrict__ d_bend, uint8_t *__restrict__ d_bflags,
                   uint32_t *__restrict__ d_nbursts, OokSeam *__restrict__ seam)
{
    __shared__ float s_sum[4][KB_STREAMS * KB_LD];        // tile t in buffer t & 3: copies run two tiles ahead of the divisions
    __shared__ float s_q[2][KB_STREAMS * KB_LD];
    __shared__ int32_t s_tag[2][KB_STREAMS * KB_LD];      // explicit tags of a tile the keeper walked block by block
    __shared__ uint32_t s_cm[4][KB_STREAMS], s_sm[4][KB_STREAMS];   // per tile and stream: blocks collected / blocks that send
    __shared__ uint32_t s_b0[2][KB_STREAMS];              // burst index of the stream when the tile starts
    __shared__ uint32_t s_mode[2];                        // 1 = the tile's tags are in s_tag
    const int tid = threadIdx.x, lane = tid & 31;
    const size_t st0 = (size_t)blockIdx.x * KB_STREAMS;
    const int n_tiles = (int)((n_blocks + KB_TILE - 1) / KB_TILE);
    // Round-2 split of the walk.  The reference's statements fall into a CHAIN -- threshold and trigger counter (:46, :57-70), each
    // block's values needing the previous block's -- and BOOK-KEEPING that only reads the counter (:52-54 guard, :73-81 collect and
    // send).  The walker warp (threads 0-31) runs the chain alone and leaves two bit masks per tile of 32 blocks: counter > 1
    // (collect) and counter == 0 (send).  The keeper warp (threads 32-63, same lane = same stream), one tile behind, does not walk
    // blocks at all: it steps from SEND to SEND (a handful per stream and capture), counting the collected blocks in between with
    // popc for the buffer length; the tags are expanded from the masks by the helper warps (tag = burst index at the start of the
    // tile + sends before the block), and a burst's maximum is taken afterwards, in parallel, by ook_burst_kernel from the per-block
    // maxima and the tags.  Only a tile in which the OOM guard could fire (buffer within 32 blocks of the limit: 100 s of
    // uninterrupted burst) is walked block by block, with the tags written out explicitly.
    // Measured on the way here (4096 streams x 500 blocks): one warp doing everything 133 us; walker + helpers 60 us; walker +
    // per-block keeper 53 us with the KEEPER the bound (40 instructions per block against the chain's 21, ncu source page:
    // profiles/r2_ae_ookB_ncu_keys.txt).
    const bool walker = tid < KB_STREAMS;
    const bool keeper = tid >= KB_STREAMS && tid < 2 * KB_STREAMS;
    const bool helper = tid >= 2 * KB_STREAMS;
    const int ht = tid - 2 * KB_STREAMS, hwarp = ht >> 5;              // helpers: warp w moves rows w, w + 12, ...
    const uint32_t mb = (uint32_t)(max_bursts < 0x7fffffffull ? max_bursts : 0x7fffffffull);
    // cp.async (LDGSTS) of tile `tile` into its buffer: a helper warp moves 32 consecutive floats of one stream per step
    auto stage = [&](int tile) {
        if (tile < n_tiles) {
            const size_t b = (size_t)tile * KB_TILE + lane;
            for (int r = hwarp; r < KB_STREAMS; r += KB_HELPERS / 32) {
                const size_t s = st0 + r;
                float *ds = &s_sum[tile & 3][r * KB_LD + lane];
                if (s < n_streams && b < n_blocks)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(smem_u32(ds)), "l"(d_sum + s * n_blocks + b) : "memory");
                else
                    *ds = 0.0f;
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // s / 1000 (:63) of tile `tile`, whose copies have landed: 1024 independent IEEE divisions over 96 threads
    auto quotients = [&](int tile) {
        if (tile >= n_tiles) return;
        const float *src = s_sum[tile & 3];
        float *dst = s_q[tile & 1];
        for (int i = ht; i < KB_STREAMS * KB_TILE; i += KB_HELPERS) {
            const int r = i >> 5, c = i & 31;
            dst[r * KB_LD + c] = __fdiv_rn(src[r * KB_LD + c], 1000.0f);
        }
    };
    // tags of tile `tile` to global memory: lane = block, a helper warp takes a stream per step
    auto tags_out = [&](int tile) {
        if (tile < 0 || tile >= n_tiles) return;
        const bool expl = s_mode[tile & 1] != 0u;
        const int32_t *src = s_tag[tile & 1];
        const size_t b = (size_t)tile * KB_TILE + lane;
        for (int r = hwarp; r < KB_STREAMS; r += KB_HELPERS / 32) {
            const size_t s = st0 + r;
            if (s < n_streams && b < n_blocks) {
                int32_t tg;
                if (expl) {
                    tg = src[r * KB_LD + lane];
                } else {
                    const uint32_t cm = s_cm[tile & 3][r], sm = s_sm[tile & 3][r];
                    const uint32_t bi = s_b0[tile & 1][r] + (uint32_t)__popc(sm & ((1u << lane) - 1u));
                    tg = ((cm >> lane) & 1u) && bi < mb ? (int32_t)bi : -1;
                }
                d_tag[s * n_blocks + b] = tg;
            }
        }
    };
    // one stream per lane, in the walker and in the keeper
    const size_t st = st0 + lane;
    const bool live = (walker || keeper) && st < n_streams;
    uint32_t *bend = d_bend + st * max_bursts;
    uint8_t *flags = d_bflags + st * max_bursts;
    // walker state
    int trigger = 0;                          // :41 (isize there; |trigger| <= n_blocks here)
    float threshold = 0.0f;                   // :44
    bool fired = false, low2 = true;          // the block before did not fire, the counter two blocks back was below 2: 0 - 1 < 0
    // keeper state
    uint32_t buf_len = 1;                     // :43 sample_buffer = vec!(0.0); capped at the guard + 512 below
    bool lead0 = true;                        // the buffer currently starts with that 0.0
    uint32_t burst = 0;                       // index of the burst being collected
    bool dropped = false;                     // the OOM guard abandoned a burst of this stream
    // the walker's state after the last block of the push (the walk goes on over the padding of a ragged last tile)
    int sv_trigger = 0; float sv_threshold = 0.0f; bool sv_fired = false, sv_low2 = true;
    if (STREAM && live) {
        const OokSeam &z = seam[st];
        trigger = z.trig; threshold = z.threshold; fired = z.fired != 0; low2 = z.low2 != 0;
        buf_len = z.buf_len; lead0 = z.lead0 != 0;
    }
    if (helper) {
        stage(0);
        stage(1);
        stage(2);
        asm volatile("cp.async.wait_group 2;" ::: "memory");            // tile 0 has landed (this thread's part)
        named_bar_sync(1, KB_HELPERS);
        quotients(0);
    }
    __syncthreads();
    // iteration i: helpers tile i + 1 / i + 2 in, tags of tile i - 2 out; walker tile i; keeper tile i - 1
    for (int tile = 0; tile <= n_tiles + 1; ++tile) {
        if (helper) {
            asm volatile("cp.async.wait_group 1;" ::: "memory");        // tile + 1 (issued two iterations ago; tile + 2 may be in flight)
            named_bar_sync(1, KB_HELPERS);                              // ... every helper's part of it
            quotients(tile + 1);
            tags_out(tile - 2);
            stage(tile + 3);                                            // its buffer was last read in iteration tile - 1
        } else if (walker) {
            if (tile < n_tiles) {
                const float *t_sum = s_sum[tile & 3] + lane * KB_LD;
                const float *t_q = s_q[tile & 1] + lane * KB_LD;
                const size_t b0 = (size_t)tile * KB_TILE;
                const int nb = (int)((n_blocks - b0) < (size_t)KB_TILE ? (n_blocks - b0) : (size_t)KB_TILE);
                uint32_t cm = 0u, sm = 0u;
#pragma unroll 1
                for (int u0 = 0; u0 < KB_TILE; u0 += 8) {
                    // the block's inputs do not depend on the chain: eight blocks ahead into registers
                    float sr[8], qr[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) { sr[k] = t_sum[u0 + k]; qr[k] = t_q[u0 + k]; }
                    uint32_t c8 = 0u, s8 = 0u;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        // (blocks past the end of a ragged last tile are walked too, on zero sums: their bits are masked off
                        // below and the walker's state is not used after the last tile)
                        // `trigger < 0` after the decrement (:46, :62) is taken from PREDICATES instead of the counter: the counter
                        // of the block before was `fired ? 50 : c - 1` (c: the counter two blocks back), so it is below 1 iff that
                        // block did not fire and c < 2 -- the latter known a block early.  The threshold's critical path is then
                        // compare -> predicate -> predicated add, not compare -> select -> compare -> predicated add.
                        const bool upd = !fired && low2;
                        low2 = trigger < 2;
                        trigger -= 1;                                                       // :46
                        const float s = sr[k];                                              // :48
                        // the chain is kept short: the `threshold == 0` case (:57-59) is evaluated beside the add it feeds -- both
                        // candidate sums exist before the select -- and the fire test s > threshold * 4 (:68-70) is made as
                        // s / 4 > threshold with s / 4 taken off the chain: both scalings by a power of two are exact (s is 0 or
                        // >= 0.0078, the smallest non-zero envelope), so the comparison is the same one
                        // both outcomes of `threshold == 0` (:57-59) are carried through the update (:62-65) and selected at the end: the
                        // one that starts from s never touches the chain, the other is three dependent operations from the old threshold
                        const bool unset = threshold == 0.0f;                               // :57-59
                        const float a1 = __fadd_rn(s, qr[k]);                               // :62-65 from threshold = s
                        const float a2 = __fsub_rn(a1, __fmul_rn(a1, 0.002f));
                        const float b1 = __fadd_rn(threshold, qr[k]);                       // :62-65 from the old threshold
                        const float b2 = __fsub_rn(b1, __fmul_rn(b1, 0.002f));
                        const float thr0 = unset ? s : threshold;
                        const float thr2 = unset ? a2 : b2;
                        threshold = upd ? thr2 : thr0;                                      // upd == (trigger < 0)
                        fired = __fmul_rn(s, 0.25f) > threshold;                            // :68-70
                        trigger = fired ? OOK_TRIGGER_DURATION : trigger;
                        // what the book-keeping needs of the counter: collect (:73) and send (:78)
                        c8 |= (trigger > 1 ? 1u : 0u) << k;
                        s8 |= (trigger == 0 ? 1u : 0u) << k;
                        if (STREAM && u0 + k == nb - 1 && tile == n_tiles - 1) {     // off the chain: selects only
                            sv_trigger = trigger; sv_threshold = threshold; sv_fired = fired; sv_low2 = low2;
                        }
                    }
                    cm |= c8 << u0;
                    sm |= s8 << u0;
                }
                const uint32_t valid = nb >= 32 ? 0xffffffffu : ((1u << nb) - 1u);
                s_cm[tile & 3][lane] = cm & valid;
                s_sm[tile & 3][lane] = sm & valid;
            }
        } else if (tile >= 1 && tile <= n_tiles) {                      // keeper, one tile behind
            const int kt = tile - 1;
            const uint32_t cm = s_cm[kt & 3][lane], sm = s_sm[kt & 3][lane];
            const size_t b0 = (size_t)kt * KB_TILE;
            s_b0[kt & 1][lane] = burst;
            // could the guard fire in this tile?  It looks at the buffer before a block is pushed (:52), and the buffer grows by
            // at most 32 blocks here
            const bool near_guard = live && buf_len + (uint32_t)(KB_TILE * OOK_BLOCK) > guard_samples;
            if (!__any_sync(0xffffffffu, near_guard)) {
                if (lane == 0) s_mode[kt & 1] = 0u;
                // from send to send: the blocks collected since the last one lengthen the buffer (:73-75), the send empties it
                uint32_t rem = live ? sm : 0u, done = 0u;                // `done`: bits of the blocks already accounted for
                while (rem) {
                    const int u = __ffs(rem) - 1;
                    rem &= rem - 1u;
                    const uint32_t upto = (1u << u) - 1u;                // blocks before u (u itself sends, it is not collected)
                    buf_len += (uint32_t)OOK_BLOCK * (uint32_t)__popc(cm & upto & ~done);
                    done = upto | (1u << u);
                    if (burst < mb) {                                                   // :78-81 send, buffer = vec!()
                        bend[burst] = (uint32_t)(b0 + u);
                        flags[burst] = (uint8_t)(1u | (lead0 ? 2u : 0u));
                    }
                    burst += 1;
                    buf_len = 0; lead0 = false;
                }
                buf_len += (uint32_t)OOK_BLOCK * (uint32_t)__popc(cm & ~done);
            } else {
                if (lane == 0) s_mode[kt & 1] = 1u;
                int32_t *t_tag = s_tag[kt & 1] + lane * KB_LD;
                const int nb = (int)((n_blocks - b0) < (size_t)KB_TILE ? (n_blocks - b0) : (size_t)KB_TILE);
                for (int u = 0; u < nb; ++u) {
                    // :52-54 OOM guard (a burst longer than 50 000 blocks = 100 s at 256 ksps): what was collected is dropped -- the
                    // burst index is abandoned with its flag clear -- and collection goes on in a fresh buffer [0.0].  When the
                    // guard fires with the counter at 1 nothing is pushed after the reset and the next block sends the buffer [0.0]
                    // as it is: a sent burst (flags 3, max/2 = 0) without a tagged block, which the slicer turns into its one 0 bit.
                    if (buf_len > guard_samples) {
                        if (live && burst < mb) { flags[burst] = 0; bend[burst] = (uint32_t)(b0 + u) - 1u; }
                        burst += 1; dropped = true;
                        buf_len = 1; lead0 = true;
                    }
                    const bool collect = ((cm >> u) & 1u) != 0u;                        // :73-75 push_all
                    buf_len += collect ? (uint32_t)OOK_BLOCK : 0u;
                    t_tag[u] = (collect && burst < mb) ? (int32_t)burst : -1;
                    if ((sm >> u) & 1u) {                                               // :78-81 send, buffer = vec!()
                        if (live && burst < mb) {
                            bend[burst] = (uint32_t)(b0 + u);
                            flags[burst] = (uint8_t)(1u | (lead0 ? 2u : 0u));
                        }
                        burst += 1;
                        buf_len = 0; lead0 = false;
                    }
                }
            }
        }
        __syncthreads();
    }
    // a burst still open when the capture ends is never sent: its blocks (at most the tail of the capture) are un-tagged, and so
    // are -- in one pass over the stream's tags, which only a capture that tripped the OOM guard pays for -- the blocks of the
    // bursts the guard abandoned (flag bit 0 clear).  The slicer only ever sees blocks of bursts that were sent.  The whole CTA
    // does it, a stream at a time with coalesced accesses, and it simply looks for the index of the burst that was never sent (the
    // walk itself carries no "first block of this burst" bookkeeping: every instruction in it is latency on the chain).
    uint32_t *s_open = reinterpret_cast<uint32_t *>(s_q[0]);         // [32] 1 = live stream, [32] index of its unsent burst,
    if (keeper && live) {                                             // [32] guard fired -- s_q is free after the last tile
        if (burst < max_bursts) flags[burst] = 0;
        d_nbursts[st] = burst;                // may exceed max_bursts -> reported by fetch
        if (STREAM) {
            seam[st].buf_len = buf_len; seam[st].lead0 = lead0 ? 1 : 0;
            if (burst >= max_bursts) seam[st].err |= OOK_ERR_BURSTS;  // the open burst's blocks could not be tagged
        }
    }
    if (STREAM && walker && live) {
        seam[st].trig = sv_trigger < -1 ? -1 : sv_trigger; seam[st].threshold = sv_threshold;
        seam[st].fired = sv_fired ? 1 : 0; seam[st].low2 = sv_low2 ? 1 : 0;
    }
    __syncthreads();                          // all tags are in global memory, s_q is no longer read
    if (keeper) {
        s_open[lane] = live ? 1u : 0u;
        s_open[32 + lane] = burst;
        s_open[64 + lane] = live && dropped ? 1u : 0u;
    }
    __syncthreads();
    // The unsent burst's blocks end within the last two blocks of the capture (it is still being collected, or the counter just
    // reached 1) and lie at most one block apart.  A stream plan tags them OOK_TAG_OPEN: ook_carry_kernel appends them to the carry.  The warps share the streams out (warp w: streams w, w + 14, w + 28): the last 64
    // tags of a warp's streams are loaded first (independent loads, one latency), matched and cleared; a run longer than that
    // (rare) is followed backwards chunk by chunk.
    {
        constexpr int NW = KB_THREADS / 32, NJ = (KB_STREAMS + NW - 1) / NW;
        const int w = tid >> 5;
        int32_t t0[NJ], t1[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int r = w + NW * j;
            const size_t s = st0 + r;
            const long long k0 = (long long)n_blocks - 1 - lane, k1 = k0 - 32;
            const bool on = r < KB_STREAMS && s < n_streams && s_open[r];
            t0[j] = on && k0 >= 0 ? d_tag[s * n_blocks + k0] : -1;
            t1[j] = on && k1 >= 0 ? d_tag[s * n_blocks + k1] : -1;
        }
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int r = w + NW * j;
            const size_t s = st0 + r;
            if (r >= KB_STREAMS || s >= n_streams || !s_open[r]) continue;     // warp-uniform
            int32_t *tag = d_tag + s * n_blocks;
            const int32_t bidx = (int32_t)s_open[32 + r];
            const long long k0 = (long long)n_blocks - 1 - lane, k1 = k0 - 32;
            const bool m0 = t0[j] == bidx, m1 = t1[j] == bidx;
            const int32_t untag = STREAM ? OOK_TAG_OPEN : -1;
            if (m0) tag[k0] = untag;
            if (m1) tag[k1] = untag;
            // the burst reaches past the 64 tags: keep going while a chunk of 32 still holds one of its blocks (a burst may skip
            // single blocks -- the block at counter 1 is not collected, a re-fire on the next one continues the burst -- so a
            // chunk without any of its blocks is the end)
            long long k = k1 - 32;
            bool more = __any_sync(0xffffffffu, m1);
            while (more && __any_sync(0xffffffffu, k >= 0)) {
                const bool m = k >= 0 && tag[k] == bidx;
                if (m) tag[k] = untag;
                more = __any_sync(0xffffffffu, m);
                k -= 32;
            }
        }
    }
    // bursts the OOM guard abandoned: one pass over the stream's tags, which only a capture that tripped the guard pays for
    for (int r = 0; r < KB_STREAMS; ++r) {
        const size_t s = st0 + r;
        if (s >= n_streams) break;
        if (s_open[64 + r]) {
            __syncthreads();                  // uniform: s_open is the same for every thread
            int32_t *tag = d_tag + s * n_blocks;
            const uint8_t *fl = d_bflags + s * max_bursts;
            for (size_t k = tid; k < n_blocks; k += KB_THREADS) {
                const int32_t tg = tag[k];
                if (tg >= 0 && !(fl[tg] & 1u)) tag[k] = -1;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K-C: discretize + rle as bit masks.  A warp slices a collected block at a time, lane l owns samples
// [16 l, 16 l + 16) of it (32 contiguous bytes).  The positions (in the flattened bit stream) where the value
// changes make up the stream's transition list, in order.
//
// The slicer `x > max/2` (bitfount.rs:91) never needs the envelope VALUE here, only its order against the
// threshold: the plan holds rank[b0 | b1 << 8] = index of the pair's envelope among the 32 k distinct
// envelope values in ascending order (a 128 KB u16 table indexed by the raw byte pair -- no max/min, no
// triangular index); a burst's max/2 becomes the rank threshold #{values <= max/2} by a warp-wide 32-ary
// search of the sorted values (ook_burst_kernel); then x > max/2  <=>  rank(x) >= threshold,
// exactly, for every byte pair.  Neighbouring byte pairs (a noise floor sits within a few codes of 127/127)
// would all fall into the banks of byte0 >> 1 with a pitch of 256 entries, so a byte1 row is 264 entries long:
// 132 words = 4 banks further per row, which spreads an 8 x 8 neighbourhood over all 32 banks.  The per-sample
// work is six instructions: the raw halfword (LOP3, or IMAD.HI on the FMA pipe), its slot and address (LEA.HI,
// IADD3), the load, one subtraction and one funnel shift that moves the comparison's sign bit into the mask
// (bits arrive reversed; one BREV per 16 samples).
//
// QUIET BLOCKS.  The block-sum kernel left every block's maximum; a collected block whose maximum does not exceed the burst's
// max/2 slices to 512 zeros (x <= block max <= max/2 for each of its samples: `x > max/2` is false, bitfount.rs:91) -- without
// being read.  That is the noise the trigger keeps collecting for 49 blocks after a burst and most of the gaps between the
// pulses of a packet: the slicer's share of the capture drops from the collected half to the blocks that hold a pulse.
// ---------------------------------------------------------------------------------------------
constexpr int OOK_RANK_PITCH = 264;                           // u16 entries per byte1 row (256 used)
constexpr int OOK_RANK_N = 256 * OOK_RANK_PITCH;
constexpr int OOK_RANK_BYTES = OOK_RANK_N * 2;                // 135 168
static_assert(OOK_RANK_BYTES % 16 == 0, "table is copied as uint4");
// slot of the byte pair (b0 = I, b1 = Q): with raw = b0 | b1 << 8 -- the sample's 16 bits as they sit in the capture --
// raw + (raw >> 5) = 264 b1 + b0 + (b0 >> 5): the skewed row layout above, reached from the raw halfword with ONE LEA.HI
// instead of two byte extractions and a multiply-add (b0 + (b0 >> 5) <= 262 < 264: injective)
__host__ __device__ __forceinline__ uint32_t ook_rank_slot(uint32_t b0, uint32_t b1)
{
    const uint32_t raw = b0 | (b1 << 8);
    return raw + (raw >> 5);
}
static_assert(65535 + (65535 >> 5) < OOK_RANK_N, "rank table covers every slot");

// #{i : uniq[i] <= h} for ascending uniq[0..n): every lane probes one position per round
__device__ __forceinline__ uint32_t warp_upper_bound(const float *__restrict__ uniq, uint32_t n, float h, int lane)
{
    uint32_t lo = 0, hi = n;          // the answer is in [lo, hi]: uniq[i] <= h for i < lo, uniq[i] > h for i >= hi
    while (lo < hi) {
        const uint32_t step = (hi - lo + 31) / 32;
        const uint32_t p = lo + (lane + 1) * step - 1;
        const bool le = p < hi ? (__ldg(uniq + p) <= h) : false;
        const uint32_t c = __popc(__ballot_sync(0xffffffffu, le));
        const uint32_t nlo = lo + c * step;
        const uint32_t cap = lo + (c + 1) * step - 1;
        hi = cap < hi ? cap : hi;
        lo = nlo;
    }
    return lo;
}

// ---------------------------------------------------------------------------------------------
// K-C in three kernels, so that nothing heavy is tied to the walk along a stream (a warp that reads and slices a stream's
// collected blocks one after the other is bound by the latency of that walk, and a shard of 512 streams leaves three such warps
// per SM: see the rejected forms at the top of the file):
//   C1 ook_slice_kernel   : every (stream, group of 32 blocks) is an independent unit of work (grid-stride, one CTA per SM beside
//                           the rank table): collected blocks -> 512-bit masks (64 B per block) and a summary word per block
//                           {transitions between its own bits, first bit, last bit};
//   C2 ook_scan_kernel    : one warp per stream, 32 blocks per step with warp scans: bits inserted before a block (the 0.0 of
//                           vec!(0.0) that leads a burst, lone [0.0] bursts), position of every block in the flattened bit stream,
//                           index of its first entry in the transition list, transition at its first bit -- 20 bytes per block in,
//                           16 out, no sample is touched;
//   C3 ook_scatter_kernel : every (stream, group) independent again: blocks that hold a transition write them at their place.
// ---------------------------------------------------------------------------------------------
constexpr int KC1_WARPS = 28;
constexpr uint32_t KC_SUM_FIRST = 1u << 30, KC_SUM_LAST = 1u << 31, KC_SUM_CNT = 0x3ffu;

// bit i of the result: sample i of the lane's 16 (32 contiguous bytes) has rank >= h, i.e. x > max/2f32 (bitfount.rs:91)
__device__ __forceinline__ uint32_t kc_slice16(uint32_t rank_s, uint32_t hm1, const uint4 &q0, const uint4 &q1)
{
    const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t raw0 = w[i] & 0xffffu, raw1 = __umulhi(w[i], 65536u);        // w >> 16 on the FMA pipe
        const uint32_t a0 = rank_s + 2u * (raw0 + (raw0 >> 5)), a1 = rank_s + 2u * (raw1 + (raw1 >> 5));
        unsigned short r0, r1;
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r0) : "r"(a0));
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r1) : "r"(a1));
        m = __funnelshift_l(hm1 - (uint32_t)r0, m, 1);                   // rank >= h  <=>  (h - 1) - rank < 0: the sign bit
        m = __funnelshift_l(hm1 - (uint32_t)r1, m, 1);
    }
    return __brev(m) >> 16;                                              // bits arrive reversed: sample i -> bit i
}

// transitions BETWEEN the 512 bits of one block (lane l holds bits 16 l .. 16 l + 15): bit i of the result is set when sample
// 16 l + i differs from the one before it; the block's very first bit is left out (it depends on what precedes the block)
__device__ __forceinline__ uint32_t kc_inner_transitions(uint32_t m, int lane)
{
    const uint32_t pb = __shfl_up_sync(0xffffffffu, m >> 15, 1) & 1u;
    uint32_t tm = (m ^ ((m << 1) | pb)) & 0xffffu;
    if (lane == 0) tm &= ~1u;
    return tm;
}

// K-B2: what the trigger kernel leaves open about a sent burst, one warp per (stream, burst): its maximum (bitfount.rs:90 fold(0.0,
// max) -- order-free, so the per-block maxima of the blocks that carry its tag can be reduced in any order), max/2 (:91), and that
// threshold in the rank domain  #{distinct envelope values <= max/2}  (see K-C above).  The burst's blocks lie between the
// block that ended the previous burst and the one that ended this one (d_bend).
// Stream plans (STREAM): burst 0 is the one that was open when the push started; its carried blocks' running maximum is folded
// in, and the carried blocks take part in this push's slicing (live = their number) only if it is sent here.
constexpr int KC0_WARPS = 8;
template <bool STREAM>
__global__ void __launch_bounds__(KC0_WARPS * 32)
ook_burst_kernel(size_t n_streams, size_t n_blocks, size_t max_bursts, const float *__restrict__ d_max,
                 const int32_t *__restrict__ d_tag, const uint32_t *__restrict__ d_bend, const uint8_t *__restrict__ d_bflags,
                 const uint32_t *__restrict__ d_nbursts, const float *__restrict__ uniq, uint32_t n_uniq,
                 float *__restrict__ d_half, uint32_t *__restrict__ d_hrank, uint32_t *__restrict__ d_next, uint32_t next_init,
                 const OokSeam *__restrict__ seam, uint32_t *__restrict__ d_live)
{
    const int lane = threadIdx.x & 31;
    const size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) *d_next = next_init;         // the slice kernel's group counter (it runs after this one)
    if (w >= n_streams * max_bursts) return;
    const size_t st = w / max_bursts, j = w % max_bursts;
    const uint32_t nbu = d_nbursts[st], fl = d_bflags[w];                // independent loads: one latency (slots past the stream's
    const uint32_t hi = d_bend[w], lo = j ? d_bend[w - 1] + 1u : 0u;     // last burst hold stale values, never used)
    const bool sent = j < nbu && (fl & 1u);
    if (STREAM && j == 0 && lane == 0) d_live[st] = sent ? seam[st].n_carry : 0u;
    if (!sent) return;                                                   // never sent: no block carries its index
    float mx = STREAM && j == 0 ? seam[st].run_max : 0.0f;
    const size_t end = (size_t)hi + 1 < n_blocks ? (size_t)hi + 1 : n_blocks;
    for (size_t b0 = lo; b0 < end; b0 += 128) {                          // 128 blocks per step, all loads independent: one latency
        int32_t tg[4]; float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const size_t b = b0 + 32 * i + lane;
            tg[i] = b < end ? d_tag[st * n_blocks + b] : -1;
            v[i] = b < end ? d_max[st * n_blocks + b] : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) mx = tg[i] == (int32_t)j ? fmaxf(mx, v[i]) : mx;
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    const float hv = __fdiv_rn(mx, 2.0f);                                // discretize :90-91 max/2f32
    // (a two-level search -- every 32nd value staged in shared memory, one global load for the run that holds the boundary -- was
    // measured slower: 15.3 us against 13.2 for 4096 streams; every CTA pays the staging and the barrier, most warps leave at once)
    const uint32_t h = warp_upper_bound(uniq, n_uniq, hv, lane);
    if (lane == 0) { d_half[w] = hv; d_hrank[w] = h; }
}

template <bool STREAM>
__global__ void __launch_bounds__(KC1_WARPS * 32, 1)
ook_slice_kernel(const uint8_t *__restrict__ iq, size_t stream_stride, size_t n_streams, size_t n_blocks, size_t max_bursts,
                 const uint16_t *__restrict__ g_rank, const int32_t *__restrict__ d_tag, const uint32_t *__restrict__ d_hrank,
                 const float *__restrict__ d_half, const float *__restrict__ d_max,
                 uint32_t *__restrict__ d_next, uint16_t *__restrict__ d_mask, uint32_t *__restrict__ d_bsum, OokCarry carry)
{
    extern __shared__ __align__(16) uint16_t kc_rank[];
    for (int i = threadIdx.x; i < OOK_RANK_BYTES / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(kc_rank)[i] = __ldg(reinterpret_cast<const uint4 *>(g_rank) + i);
    __syncthreads();
    // warp index through a shuffle: the compiler then knows it -- and the group loop that starts from it -- is warp-uniform, and
    // leaves out the divergence guards (BRA.DIV / WARPSYNC.COLLECTIVE) it put around every vote and shuffle of the loop
    const int lane = threadIdx.x & 31, warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const uint32_t rank_s = smem_u32(kc_rank);
    // a stream's row: carry.cpitch carried slots, then the push's blocks (a batch plan has no carry)
    const size_t cp = STREAM ? carry.cpitch : 0, row = cp + n_blocks;
    const size_t groups_per_stream = (row + 31) / 32;
    const size_t n_groups = groups_per_stream * n_streams;
    const size_t warps_total = (size_t)gridDim.x * KC1_WARPS;
    constexpr int PF = 2;
    // lane l of a group looks after block l's tag and rank threshold; both are fetched ahead of the group that uses them (tags two
    // groups ahead, the thresholds -- addressed by the tags -- one), so a group starts with everything but its samples in registers.
    // Groups are handed out through a counter: the work in a group is the number of its collected blocks, 0 to 32, and bursts sit
    // at similar places in similar streams -- with a fixed stride (4144 warps = 259 x 16 groups per stream) a warp met the SAME
    // place of every stream it visited: 13 of 28 warps per SM busy on average, 340 us.  The first three groups of a warp are fixed
    // (no start-up latency), the counter -- set to 3 x warps by ook_burst_kernel -- gives out the rest three groups ahead.
    // (Handing out everything but a warp's first group through the counter was measured too: 2 % faster at 2048 and 4096 streams,
    // but a 512-stream shard -- two groups per warp, no steady state -- pays the start-up: slice 50 -> 59 us.  tools/runs/r2aw.sh)
    const uint32_t gps = (uint32_t)groups_per_stream, ng = (uint32_t)n_groups;
    auto tag_of = [&](uint32_t g) -> int32_t {
        if (g >= ng) return -1;
        const size_t b = (size_t)(g % gps) * 32 + lane;
        if (STREAM && b < cp) return b < carry.live[g / gps] ? 0 : -1;                            // carried blocks belong to burst 0
        return b - cp < n_blocks ? d_tag[(size_t)(g / gps) * n_blocks + b - cp] : -1;
    };
    auto thr_of = [&](uint32_t g, int32_t tg) -> uint32_t {
        return tg >= 0 ? d_hrank[(size_t)(g / gps) * max_bursts + tg] - 1u : 0u;           // rank >= h  <=>  (h - 1) - rank < 0
    };
    // quiet block (see QUIET BLOCKS above): its maximum does not exceed the burst's max/2, it slices to 512 zeros without being read
    auto quiet_of = [&](uint32_t g, int32_t tg) -> bool {
        if (tg < 0) return false;
        const size_t st = g / gps, b = (size_t)(g % gps) * 32 + lane;
        const float bm = STREAM && b < cp ? carry.bmax[st * cp + b] : d_max[st * n_blocks + b - cp];
        return bm <= d_half[st * max_bursts + tg];
    };
    const uint32_t wt = (uint32_t)warps_total;
    uint32_t g0 = blockIdx.x * KC1_WARPS + warp, g1 = g0 + wt, g2 = g1 + wt;
    int32_t tg_l = tag_of(g0), tg_n1 = tag_of(g1);
    uint32_t hm1_l = thr_of(g0, tg_l);
    bool q_l = quiet_of(g0, tg_l);
    while (g0 < ng) {
        uint32_t g3 = 0;
        if (lane == 0) g3 = atomicAdd(d_next, 1u);                         // consumed at the end of the iteration
        const uint32_t hm1_n1 = thr_of(g1, tg_n1);
        const bool q_n1 = quiet_of(g1, tg_n1);
        const int32_t tg_n2 = tag_of(g2);
        const size_t st = g0 / gps, b0 = (size_t)(g0 % gps) * 32;
        if (tg_l >= 0 && q_l) d_bsum[st * row + b0 + lane] = 0u;           // quiet: no transition inside, first and last bit 0
        unsigned rem = __ballot_sync(0xffffffffu, tg_l >= 0 && !q_l);
        if (rem != 0u) {
            const uint8_t *base = STREAM && b0 < cp ? carry.bytes + (st * cp + b0) * (size_t)(OOK_BLOCK * 2)
                                          : iq + st * stream_stride + (b0 - cp) * (size_t)(OOK_BLOCK * 2);
            int kA[PF], kB[PF];
            uint4 dA[PF][2], dB[PF][2];
            auto take = [&](int (&ks)[PF], uint4 (&d)[PF][2]) {
#pragma unroll
                for (int i = 0; i < PF; ++i) {
                    ks[i] = rem ? __ffs(rem) - 1 : -1;
                    if (rem) rem &= rem - 1;
                    if (ks[i] >= 0) {
                        const uint4 *p = reinterpret_cast<const uint4 *>(base + ks[i] * (size_t)(OOK_BLOCK * 2) + lane * 32);
                        d[i][0] = ldg_stream_u4(p); d[i][1] = ldg_stream_u4(p + 1);
                    }
                }
            };
            // the group's rows of the two outputs: a block adds its index
            uint16_t *mask_g = d_mask + (st * row + b0) * 32 + lane;
            uint32_t *bsum_g = d_bsum + st * row + b0;
            auto slice = [&](const int (&ks)[PF], const uint4 (&d)[PF][2]) {
#pragma unroll
                for (int i = 0; i < PF; ++i) {
                    if (ks[i] < 0) continue;                              // warp-uniform
                    const uint32_t hm1 = __shfl_sync(0xffffffffu, hm1_l, ks[i]);
                    const uint32_t m = kc_slice16(rank_s, hm1, d[i][0], d[i][1]);
                    mask_g[ks[i] * 32] = (uint16_t)m;                     // 64 contiguous bytes per block
                    const uint32_t tm = kc_inner_transitions(m, lane);
                    uint32_t cnt = 0;
                    if (__ballot_sync(0xffffffffu, tm != 0u) != 0u) cnt = __reduce_add_sync(0xffffffffu, __popc(tm));
                    const uint32_t first = __ballot_sync(0xffffffffu, m & 1u) & 1u;              // lane 0, bit 0
                    const uint32_t last = __ballot_sync(0xffffffffu, m & 0x8000u) >> 31;         // lane 31, bit 15
                    if (lane == 0) bsum_g[ks[i]] = cnt | (first ? KC_SUM_FIRST : 0u) | (last ? KC_SUM_LAST : 0u);
                }
            };
            // two batches in turn: one is sliced while the other's loads are in flight (no register copies between them).
            // (A half-warp per block -- 32 samples = 64 bytes per lane, two blocks per step, half the per-block overhead per lane --
            // was measured slower: slice 254 us against 225 for 4096 streams, 0.185 against 0.184 ms for a 512-stream chain.  The
            // kernel is not bound by its instruction count.  Nor by the data in flight: three batches in turn on 20 warps x 102
            // registers measured 232 us; nor by the L2 being asked for every 32-byte sector twice -- the two 128-bit loads of a
            // lane share a sector -- since loads that allocate in L1 changed nothing: tools/runs/r2ao.sh.)
            take(kA, dA);
            while (true) {
                take(kB, dB);
                slice(kA, dA);
                if (kB[0] < 0) break;
                take(kA, dA);
                slice(kB, dB);
                if (kA[0] < 0) break;
            }
        }
        tg_l = tg_n1; hm1_l = hm1_n1; q_l = q_n1; tg_n1 = tg_n2;
        g0 = g1; g1 = g2; g2 = __shfl_sync(0xffffffffu, g3, 0);
    }
}

// per collected block, written by C2: .x position of its first bit in the flattened bit stream, .y index of its first entry in the
// transition list, .z position of the transition made by the zeros inserted before it (valid with KC_INFO_PRE), .w flags
constexpr uint32_t KC_INFO_PRE = 1u, KC_INFO_FIRST = 2u;
constexpr int KC2_WARPS = 4;

template <bool STREAM>
__global__ void __launch_bounds__(KC2_WARPS * 32)
ook_scan_kernel(size_t n_streams, size_t n_blocks, size_t max_bursts, size_t max_runs, const int32_t *__restrict__ d_tag,
                const uint32_t *__restrict__ d_bsum, const uint8_t *__restrict__ d_bflags, const uint32_t *__restrict__ d_nbursts,
                uint4 *__restrict__ d_binfo, uint32_t *__restrict__ d_trans, uint32_t *__restrict__ d_ntrans,
                uint32_t *__restrict__ d_nbits, OokCarry carry, OokSeam *__restrict__ seam)
{
    const int lane = threadIdx.x & 31;
    const size_t st = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (st >= n_streams) return;
    const size_t cp = STREAM ? carry.cpitch : 0, row = cp + n_blocks;
    const int32_t *tag = d_tag + st * n_blocks;
    const uint32_t *bsum = d_bsum + st * row;
    const uint8_t *flags = d_bflags + st * max_bursts;
    uint4 *binfo = d_binfo + st * row;
    // bursts that were sent without a collected block (the OOM guard reset the buffer to [0.0] with the counter at 1, :52-54 and
    // :78-81): one 0 bit each, found among the burst indices the walk steps over (flags == 3: sent, leading 0.0)
    auto lone_zero_bursts = [&](int32_t from, int32_t to) {
        uint32_t n = 0;
        for (int32_t j = from; j < to; ++j) n += (flags[j] & 3u) == 3u ? 1u : 0u;
        return n;
    };
    uint32_t pos = 0, ntr = 0, prev = 0;          // the walk's carry: bits so far, transitions so far, value of the last bit
    // a stream plan's bit positions count from the start of the push; `any`: bits were emitted before it (the value of the last one
    // is `prev`), so the push's very first bit may be a transition
    const bool any = STREAM && seam[st].any;
    if (any) prev = seam[st].prev;
    int32_t cur_burst = -1;
    constexpr int CH = 4;                         // groups whose tags and summaries are fetched together (one latency per 128 blocks)
    // the row: the carried blocks of a burst sent in this push (all of burst 0), then the push's blocks
    const size_t live = STREAM ? carry.live[st] : 0;
    // one step: 32 x CH blocks of the row from c0 (row positions below hi); carried blocks all belong to burst 0
    auto step = [&](size_t c0, size_t hi, bool carried) {
        int32_t tgs[CH]; uint32_t sms[CH];
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const size_t b = c0 + 32 * c + lane;
            tgs[c] = b < hi ? (carried ? 0 : tag[b - cp]) : -1;
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const size_t b = c0 + 32 * c + lane;
            sms[c] = b < hi ? bsum[b] : 0u;                // not behind the tag's latency; only read where the block is collected
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int32_t tg = tgs[c];
            const bool col = tg >= 0;
            const unsigned cmask = __ballot_sync(0xffffffffu, col);
            if (cmask == 0u) continue;                                     // warp-uniform
            const uint32_t sm = sms[c];
            const uint32_t first = (sm & KC_SUM_FIRST) ? 1u : 0u, last = (sm & KC_SUM_LAST) ? 1u : 0u, cnt = sm & KC_SUM_CNT;
            // the collected block before this one: in the group, or the carry
            const unsigned lower = cmask & ((1u << lane) - 1u);
            const int pidx = lower ? 31 - __clz(lower) : 0;
            const int32_t ptag_g = __shfl_sync(0xffffffffu, tg, pidx);
            const uint32_t plast_g = __shfl_sync(0xffffffffu, last, pidx);
            const int32_t ptag = lower ? ptag_g : cur_burst;
            const uint32_t plast = lower ? plast_g : prev;
            // bits inserted before the block: lone [0.0] bursts stepped over, then the burst's own leading 0.0
            uint32_t n_ins = 0;
            if (col && tg != ptag) n_ins = lone_zero_bursts(ptag + 1, tg) + ((flags[tg] & 2u) ? 1u : 0u);
            const uint32_t bits = col ? (uint32_t)OOK_BLOCK + n_ins : 0u;
            uint32_t incl = bits;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += v;
            }
            const uint32_t pos_ins = pos + incl - bits;                    // where the inserted zeros start
            const uint32_t pos_base = pos_ins + n_ins;                     // the block's first bit
            const uint32_t before = n_ins ? 0u : plast;                    // value of the bit before it
            const bool pre = col && n_ins && (pos_ins > 0u || any) && plast != 0u;   // 1 -> 0 at the first inserted zero
            const bool firstT = col && (pos_base > 0u || any) && first != before;
            const uint32_t mine = col ? cnt + (pre ? 1u : 0u) + (firstT ? 1u : 0u) : 0u;
            uint32_t tincl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, tincl, d);
                if (lane >= d) tincl += v;
            }
            if (col)
                binfo[c0 + 32 * c + lane] = make_uint4(pos_base, ntr + tincl - mine, pos_ins,
                                                       (pre ? KC_INFO_PRE : 0u) | (firstT ? KC_INFO_FIRST : 0u));
            const int lastc = 31 - __clz(cmask);
            pos += __shfl_sync(0xffffffffu, incl, 31);
            ntr += __shfl_sync(0xffffffffu, tincl, 31);
            cur_burst = __shfl_sync(0xffffffffu, tg, lastc);
            prev = __shfl_sync(0xffffffffu, last, lastc);
        }
    };
    if constexpr (STREAM)
        for (size_t c0 = 0; c0 < live; c0 += 32 * CH) step(c0, live, true);
    for (size_t c0 = cp; c0 < row; c0 += 32 * CH) step(c0, row, false);
    {   // lone [0.0] bursts after the last collected block
        const uint32_t nbu = d_nbursts[st];
        const uint32_t n = lone_zero_bursts(cur_burst + 1, (int32_t)(nbu < max_bursts ? nbu : max_bursts));
        if (n) {
            if ((pos > 0u || any) && prev != 0u) { if (lane == 0 && ntr < max_runs) d_trans[st * max_runs + ntr] = pos; ntr++; }
            pos += n;
            prev = 0u;
        }
    }
    if (lane == 0) {
        d_ntrans[st] = ntr; d_nbits[st] = pos;
        if (STREAM && pos > 0u) { seam[st].prev = prev; seam[st].any = 1u; }
    }
}

constexpr int KC3_WARPS = 8;

// C3: lane l of a warp owns block l of a (stream, group): its transitions go to consecutive entries of the list starting at the
// index C2 gave it, so no lane needs another's count -- the blocks of a group are written side by side, each lane fetching the 64
// bytes of its own mask in one go
template <bool STREAM>
__global__ void __launch_bounds__(KC3_WARPS * 32)
ook_scatter_kernel(size_t n_streams, size_t n_blocks, size_t max_runs, const int32_t *__restrict__ d_tag,
                   const uint32_t *__restrict__ d_bsum, const uint4 *__restrict__ d_binfo, const uint16_t *__restrict__ d_mask,
                   uint32_t *__restrict__ d_trans, OokCarry carry)
{
    const int lane = threadIdx.x & 31;
    const size_t cp = STREAM ? carry.cpitch : 0, row = cp + n_blocks;
    const size_t groups_per_stream = (row + 31) / 32;
    const size_t n_groups = groups_per_stream * n_streams;
    const size_t grp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (grp >= n_groups) return;
    const size_t st = grp / groups_per_stream, b = (grp % groups_per_stream) * 32 + lane;
    if (b >= row) return;
    if (STREAM && b < cp ? b >= carry.live[st] : d_tag[st * n_blocks + b - cp] < 0) return;
    const size_t blk = st * row + b;
    const uint32_t sm = d_bsum[blk];
    const uint4 info = d_binfo[blk];
    uint32_t *trans = d_trans + st * max_runs;
    uint32_t o = info.y;
    if (info.w & KC_INFO_PRE) { if (o < max_runs) trans[o] = info.z; ++o; }        // 1 -> 0 at the zeros inserted before the block
    if (info.w & KC_INFO_FIRST) { if (o < max_runs) trans[o] = info.x; ++o; }      // at the block's first bit
    if ((sm & KC_SUM_CNT) == 0u) return;
    const uint4 *mp = reinterpret_cast<const uint4 *>(d_mask + blk * 32);
    uint4 q[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) q[i] = __ldg(mp + i);
    uint32_t prevbit = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint4 &v = q[i >> 2];
        const uint32_t w = (i & 3) == 0 ? v.x : (i & 3) == 1 ? v.y : (i & 3) == 2 ? v.z : v.w;
        uint32_t tm = w ^ ((w << 1) | prevbit);
        if (i == 0) tm &= ~1u;                                                     // the first bit was dealt with above
        prevbit = w >> 31;
        while (tm) {
            const int b = __ffs(tm) - 1;
            tm &= tm - 1;
            if (o < max_runs) trans[o] = info.x + 32u * i + b;
            ++o;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K-D: dle + matchers + shaper_optional, one thread per stream
// ---------------------------------------------------------------------------------------------

// The pulse-pair matchers of ratpak.rs:88-97 (looper bodies) and shaper_optional (kpn.rs:266-275), one run at a time.
// Lane 0 runs protocol A and lane 1 protocol B in the same warp, so the two state machines are written as ONE instruction
// stream of selects over per-protocol constants (as branches the lanes would take turns, and every run costs a reconvergence):
//   idle      : run value 1 with a duration in [a1lo, a1hi] or [a2lo, a2hi] starts a pair (the FOLLOWING run is consumed,
//               `a.next().unwrap()`), anything else is None for the shaper
//   pair open : the run must be a 0 with a duration in [s1lo, s1hi] or [s2lo, s2hi]: Some(bit), bit = "second range" for
//               protocol A (:91-92), d > e for protocol B (:96); anything else None
//   shaper    : Some(y) => push; None => the collected bits are sent iff there are exactly `want` of them, then cleared.
// A pulse still pending when the runs end: the reference block dies in unwrap() with nothing sent.
struct Matcher {
    float a1lo, a1hi, a2lo, a2hi, s1lo, s1hi, s2lo, s2hi;
    bool  proto_b;
    bool  pending; float d;
    unsigned long long acc; uint32_t n, want, count, base;      // out[k] holds packet base + k
    unsigned long long *out; size_t cap;
    __device__ __forceinline__ void init(int proto, unsigned long long *o, size_t c)
    {
        proto_b = proto != 0;
        a1lo = proto_b ? 125e-6f : 2e-4f;  a1hi = proto_b ? 250e-6f : 6e-4f;                 // ratpak.rs:91 / :96, first run
        a2lo = proto_b ? 500e-6f : 1.0f;   a2hi = proto_b ? 650e-6f : 0.0f;                  // (A has no second range: empty)
        s1lo = proto_b ? 500e-6f : 1.5e-3f; s1hi = proto_b ? 650e-6f : 2.5e-3f;              // second run
        s2lo = proto_b ? 125e-6f : 3.5e-3f; s2hi = proto_b ? 250e-6f : 4.5e-3f;
        pending = false; d = 0.0f; acc = 0ull; n = 0u; want = proto_b ? 24u : 36u; count = 0u; base = 0u; out = o; cap = c;
    }
    __device__ __forceinline__ void load(const OokSeam &z, int p, uint32_t b)
    {
        pending = z.m_pending[p] != 0; d = z.m_d[p]; acc = z.m_acc[p]; n = z.m_n[p]; count = z.m_count[p]; base = b;
    }
    __device__ __forceinline__ void store(OokSeam &z, int p) const
    {
        z.m_pending[p] = pending ? 1u : 0u; z.m_d[p] = d; z.m_acc[p] = acc; z.m_n[p] = n; z.m_count[p] = count;
    }
    __device__ __forceinline__ void feed(uint32_t v, float dur)
    {
        const bool first_ok = v == 1u && ((dur >= a1lo && dur <= a1hi) || (dur >= a2lo && dur <= a2hi));
        const bool r1 = dur >= s1lo && dur <= s1hi, r2 = dur >= s2lo && dur <= s2hi;
        const bool second_ok = v == 0u && (r1 || r2);
        const uint32_t bit = proto_b ? (d > dur ? 1u : 0u) : (r1 ? 0u : 1u);
        const bool push = pending && second_ok;
        const bool none = pending ? !second_ok : !first_ok;
        d = pending ? d : dur;                                    // only read while a pair is open
        pending = !pending && first_ok;
        // Some(y) => x.push(y)
        const unsigned long long pushed = (acc << 1) | (unsigned long long)bit;
        acc = push && n < 64u ? pushed : acc;
        n += push ? 1u : 0u;
        // None if x.len() == l => send; None => clear
        if (none) {
            if (n == want) { if (count - base < cap) out[count - base] = acc; count++; }
            n = 0u; acc = 0ull;
        }
    }
};

// One warp per stream.  Run lengths -> seconds (dle) is data-parallel: the lanes turn a chunk of 256
// transitions into durations in shared memory with coalesced reads; the matchers are sequential, so lane 0
// (proto A) and lane 1 (proto B) then walk the chunk from shared memory instead of chasing global loads.
// Stream plans (STREAM): the first run of the push continues the open run carried from the pushes before, the matchers
// resume where they stopped, packets are numbered on from there and stored from d_pbase (the first one not fetched yet).
constexpr int KD_WARPS = 4, KD_CHUNK = 256;

template <bool STREAM>
__global__ void __launch_bounds__(KD_WARPS * 32)
ook_match_kernel(const uint32_t *__restrict__ d_trans, const uint32_t *__restrict__ d_ntrans, size_t n_streams,
                 size_t max_runs, size_t max_packets, float s_rate_f, unsigned long long *__restrict__ d_packets,
                 uint32_t *__restrict__ d_npackets, uint32_t *__restrict__ d_runs_dbg,
                 OokSeam *__restrict__ seam, const uint32_t *__restrict__ d_nbits, const uint32_t *__restrict__ d_pbase)
{
    __shared__ float s_dur[KD_WARPS][KD_CHUNK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t st = (size_t)blockIdx.x * KD_WARPS + warp;
    if (st >= n_streams) return;
    const uint32_t *tr = d_trans + st * max_runs;
    const uint32_t nr_all = d_ntrans[st];
    uint32_t nr = nr_all;
    if (nr > max_runs) nr = (uint32_t)max_runs;           // overflow is reported by fetch
    // run k: value = (v0 + k) & 1, length = tr[k] - tr[k-1]; the stream starts with the 0 bit of vec!(0.0), so v0 = 0 from the
    // initial state; the first run of a push adds the length the open run had reached before it
    const unsigned long long len0 = STREAM ? seam[st].run_len : 0ull;
    const uint32_t v0 = STREAM ? seam[st].run_val : 0u;
    uint32_t *dbg = d_runs_dbg + st * max_runs;
    Matcher mt;
    mt.init(lane & 1, d_packets + (st * 2 + (lane & 1)) * max_packets, max_packets);
    if (STREAM && lane < 2) mt.load(seam[st], lane, d_pbase[st * 2 + lane]);
    float *dur = s_dur[warp];
    for (uint32_t k0 = 0; k0 < nr; k0 += KD_CHUNK) {
        const uint32_t nk = nr - k0 < (uint32_t)KD_CHUNK ? nr - k0 : (uint32_t)KD_CHUNK;
        for (uint32_t i = lane; i < nk; i += 32) {
            const uint32_t k = k0 + i;
            const uint32_t len = tr[k] - (k ? tr[k - 1] : 0u);
            const uint32_t v = (v0 + k) & 1u;
            if (k == 0 && len0) {
                const unsigned long long l = len0 + len;
                dbg[k] = (v << 31) | (uint32_t)(l < 0x7fffffffull ? l : 0x7fffffffull);
                dur[i] = __fdiv_rn(__ull2float_rn(l), s_rate_f);                         // dle kpn.rs:35 (ct as f32)
            } else {
                dbg[k] = (v << 31) | len;
                dur[i] = __fdiv_rn((float)len, s_rate_f);                               // dle kpn.rs:35
            }
        }
        __syncwarp();
        if (lane < 2)
            for (uint32_t i = 0; i < nk; ++i) mt.feed((v0 + k0 + i) & 1u, dur[i]);
        __syncwarp();
    }
    if (lane < 2) d_npackets[st * 2 + lane] = mt.count;
    if (STREAM) {
        if (lane < 2) mt.store(seam[st], lane);
        if (lane == 0) {
            const uint32_t nbits = d_nbits[st];
            OokSeam &z = seam[st];
            if (nr == 0) z.run_len = len0 + nbits;
            else { z.run_len = nbits - tr[nr - 1]; z.run_val = (v0 + nr) & 1u; }
            if (nr_all > max_runs) z.err |= OOK_ERR_RUNS;
        }
    }
}

// Stream plans, after the slicer: the blocks of the burst still open at the end of the push (tagged OOK_TAG_OPEN by the trigger
// kernel) are appended to the stream's carry region with their maxima.  discretize (bitfount.rs:87-96) needs the burst's maximum
// before its first bit, so they are sliced in the push that sends the burst, read in place from here.  If no burst was sent or
// dropped in this push (d_nbursts = 0) the open burst is the one carried in and they go after its blocks; otherwise the carry
// starts over.  One warp per stream copies four blocks at a time (32 bytes per lane per block).
constexpr int KCY_WARPS = 4;
__global__ void __launch_bounds__(KCY_WARPS * 32)
ook_carry_kernel(const uint8_t *__restrict__ iq, size_t stream_stride, size_t n_streams, size_t n_blocks, size_t cpitch,
                 size_t max_carry, const int32_t *__restrict__ d_tag, const float *__restrict__ d_max,
                 const uint32_t *__restrict__ d_nbursts, uint8_t *__restrict__ d_carry, float *__restrict__ d_cmax,
                 OokSeam *__restrict__ seam)
{
    const int lane = threadIdx.x & 31;
    const size_t st = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (st >= n_streams) return;
    const bool cont = d_nbursts[st] == 0u;
    size_t n = cont ? seam[st].n_carry : 0u;
    float mx = cont ? seam[st].run_max : 0.0f;
    const int32_t *tag = d_tag + st * n_blocks;
    const float *bmax = d_max + st * n_blocks;
    const uint8_t *src = iq + st * stream_stride + lane * 32;
    uint8_t *dst = d_carry + st * cpitch * (size_t)(OOK_BLOCK * 2) + lane * 32;
    float *cmax = d_cmax + st * cpitch;
    for (size_t b0 = 0; b0 < n_blocks; b0 += 32) {
        const size_t b = b0 + lane;
        const bool open = b < n_blocks && tag[b] == OOK_TAG_OPEN;
        unsigned rem = __ballot_sync(0xffffffffu, open);
        if (!rem) continue;                                                      // warp-uniform
        const float bm = open ? bmax[b] : 0.0f;
        mx = fmaxf(mx, bm);
        if (open && n + __popc(rem & ((1u << lane) - 1u)) < max_carry) cmax[n + __popc(rem & ((1u << lane) - 1u))] = bm;
        while (rem) {
            int k[4]; uint4 v[4][2];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                k[i] = rem ? __ffs(rem) - 1 : -1;
                if (rem) rem &= rem - 1u;
                if (k[i] >= 0 && n + i < max_carry) {
                    const uint4 *p = reinterpret_cast<const uint4 *>(src + (b0 + k[i]) * (size_t)(OOK_BLOCK * 2));
                    v[i][0] = ldg_stream_u4(p); v[i][1] = ldg_stream_u4(p + 1);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (k[i] < 0) break;
                if (n < max_carry) {
                    uint4 *q = reinterpret_cast<uint4 *>(dst + n * (size_t)(OOK_BLOCK * 2));
                    q[0] = v[i][0]; q[1] = v[i][1];
                }
                ++n;
            }
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    if (lane == 0) {
        if (n > max_carry) { seam[st].err |= OOK_ERR_CARRY; n = max_carry; }
        seam[st].n_carry = (uint32_t)n;
        seam[st].run_max = mx;
    }
}

__global__ void ook_envelope_table_kernel(float *__restrict__ table)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 65536u) table[i] = lr_envelope(i >> 8, i & 0xffu);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// bitfount.rs:52 `1000*trigger_duration*block_size`.  LRC_OOK_TEST_GUARD_BLOCKS shrinks it (in blocks) so that a test can reach
// the guard with a capture of a few hundred blocks instead of 50 000; the oracle has the same hook (orc_test_set_trigger_guard)
static size_t ook_guard_blocks()
{
    if (const char *g = getenv("LRC_OOK_TEST_GUARD_BLOCKS")) { const long v = atol(g); if (v >= 1) return (size_t)v; }
    return 1000u * (size_t)OOK_TRIGGER_DURATION;
}

// stream s's packets of both protocols from the matcher's output pk ([stream][2][mp], packed MSB-first): n[proto] of them,
// numbered from seq0[proto], written from `out` on; returns the end of what it wrote
static lrc_ook_packet *ook_put_packets(lrc_ook_packet *out, const unsigned long long *pk, size_t mp, size_t s, const uint32_t n[2],
                                       const uint32_t seq0[2])
{
    for (int proto = 0; proto < 2; ++proto) {
        const uint32_t nbits = proto == 0 ? 36u : 24u;
        for (uint32_t k = 0; k < n[proto]; ++k) {
            lrc_ook_packet &p = *out++;
            p.stream = (uint32_t)s; p.proto = (uint32_t)proto; p.seq = seq0[proto] + k; p.nbits = nbits;
            memset(p.bits, 0, sizeof(p.bits));
            const unsigned long long v = pk[(s * 2 + proto) * mp + k];
            for (uint32_t i = 0; i < nbits; ++i) p.bits[i] = (uint8_t)((v >> (nbits - 1 - i)) & 1ull);
        }
    }
    return out;
}

// cpitch: carry slots per stream in front of the blocks of the slicer's per-block arrays (stream plans; 0 for a batch plan)
static int ook_create(lrc_ctx *ctx, size_t n_streams, size_t n_blocks, size_t cpitch, unsigned sample_rate,
                      size_t max_runs, size_t max_packets, lrc_ook **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && n_streams >= 1 && n_blocks >= 1 && sample_rate >= 1, LRC_ERR_INVALID, "lrc_ook_create: bad arguments");
    LRC_REQUIRE(n_blocks * (size_t)OOK_BLOCK < 0xffffffffull, LRC_ERR_UNSUPPORTED, "lrc_ook_create: capture too long (2^32 samples)");
    LRC_REQUIRE(n_streams * ((cpitch + n_blocks + 31) / 32) < 0x7fffffffull, LRC_ERR_UNSUPPORTED,
                "lrc_ook_create: too many 32-block groups (2^31)");
    lrc_ook *o = new (std::nothrow) lrc_ook();
    LRC_REQUIRE(o != nullptr, LRC_ERR_NOMEM, "out of host memory");
    o->ctx = ctx; o->n_streams = n_streams; o->n_blocks = n_blocks; o->sample_rate = sample_rate; o->cpitch = cpitch;
    o->max_runs = max_runs ? max_runs : 4096;
    o->max_packets = max_packets ? max_packets : 64;
    const size_t guard_blocks = ook_guard_blocks();
    o->guard_samples = (uint32_t)(guard_blocks * OOK_BLOCK);
    // a sent burst is at least 49 collected blocks, except the pieces the guard cuts one into (an abandoned burst of more than
    // guard_blocks blocks followed by its remainder, possibly empty): at least guard_blocks / 2 blocks per index on average
    const size_t min_burst = std::min<size_t>(49, std::max<size_t>(1, guard_blocks / 2));
    // (+ 1 for a stream plan: the burst carried in may be dropped by the guard, and a lone [0.0] sent, within two blocks)
    o->max_bursts = n_blocks / min_burst + 2 + (cpitch ? 1 : 0);
    const size_t sb = n_streams * n_blocks, sr = n_streams * (cpitch + n_blocks);
    cudaError_t e = cudaSuccess;
#define OOK_ALLOC(buf, count) if (e == cudaSuccess) e = o->buf.alloc(count)
    OOK_ALLOC(d_sum, sb); OOK_ALLOC(d_max, sb); OOK_ALLOC(d_tag, sb);
    OOK_ALLOC(d_half, n_streams * o->max_bursts); OOK_ALLOC(d_bflags, n_streams * o->max_bursts);
    OOK_ALLOC(d_bend, n_streams * o->max_bursts);
    OOK_ALLOC(d_nbursts, n_streams);
    OOK_ALLOC(d_trans, n_streams * o->max_runs); OOK_ALLOC(d_ntrans, n_streams); OOK_ALLOC(d_nbits, n_streams);
    OOK_ALLOC(d_packets, n_streams * 2 * o->max_packets); OOK_ALLOC(d_npackets, n_streams * 2);
    OOK_ALLOC(d_runs_dbg, n_streams * o->max_runs);
    OOK_ALLOC(d_mask, sr * 32); OOK_ALLOC(d_bsum, sr); OOK_ALLOC(d_binfo, sr); OOK_ALLOC(d_hrank, n_streams * o->max_bursts); OOK_ALLOC(d_next, 1);
    OOK_ALLOC(d_flut, (size_t)OOK_FLUT_N);
    OOK_ALLOC(d_rank, (size_t)OOK_RANK_N); OOK_ALLOC(d_uniq, (size_t)65536);
#undef OOK_ALLOC
    if (e == cudaSuccess) {
        e = cudaMemsetAsync(o->d_flut, 0, OOK_FLUT_BYTES, ctx->stream);   // the row skew gaps are never read
        if (e == cudaSuccess) {
            ook_build_flut_kernel<<<256, 256, 0, ctx->stream>>>(o->d_flut);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ook_block_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KA2_SMEM_BYTES);
        if (e == cudaSuccess) {
            cudaDriverEntryPointQueryResult qr;
            e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &o->encode_tiled, cudaEnableDefault, &qr);
            if (e == cudaSuccess && (qr != cudaDriverEntryPointSuccess || !o->encode_tiled)) {
                lrc_set_error("lrc_ook_create: the driver does not export cuTensorMapEncodeTiled");
                lrc_ook_destroy(o);
                return LRC_ERR_UNSUPPORTED;
            }
        }
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ook_slice_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, OOK_RANK_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ook_slice_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, OOK_RANK_BYTES);
    }
    if (e == cudaSuccess) {
        // rank table for the slicer: the envelope of every byte pair, computed ON THE DEVICE by the routine the
        // block-sum kernel uses, ordered on the host (a plain sort of 65536 floats, no arithmetic)
        ook_envelope_table_kernel<<<256, 256, 0, ctx->stream>>>(o->d_uniq);          // d_uniq as scratch: index b0*256 + b1
        e = cudaGetLastError();
        std::vector<float> tab(65536);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpy(tab.data(), o->d_uniq, 65536 * sizeof(float), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) {
            std::vector<float> uq(tab);
            std::sort(uq.begin(), uq.end());
            uq.erase(std::unique(uq.begin(), uq.end()), uq.end());
            std::vector<uint16_t> rank(OOK_RANK_N, 0);
            // tab index = b0 * 256 + b1; the table is symmetric in the two bytes
            for (uint32_t i = 0; i < 65536; ++i)
                rank[ook_rank_slot(i >> 8, i & 0xffu)] = (uint16_t)(std::lower_bound(uq.begin(), uq.end(), tab[i]) - uq.begin());
            o->n_uniq = (uint32_t)uq.size();
            e = cudaMemcpy(o->d_uniq, uq.data(), uq.size() * sizeof(float), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(o->d_rank, rank.data(), rank.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
        }
    }
    if (e != cudaSuccess) {
        lrc_set_error("lrc_ook_create: %s", cudaGetErrorString(e));
        lrc_ook_destroy(o);
        return LRC_ERR_CUDA;
    }
    *out = o;
    return LRC_OK;
}

extern "C" int lrc_ook_create(lrc_ctx *ctx, size_t n_streams, size_t n_blocks, unsigned sample_rate,
                              size_t max_runs, size_t max_packets, lrc_ook **out)
{
    return ook_create(ctx, n_streams, n_blocks, 0, sample_rate, max_runs, max_packets, out);
}

extern "C" int lrc_ook_destroy(lrc_ook *o)
{
    if (!o) return LRC_OK;
    cudaSetDevice(o->ctx->device);
    delete o;
    return LRC_OK;
}

// what a stream plan adds to a launch of the chain (null: a batch plan, every stream from the initial state)
struct OokStreamLaunch {
    OokSeam  *seam;
    OokCarry  carry;
    uint8_t  *d_carry;
    float    *d_cmax;
    uint32_t *d_live, *d_pbase;
    size_t    max_carry;
};

// the whole chain on n_blocks blocks per stream (n_blocks <= o->n_blocks: a stream plan's push may be shorter than its maximum).
// STREAM = (sl != null); the batch plan's kernels are compiled without any of the stream plan's state.
template <bool STREAM>
static int ook_launch(lrc_ook *o, const uint8_t *d_iq, size_t n_blocks, size_t stream_stride_bytes, cudaStream_t s,
                      const OokStreamLaunch *sl)
{
    const size_t groups = ((n_blocks + 31) / 32) * o->n_streams;
    const size_t cap = (size_t)o->ctx->n_sm;           // one persistent CTA per SM (the table fills its shared memory)
    // the capture as a byte tensor [stream][block][1024]: one box = 64 bytes of 32 consecutive blocks of one stream
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    CUtensorMap tm;
    const cuuint64_t dims[3] = {(cuuint64_t)OOK_BLOCK * 2, (cuuint64_t)n_blocks, (cuuint64_t)o->n_streams};
    const cuuint64_t strides[2] = {(cuuint64_t)OOK_BLOCK * 2, (cuuint64_t)stream_stride_bytes};
    const cuuint32_t box[3] = {KA2_SLAB_BYTES, 32, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult cr = reinterpret_cast<encode_fn>(o->encode_tiled)(
        &tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t *>(d_iq), dims, strides, box, estr,
        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
        lrc_set_error("lrc_ook_decode: cuTensorMapEncodeTiled -> CUresult %d (n_blocks %zu, n_streams %zu, stride %zu)",
                      (int)cr, n_blocks, o->n_streams, stream_stride_bytes);
        return LRC_ERR_CUDA;
    }
    const size_t ka_blocks = std::min(ceil_div(groups, (size_t)KA2_WARPS), cap);
    ook_block_tma_kernel<<<(unsigned)ka_blocks, KA2_WARPS * 32, KA2_SMEM_BYTES, s>>>(tm, o->n_streams, n_blocks, o->d_flut,
                                                                                   o->d_sum, o->d_max);
    LRC_CUDA(cudaGetLastError());
    ook_trigger_kernel<STREAM><<<(unsigned)ceil_div(o->n_streams, (size_t)KB_STREAMS), KB_THREADS, 0, s>>>(
        o->d_sum, o->n_streams, n_blocks, o->max_bursts, o->guard_samples, o->d_tag, o->d_bend, o->d_bflags, o->d_nbursts,
        sl ? sl->seam : nullptr);
    LRC_CUDA(cudaGetLastError());
    const OokCarry carry = sl ? sl->carry : OokCarry{0, nullptr, nullptr, nullptr};
    OokSeam *seam = sl ? sl->seam : nullptr;
    const size_t slice_groups = ((carry.cpitch + n_blocks + 31) / 32) * o->n_streams;
    const size_t kc1_blocks = std::min(ceil_div(slice_groups, (size_t)KC1_WARPS), cap);
    ook_burst_kernel<STREAM><<<(unsigned)ceil_div(o->n_streams * o->max_bursts, (size_t)KC0_WARPS), KC0_WARPS * 32, 0, s>>>(
        o->n_streams, n_blocks, o->max_bursts, o->d_max, o->d_tag, o->d_bend, o->d_bflags, o->d_nbursts, o->d_uniq, o->n_uniq,
        o->d_half, o->d_hrank, o->d_next, (uint32_t)(3 * kc1_blocks * KC1_WARPS), seam, sl ? sl->d_live : nullptr);
    LRC_CUDA(cudaGetLastError());
    ook_slice_kernel<STREAM><<<(unsigned)kc1_blocks, KC1_WARPS * 32, OOK_RANK_BYTES, s>>>(
        d_iq, stream_stride_bytes, o->n_streams, n_blocks, o->max_bursts, o->d_rank, o->d_tag, o->d_hrank, o->d_half,
        o->d_max, o->d_next, o->d_mask, o->d_bsum, carry);
    LRC_CUDA(cudaGetLastError());
    ook_scan_kernel<STREAM><<<(unsigned)ceil_div(o->n_streams, (size_t)KC2_WARPS), KC2_WARPS * 32, 0, s>>>(
        o->n_streams, n_blocks, o->max_bursts, o->max_runs, o->d_tag, o->d_bsum, o->d_bflags, o->d_nbursts, o->d_binfo,
        o->d_trans, o->d_ntrans, o->d_nbits, carry, seam);
    LRC_CUDA(cudaGetLastError());
    ook_scatter_kernel<STREAM><<<(unsigned)ceil_div(slice_groups, (size_t)KC3_WARPS), KC3_WARPS * 32, 0, s>>>(
        o->n_streams, n_blocks, o->max_runs, o->d_tag, o->d_bsum, o->d_binfo, o->d_mask, o->d_trans, carry);
    LRC_CUDA(cudaGetLastError());
    if constexpr (STREAM) {
        // after the slicer has read the carried blocks of a burst sent in this push: the carry may start over
        ook_carry_kernel<<<(unsigned)ceil_div(o->n_streams, (size_t)KCY_WARPS), KCY_WARPS * 32, 0, s>>>(
            d_iq, stream_stride_bytes, o->n_streams, n_blocks, carry.cpitch, sl->max_carry, o->d_tag, o->d_max, o->d_nbursts,
            sl->d_carry, sl->d_cmax, sl->seam);
        LRC_CUDA(cudaGetLastError());
    }
    ook_match_kernel<STREAM><<<(unsigned)ceil_div(o->n_streams, (size_t)KD_WARPS), KD_WARPS * 32, 0, s>>>(
        o->d_trans, o->d_ntrans, o->n_streams, o->max_runs, o->max_packets, (float)o->sample_rate, o->d_packets,
        o->d_npackets, o->d_runs_dbg, seam, o->d_nbits, sl ? sl->d_pbase : nullptr);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_ook_decode(lrc_ook *o, const uint8_t *d_iq, size_t stream_stride_bytes, void *stream)
{
    LRC_REQUIRE(o != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(o->ctx);
    LRC_REQUIRE(d_iq != nullptr, LRC_ERR_INVALID, "lrc_ook_decode: null input");
    LRC_REQUIRE(stream_stride_bytes >= o->n_blocks * (size_t)OOK_BLOCK * 2, LRC_ERR_INVALID, "lrc_ook_decode: stride too short");
    LRC_REQUIRE(((uintptr_t)d_iq & 15) == 0 && (stream_stride_bytes & 15) == 0, LRC_ERR_INVALID,
                "lrc_ook_decode: input and stream stride must be 16-byte aligned");
    return ook_launch<false>(o, d_iq, o->n_blocks, stream_stride_bytes, lrc_stream(o->ctx, stream), nullptr);
}

extern "C" int lrc_ook_fetch_packets(lrc_ook *o, lrc_ook_packet *h_packets, size_t cap, size_t *n_packets)
{
    LRC_REQUIRE(o && n_packets, LRC_ERR_INVALID, "lrc_ook_fetch_packets: null argument");
    LRC_BIND(o->ctx);
    LRC_CUDA(cudaDeviceSynchronize());
    const size_t ns = o->n_streams;
    std::vector<uint32_t> np(ns * 2), ntr(ns), nb(ns);
    LRC_CUDA(cudaMemcpy(np.data(), o->d_npackets, np.size() * 4, cudaMemcpyDeviceToHost));
    LRC_CUDA(cudaMemcpy(ntr.data(), o->d_ntrans, ns * 4, cudaMemcpyDeviceToHost));
    LRC_CUDA(cudaMemcpy(nb.data(), o->d_nbursts, ns * 4, cudaMemcpyDeviceToHost));
    size_t total = 0;
    for (size_t s = 0; s < ns; ++s) {
        if (ntr[s] > o->max_runs || np[2 * s] > o->max_packets || np[2 * s + 1] > o->max_packets || nb[s] > o->max_bursts) {
            lrc_set_error("lrc_ook_fetch_packets: stream %zu overflowed (runs %u/%zu, packets %u,%u/%zu, bursts %u/%zu)",
                          s, ntr[s], o->max_runs, np[2 * s], np[2 * s + 1], o->max_packets, nb[s], o->max_bursts);
            *n_packets = 0;
            return LRC_ERR_CAPACITY;
        }
        total += np[2 * s] + np[2 * s + 1];
    }
    *n_packets = total;
    if (total == 0) return LRC_OK;
    if (cap < total || !h_packets) {
        lrc_set_error("lrc_ook_fetch_packets: %zu packets, capacity %zu", total, cap);
        return LRC_ERR_CAPACITY;
    }
    std::vector<unsigned long long> pk(ns * 2 * o->max_packets);
    LRC_CUDA(cudaMemcpy(pk.data(), o->d_packets, pk.size() * 8, cudaMemcpyDeviceToHost));
    const uint32_t seq0[2] = {0, 0};
    for (size_t s = 0; s < ns; ++s) h_packets = ook_put_packets(h_packets, pk.data(), o->max_packets, s, &np[2 * s], seq0);
    return LRC_OK;
}

extern "C" int lrc_ook_debug_ptrs(lrc_ook *o, const float **d_block_sums, const uint32_t **d_run_counts,
                                  const uint32_t **d_runs, const uint32_t **d_n_bits)
{
    LRC_REQUIRE(o != nullptr, LRC_ERR_INVALID, "null plan");
    if (d_block_sums) *d_block_sums = o->d_sum;
    if (d_run_counts) *d_run_counts = o->d_ntrans;
    if (d_runs) *d_runs = o->d_runs_dbg;
    if (d_n_bits) *d_n_bits = o->d_nbits;
    return LRC_OK;
}

// ---- streaming plan --------------------------------------------------------------------------------------------------------------
struct lrc_ook_stream {
    lrc_ook  *o;                      // the chain's buffers, sized for max_push_blocks; its d_mask / d_bsum / d_binfo rows start
                                      // with cpitch carry slots
    size_t    max_carry, max_packets;
    DevBuf<OokSeam>  d_seam;          // [n_streams]
    DevBuf<uint8_t>  d_carry;         // [n_streams][cpitch][1024] the open burst's collected blocks
    DevBuf<float>    d_cmax;          // [n_streams][cpitch] their maxima
    DevBuf<uint32_t> d_live;          // [n_streams] carried blocks sliced in the current push
    DevBuf<uint32_t> d_pbase;         // [n_streams][2] sequence number of the first packet not fetched yet
    size_t    last_push;              // blocks per stream of the last push (the debug block sums' row length)
    bool      failed;                 // a fetch reported an overflow: every call fails until reset
};

extern "C" int lrc_ook_stream_reset(lrc_ook_stream *st)
{
    LRC_REQUIRE(st != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(st->o->ctx);
    const size_t ns = st->o->n_streams;
    std::vector<OokSeam> z(ns, ook_seam_initial());
    LRC_CUDA(cudaDeviceSynchronize());
    LRC_CUDA(cudaMemcpy(st->d_seam, z.data(), ns * sizeof(OokSeam), cudaMemcpyHostToDevice));
    LRC_CUDA(cudaMemset(st->d_pbase, 0, ns * 2 * sizeof(uint32_t)));
    st->failed = false;
    st->last_push = 0;
    return LRC_OK;
}

extern "C" int lrc_ook_stream_destroy(lrc_ook_stream *st)
{
    if (!st) return LRC_OK;
    cudaSetDevice(st->o->ctx->device);
    lrc_ook_destroy(st->o);
    delete st;
    return LRC_OK;
}

extern "C" int lrc_ook_stream_create(lrc_ctx *ctx, size_t n_streams, size_t max_push_blocks, unsigned sample_rate,
                                     size_t max_carry_blocks, size_t max_runs_per_push, size_t max_packets_per_fetch,
                                     lrc_ook_stream **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && n_streams >= 1 && max_push_blocks >= 1 && sample_rate >= 1, LRC_ERR_INVALID,
                "lrc_ook_stream_create: bad arguments");
    // an open burst never holds more than guard + 1 blocks (bitfount.rs:52-54): the buffer is reset before a block is pushed once it
    // exceeds the guard, so it ends at most one block past it, plus one more when it did not start with the 0.0.  That carry is
    // exact for every input; a smaller one is the caller's memory choice, and a burst that outgrows it is reported.
    const size_t max_carry = max_carry_blocks ? max_carry_blocks : ook_guard_blocks() + 1;
    const size_t cpitch = (max_carry + 31) / 32 * 32;
    lrc_ook_stream *st = new (std::nothrow) lrc_ook_stream();
    LRC_REQUIRE(st != nullptr, LRC_ERR_NOMEM, "out of host memory");
    const int rc = ook_create(ctx, n_streams, max_push_blocks, cpitch, sample_rate, max_runs_per_push, max_packets_per_fetch, &st->o);
    if (rc != LRC_OK) { delete st; return rc; }
    st->max_carry = max_carry;
    st->max_packets = st->o->max_packets;
    cudaError_t e = st->d_seam.alloc(n_streams);
    if (e == cudaSuccess) e = st->d_carry.alloc(n_streams * cpitch * (size_t)(OOK_BLOCK * 2));
    if (e == cudaSuccess) e = st->d_cmax.alloc(n_streams * cpitch);
    if (e == cudaSuccess) e = st->d_live.alloc(n_streams);
    if (e == cudaSuccess) e = st->d_pbase.alloc(n_streams * 2);
    if (e != cudaSuccess) {
        lrc_set_error("lrc_ook_stream_create: %s (carry of %zu blocks x %zu streams)", cudaGetErrorString(e), max_carry, n_streams);
        lrc_ook_stream_destroy(st);
        return e == cudaErrorMemoryAllocation ? LRC_ERR_NOMEM : LRC_ERR_CUDA;
    }
    const int r2 = lrc_ook_stream_reset(st);
    if (r2 != LRC_OK) { lrc_ook_stream_destroy(st); return r2; }
    *out = st;
    return LRC_OK;
}

extern "C" int lrc_ook_stream_push(lrc_ook_stream *st, const uint8_t *d_iq, size_t n_blocks, size_t stream_stride_bytes, void *stream)
{
    LRC_REQUIRE(st != nullptr, LRC_ERR_INVALID, "null plan");
    lrc_ook *o = st->o;
    LRC_BIND(o->ctx);
    LRC_REQUIRE(!st->failed, LRC_ERR_CAPACITY, "lrc_ook_stream_push: the plan overflowed (see the fetch that reported it); reset it");
    LRC_REQUIRE(d_iq != nullptr, LRC_ERR_INVALID, "lrc_ook_stream_push: null input");
    LRC_REQUIRE(n_blocks >= 1 && n_blocks <= o->n_blocks, LRC_ERR_INVALID, "lrc_ook_stream_push: n_blocks outside 1..max_push_blocks");
    LRC_REQUIRE(stream_stride_bytes >= n_blocks * (size_t)OOK_BLOCK * 2, LRC_ERR_INVALID, "lrc_ook_stream_push: stride too short");
    LRC_REQUIRE(((uintptr_t)d_iq & 15) == 0 && (stream_stride_bytes & 15) == 0, LRC_ERR_INVALID,
                "lrc_ook_stream_push: input and stream stride must be 16-byte aligned");
    OokStreamLaunch sl;
    sl.seam = st->d_seam;
    sl.carry = OokCarry{o->cpitch, st->d_carry, st->d_cmax, st->d_live};
    sl.d_carry = st->d_carry; sl.d_cmax = st->d_cmax; sl.d_live = st->d_live; sl.d_pbase = st->d_pbase;
    sl.max_carry = st->max_carry;
    const int rc = ook_launch<true>(o, d_iq, n_blocks, stream_stride_bytes, lrc_stream(o->ctx, stream), &sl);
    if (rc == LRC_OK) st->last_push = n_blocks;
    return rc;
}

extern "C" int lrc_ook_stream_fetch_packets(lrc_ook_stream *st, lrc_ook_packet *h_packets, size_t cap, size_t *n_packets)
{
    LRC_REQUIRE(st && n_packets, LRC_ERR_INVALID, "lrc_ook_stream_fetch_packets: null argument");
    lrc_ook *o = st->o;
    LRC_BIND(o->ctx);
    *n_packets = 0;
    LRC_REQUIRE(!st->failed, LRC_ERR_CAPACITY, "lrc_ook_stream_fetch_packets: the plan overflowed earlier; reset it");
    LRC_CUDA(cudaDeviceSynchronize());
    const size_t ns = o->n_streams, mp = st->max_packets;
    std::vector<OokSeam> z(ns);
    std::vector<uint32_t> base(ns * 2);
    LRC_CUDA(cudaMemcpy(z.data(), st->d_seam, ns * sizeof(OokSeam), cudaMemcpyDeviceToHost));
    LRC_CUDA(cudaMemcpy(base.data(), st->d_pbase, ns * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    size_t total = 0;
    for (size_t s = 0; s < ns; ++s) {
        const uint32_t na = z[s].m_count[0] - base[2 * s], nb = z[s].m_count[1] - base[2 * s + 1];
        if (z[s].err || na > mp || nb > mp) {
            st->failed = true;
            lrc_set_error("lrc_ook_stream_fetch_packets: stream %zu overflowed:%s%s%s%s (carry %zu blocks, runs per push %zu, bursts per "
                          "push %zu, packets per fetch %zu); the plan fails until reset", s,
                          (z[s].err & OOK_ERR_CARRY) ? " its open burst outgrew max_carry_blocks" : "",
                          (z[s].err & OOK_ERR_RUNS) ? " runs" : "", (z[s].err & OOK_ERR_BURSTS) ? " bursts" : "",
                          (na > mp || nb > mp) ? " packets" : "", st->max_carry, o->max_runs, o->max_bursts, mp);
            return LRC_ERR_CAPACITY;
        }
        total += na + nb;
    }
    *n_packets = total;
    if (total == 0) return LRC_OK;
    if (cap < total || !h_packets) {
        lrc_set_error("lrc_ook_stream_fetch_packets: %zu packets, capacity %zu", total, cap);
        return LRC_ERR_CAPACITY;
    }
    std::vector<unsigned long long> pk(ns * 2 * mp);
    LRC_CUDA(cudaMemcpy(pk.data(), o->d_packets, pk.size() * 8, cudaMemcpyDeviceToHost));
    for (size_t s = 0; s < ns; ++s) {
        const uint32_t n[2] = {z[s].m_count[0] - base[2 * s], z[s].m_count[1] - base[2 * s + 1]};
        h_packets = ook_put_packets(h_packets, pk.data(), mp, s, n, &base[2 * s]);
    }
    for (size_t s = 0; s < ns; ++s) { base[2 * s] = z[s].m_count[0]; base[2 * s + 1] = z[s].m_count[1]; }
    LRC_CUDA(cudaMemcpy(st->d_pbase, base.data(), ns * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return LRC_OK;
}

extern "C" int lrc_ook_stream_debug_ptrs(lrc_ook_stream *st, const float **d_block_sums, const uint32_t **d_run_counts,
                                         const uint32_t **d_runs, const uint32_t **d_n_bits)
{
    LRC_REQUIRE(st != nullptr, LRC_ERR_INVALID, "null plan");
    return lrc_ook_debug_ptrs(st->o, d_block_sums, d_run_counts, d_runs, d_n_bits);
}

extern "C" int lrc_eat(const uint8_t *bits, size_t nbits, const size_t *widths, size_t n_widths, size_t *out)
{
    // kpn::eat / kpn::b2d (kpn.rs:111-124): consecutive MSB-first fields
    LRC_REQUIRE(bits && widths && out, LRC_ERR_INVALID, "lrc_eat: null argument");
    size_t i = 0;
    for (size_t w = 0; w < n_widths; ++w) {
        if (i + widths[w] > nbits) {
            lrc_set_error("lrc_eat: fields need %zu bits, packet has %zu (the reference slices out of bounds and panics)",
                          i + widths[w], nbits);
            return LRC_ERR_LENGTH;
        }
        size_t v = 0;
        for (size_t k = 0; k < widths[w]; ++k) v += ((size_t)1 << (widths[w] - k - 1)) * bits[i + k];
        out[w] = v;
        i += widths[w];
    }
    return LRC_OK;
}

extern "C" int lrc_ook_envelope_table(lrc_ctx *ctx, float *d_table, void *stream)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(d_table != nullptr, LRC_ERR_INVALID, "lrc_ook_envelope_table: null output");
    ook_envelope_table_kernel<<<256, 256, 0, lrc_stream(ctx, stream)>>>(d_table);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}
