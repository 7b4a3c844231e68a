// fastfir.cuh -- what the overlap-save plan (k_fastfir.cu) and its 16384-point kernel (k_fastfir16k.cu) share.
#pragma once
#include "common.cuh"

// What a STREAM instance of an overlap-save kernel reads besides the batch arguments.  A work item is (channel c, block b)
// flattened channel-major, item = c * nblk + b.  Channel c's row is [carried history | new chunk] read in place: row
// index v is carry[c * carry_pitch + v] for v < held and in[c * in_stride + v - held] after; n_in is the row length
// held + n, the same for every channel.  Block b of channel c writes out[c * out_stride + b * ngood ..].
// step_c, step_b: gridDim.x = step_c * nblk + step_b (filled by the launch), so a CTA steps from item to item without a
// division.
struct FfStreamArgs {
    const float2 *carry;
    size_t carry_pitch, held, in_stride, out_stride, nblk, step_c, step_b;
};

void lrc_fastfir16k_permute_H(const float2 *H, float2 *Hq);
int lrc_fastfir16k_prepare(void);
// sa == nullptr: one channel, item = block (the batch kernel); otherwise the stream kernel over sa->nblk blocks per channel
int lrc_fastfir16k_launch(int n_sm, const float2 *in, size_t n_in, float2 *out, size_t full, size_t nblk, size_t ngood,
                          size_t keep, const float2 *d_tw16k, const float2 *d_tw1k, const float2 *d_Hp,
                          const FfStreamArgs *sa, cudaStream_t s);
