#!/bin/bash
# The grid sweeps behind profiles/r1_s8_grid_sweeps.txt and the scalar resampler of r1_s8_rs_configs.txt (every knob is
# read once per process, so each point is its own interpreter).  Run from the repository root on a B200; about 3 minutes.
set -u
O=gpurun_out; mkdir -p $O; export PYTHONUNBUFFERED=1
out=$O/sweeps.txt; : > $out
run() { only=$1; shift; echo "$*" | tee -a $out; env "$@" timeout 150 python tools/bench_kernels.py --only $only 2>>$O/sweeps.err | tee -a $out | cut -c1-130; }
for c in 8 16 64 256 1024 1048576; do run unpack LRC_UNPACK_CAP=$c; done
for c in 16 32 64 128 512; do run fm LRC_FM_CAP=$c; done
for k in 1 2 4 16 32 1024; do run fir,fft,fm LRC_FFT_GRID=$k LRC_PSD_GRID=$k LRC_FIRU8_GRID=$k LRC_FIR_GRID=$k LRC_RS_GRID=$k; done
run fm,fmchain LRC_RS_VARIANT=0
