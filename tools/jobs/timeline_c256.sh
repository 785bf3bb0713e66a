#!/bin/bash
cd "$(dirname "$0")/../.."
mkdir -p gpurun_out
python tools/step_timeline.py 32 4 celeba256 > gpurun_out/r2_step_timeline_celeba256.txt 2>&1
head -30 gpurun_out/r2_step_timeline_celeba256.txt
python tools/step_timeline.py 128 6 low64 > gpurun_out/r2_step_timeline_low64.txt 2>&1
head -12 gpurun_out/r2_step_timeline_low64.txt
