#!/bin/bash
# Regenerates tests/golden/<case>/ from the UNMODIFIED reference (oracle/_ref/ref_harness, built by oracle/Makefile from
# /root/reference). Needs a GPU: run on the B200 box, e.g.
#   gpurun --timeout 900 -- 'bash tests/golden/make_golden.sh gpurun_out/golden'
# then copy gpurun_out/golden/<case> into tests/golden/<case> and commit. The vectors are what pins oracle/oracle_cpu.cpp.
set -e
OUT=${1:-gpurun_out/golden}
H=oracle/_ref/ref_harness
C=tests/golden/configs
mkdir -p "$OUT"
# <case> <config> <n_in> <n_out> <batch> <n_steps> <jit>
$H dump $C/hash3d_small.json 3 3 512 10 "$OUT/hash3d_small" 0
$H dump $C/hash3d_small.json 3 3 512 10 "$OUT/hash3d_small_jit" 1
$H dump $C/dense_mix3d.json 3 2 256 10 "$OUT/dense_mix3d" 0
$H dump $C/image2d.json 2 3 512 10 "$OUT/image2d" 0
$H dump $C/tanh_w32.json 3 3 512 10 "$OUT/tanh_w32" 0
$H probe 1.5 16 16 > "$OUT/probe_s1.5_b16.json"
$H probe 2.0 16 16 > "$OUT/probe_s2.0_b16.json"
$H probe 1.5 4 8 > "$OUT/probe_s1.5_b4.json"
$H probe 1.3819 16 16 > "$OUT/probe_s1.3819_b16.json"
# Benchmarked size (T = 2^19; B = 2^16 and 2^18), sub-sampled: <stride over grid parameters> <n_head samples of per-sample arrays>
$H dumpbig $C/headline.json 3 3 65536 10 "$OUT/big_headline_b16" 0 509 2048
$H dumpbig $C/headline.json 3 3 262144 10 "$OUT/big_headline_b18" 0 509 2048
# BASELINE.json configs[0]: CutlassMLP 64 x 2 behind the Identity encoding
$H dump $C/identity_cutlass.json 3 3 512 10 "$OUT/identity_cutlass" 0
# Composite / parameter-free encodings (SURVEY.md section 8f N3): TriangleWave + OneBlob + Identity ("NRC" layout), HashGrid + SphericalHarmonics
# (the NeRF-style position + direction input), Frequency on its own
$H dump $C/composite_nrc.json 6 3 512 10 "$OUT/composite_nrc" 0
$H dump $C/composite_grid_sh.json 6 3 512 10 "$OUT/composite_grid_sh" 0
$H dump $C/frequency_top.json 3 3 512 10 "$OUT/frequency_top" 0
# Trainer::serialize() snapshots (msgpack), without and with the optimizer state, at initialisation and after 20 steps; a small
# model keeps the fixture small
for opt in 0 1; do
	for steps in 0 20; do
		mkdir -p "$OUT/snapshot_opt${opt}_step${steps}"
		$H snapshot save $C/snapshot_small.json 3 3 1024 $steps "$OUT/snapshot_opt${opt}_step${steps}" $opt > "$OUT/snapshot_opt${opt}_step${steps}/save.json"
	done
done
