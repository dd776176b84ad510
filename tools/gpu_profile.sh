#!/usr/bin/env bash
# Run on the GPU box (under gpurun): bench line + ncu launch list + two `ncu --set full` captures
# (cache flushed = ncu default, and --cache-control none = live L2 behaviour) of one step's kernels.
#   tools/gpu_profile.sh <tag> [extra bench args]
set -uo pipefail
TAG=${1:-run}; shift || true
OUT=gpurun_out
mkdir -p $OUT
KREG='regex:gemm_img|gemm_chain|token_fused|sig_attention|match_tc|match_tail|match_exact|desc_tiles'
python bench.py "$@" > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench rc=$?"; tail -c 600 $OUT/${TAG}_bench.json
ncu --metrics gpu__time_duration.sum --clock-control none -k 'regex:gemm_|token_fused|sig_attention|match_|desc_tiles|small_mlp|final_norm|argmin|mutual|segmean|dist_kernel|gather_wait' -s 23 -c 46 --csv \
    --log-file $OUT/${TAG}_launches.csv python bench.py --profile-only --steps 1 --warmup 1 "$@" > /dev/null 2>&1; echo "launch list rc=$?"
# the .ncu-rep files of 22 launches are ~40 MB each (the output directory is capped at 64 MiB): keep the raw-page CSV of both
# captures (what tools/ncu_summary.py reads) and, as a binary report, only a 4-launch capture with source correlation
TMP=/tmp/ncu_$TAG; mkdir -p $TMP
ncu --set full --clock-control none -k "$KREG" -s 22 -c 22 -f -o $TMP/full_flush \
    python bench.py --profile-only --steps 1 --warmup 1 "$@" > $OUT/${TAG}_ncu1.log 2>&1; echo "ncu flush rc=$?"
ncu -i $TMP/full_flush.ncu-rep --page raw --csv > $OUT/${TAG}_full_flush_raw.csv 2>/dev/null
ncu --set full --clock-control none --cache-control none -k "$KREG" -s 22 -c 22 -f -o $TMP/full_live \
    python bench.py --profile-only --steps 1 --warmup 1 "$@" > $OUT/${TAG}_ncu2.log 2>&1; echo "ncu live rc=$?"
ncu -i $TMP/full_live.ncu-rep --page raw --csv > $OUT/${TAG}_full_live_raw.csv 2>/dev/null
# token kernel, V projection, line chain? no: first chain (fc .. qkv0), attention, layer chain of one step, with SASS/source
# (source-level capture dropped from the default run: the binary report alone is ~10 MB)

ls -la $OUT | tail -10; du -sm $OUT
