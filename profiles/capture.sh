#!/bin/bash
# Run on the B200 box (gpurun): captures the ncu evidence bench.py's numbers are read against and summarises it.
#   bash profiles/capture.sh <tag> ["steps"]     steps: any of 1 2 3 4 (default all)
# Raw captures (.ncu-rep, launch-list CSVs: tens of MB) go to $RAW (default /tmp/ppd_cap, outside gpurun_out/, which
# only carries 64 MiB back); profiles/summarize.py then writes the small text / JSON summaries to gpurun_out/profiles_<tag>/,
# from where they are copied into profiles/.  Every ncu pass runs AFTER the same command has exited 0 without ncu.
set -u
TAG=${1:-r01}
STEPS=${2:-"1 2 3 4"}
RAW=${RAW:-/tmp/ppd_cap}
mkdir -p $RAW gpurun_out/profiles_$TAG
has() { [[ " $STEPS " == *" $1 "* ]]; }
LIST="--metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --csv"
if has 1; then
  # 1. launch list of the bench command (all kernels, serialised by ncu: shares, not absolutes)
  B="python bench.py --steps 2 --warmup 3 --no-sweep"
  $B > $RAW/${TAG}_bench_plain.log 2> $RAW/${TAG}_bench_plain.err || { echo "plain bench failed"; exit 1; }
  ncu $LIST -c 4000 --log-file $RAW/${TAG}_launches_c2.csv $B > $RAW/${TAG}_ncu_c2.log 2>&1
fi
if has 2; then
  # 2. full capture of the dominant kernel: one block per step so that the launch order is known
  #    (17 level launches per decode / replay; skip 3 warm-up decodes + 3 warm-up replays)
  B1="python bench.py --steps 1 --warmup 3 --no-sweep --blocks-per-step 1"
  PPD_HOST_THREADS=1 $B1 > /dev/null 2>&1 && PPD_HOST_THREADS=1 ncu --set full --clock-control none --import-source on -k regex:hash_level_kernel \
      --launch-skip 102 --launch-count 17 -o $RAW/${TAG}_hash_level_full $B1 > $RAW/${TAG}_ncu_full.log 2>&1
fi
if has 3; then
  # 3. config 5 (sorted leaves, 10M): launch list + full capture of the two hashing kernels
  C5="python profiles/run_c5.py 10000000 1"
  $C5 > $RAW/${TAG}_c5_plain.log 2>&1 && ncu $LIST -c 400 --log-file $RAW/${TAG}_launches_c5.csv $C5 > /dev/null 2>&1
  ncu --set full --clock-control none --import-source on -k regex:hash_ -c 14 -o $RAW/${TAG}_c5_full $C5 > $RAW/${TAG}_ncu_c5_full.log 2>&1
fi
if has 4; then
  # 4. the witness parse / arena kernels (ppd_parse.cu) on one config-2 block: plain run, launch list, and a full
  #    capture of the second (warm) decode's parse kernels
  PR="python profiles/run_parse.py"
  $PR 5 > $RAW/${TAG}_parse_plain.log 2> $RAW/${TAG}_parse_plain.err && ncu $LIST -c 2000 --log-file $RAW/${TAG}_launches_parse.csv $PR 2 > /dev/null 2>&1
  K="regex:tile_exit|group_exit|top_chain|tile_entry|tile_mark|ins_scatter|ins_info|heights_kernel|min64_i16|link_kernel16|shape_kernel|scan_block_kernel|scan_add_kernel|^emit_kernel|climb_kernel|code_list|totals_kernel"
  N=$(python profiles/summarize.py --count-parse-kernels $RAW/${TAG}_launches_parse.csv)
  ncu --set full --clock-control none --import-source on -k "$K" --launch-skip $N --launch-count $N -o $RAW/${TAG}_parse_full $PR 2 > $RAW/${TAG}_ncu_parse_full.log 2>&1
fi
SRC=$RAW DST=gpurun_out/profiles_$TAG python profiles/summarize.py $TAG
ls -la gpurun_out/profiles_$TAG
