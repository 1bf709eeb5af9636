#!/bin/bash
# Round evidence in one GPU session: parity suite (incl. the BASELINE-size cases), bench lines (ours + reference arm),
# per-op table, ncu launch lists and --set full captures of the headline, decode and merge kernels, pipeline wait
# breakdown.  Outputs land in gpurun_out/<tag>_*; summarise with profiles/ncu_*.py / tools/stamp_traffic.py and copy
# what is judged into profiles/.
tag=${1:-r2}
o=gpurun_out; mkdir -p $o
timeout 900 python -m pytest tests -m gpu -q --durations=8 > $o/${tag}_tests.log 2>&1; tail -2 $o/${tag}_tests.log
timeout 300 python bench.py --impl reference --steps 5 --warmup 2 > $o/${tag}_bench_ref.json 2> $o/${tag}_bench_ref.err; tail -c 300 $o/${tag}_bench_ref.json; echo
timeout 400 python bench.py > $o/${tag}_bench.json 2> $o/${tag}_bench.err; tail -c 400 $o/${tag}_bench.json; echo
timeout 600 python tools/bench_ops.py --out $o/${tag}_ops.json > $o/${tag}_ops.log 2>&1; tail -2 $o/${tag}_ops.log | cut -c1-300
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $o/${tag}_bench_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-e2e --no-ops --no-dense > $o/${tag}_ncu_bench.log 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:filter_pipe_kernel -s 3 -c 1 -f -o $o/${tag}_pipe \
    python bench.py --steps 3 --warmup 3 --no-e2e --no-ops --no-dense > $o/${tag}_ncu_pipe.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:mmerge3_kernel -s 1 -c 1 -f -o $o/${tag}_mmerge \
    python tools/prof_merge.py 100000000 > $o/${tag}_ncu_merge.log 2>&1
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k 'regex:^(msample|mplan2|mmerge3|mscan|mcompact|merge)_kernel' -c 60 --csv --log-file $o/${tag}_merge_launches.csv \
    python tools/prof_merge.py 100000000 > $o/${tag}_ncu_merge2.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:decode_kernel -s 1 -c 1 -f -o $o/${tag}_decode \
    python tools/prof_decode.py > $o/${tag}_ncu_decode.log 2>&1
for w in c2 c1; do
  WORKLOAD=$w PAIRS=1024 DGX_LIB=$PWD/dgraph_b200/libdgx_prof.so timeout 150 python tools/prof_pipe_waits.py > $o/${tag}_pipe_waits_$w.json 2>> $o/${tag}_pw.err
done
ls -la $o | grep ${tag}_ | awk '{print $5, $9}'
