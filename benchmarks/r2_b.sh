#!/bin/bash
# round 2, second GPU pass: parity tests of the fused locate, C4/C2 bench lines, ncu captures on C4
tag=${1:-r2b}
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/${tag}_pytest.log 2>&1; echo "pytest exit $?"
tail -3 gpurun_out/${tag}_pytest.log
timeout 600 python bench.py --only-headline --steps 5 > gpurun_out/${tag}_c4.json 2> gpurun_out/${tag}_c4.err; echo "bench c4 exit $?"
timeout 600 python bench.py --only-headline --config C2 --steps 10 > gpurun_out/${tag}_c2.json 2> gpurun_out/${tag}_c2.err; echo "bench c2 exit $?"
python - <<'PY'
import json
for f in ("c4","c2"):
    try:
        d=json.load(open(f"gpurun_out/TAG_{f}.json".replace("TAG","'"$tag"'")))
        print(f, round(d["value"]/1e9,3), "G upd/s e2e", round(d["e2e"]["value"]/1e9,3), d["stages_ms"], round(d["roofline"]["frac"],4))
    except Exception as e: print(f, "failed", e)
PY
# launch list of C4 (cold-cache, serialised)
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -k 'regex:^k_' -c 400 --csv \
    --log-file gpurun_out/${tag}_c4_launches.csv python bench.py --only-headline --steps 2 --warmup 1 --e2e-steps 1 \
    > gpurun_out/${tag}_c4_launches.log 2>&1; echo "ncu launches exit $?"
# full capture of the hot kernels of the warm-up batch (the core load launches 6 passes + locate + rebalance first)
timeout 1200 ncu --set full --clock-control none --import-source on \
    -k 'regex:^(k_rebalance_m|k_os_pass|k_locate)$' --launch-skip 8 -c 8 \
    -f -o gpurun_out/${tag}_c4_full python bench.py --only-headline --steps 1 --warmup 1 --e2e-steps 1 \
    > gpurun_out/${tag}_c4_full.log 2>&1; echo "ncu full exit $?"
ls -la gpurun_out/${tag}_*
