#!/bin/bash
# round-2 session-2 check A: two-stream saves, single-stream residual (run on a B200)
O=gpurun_out; T=${1:-r03_a}
mkdir -p $O
python -m pytest tests -x -q -m gpu > $O/${T}_pytest.log 2>&1; tail -3 $O/${T}_pytest.log
python tools/dbg/mega_time.py > $O/${T}_megatime.log 2>&1; grep -E "median|epilogue R|epilogue G|mma" $O/${T}_megatime.log
CMWG_RES_LO=1 python tools/dbg/mega_time.py > $O/${T}_megatime_lo1.log 2>&1; grep -E "median" $O/${T}_megatime_lo1.log
python bench.py --no-wsrglow --no-waveflow --no-synth-sweep --no-cpu-baseline > $O/${T}_bench.json 2> $O/${T}_bench.err; T=$T python - <<'PY'
import json,os
d=json.loads(open("gpurun_out/%s_bench.json" % os.environ["T"]).read().strip().splitlines()[-1])
print({k:d[k] for k in ("value","ms_per_step")}, d["e2e"]["value"], d["roofline"]["ms_per_launch"], d["roofline"]["frac"], d["roofline"]["kernel_classes_ms_per_step"])
print(d.get("parity")); print(d["synth"]["value"], d["clocks"])
PY
