#!/bin/bash
# Developer tool (GPU box): tree-softmax parity tests + where the yolo9000 step goes (launch list of the tail).
python -m pytest tests/test_golden_gpu.py tests/test_network_gpu.py -q -x -k "decode_nms or toy or yolo9000" 2>&1 | tail -3
timeout 200 python tools/throughput.py yolo9000 544 16 --layers 2>&1 | tail -3
ncu --metrics gpu__time_duration.sum --clock-control none -c 60 --csv --log-file gpurun_out/y9k_launches.csv python tools/throughput.py yolo9000 544 16 1 > /dev/null 2>&1
python - <<PY
import csv
rows=[r for r in csv.reader(open("gpurun_out/y9k_launches.csv")) if len(r)>8]
hdr=rows[0]; ix={h:i for i,h in enumerate(hdr)}
seq=[(r[ix["Kernel Name"]][:60], float(r[ix["Metric Value"]])/1000) for r in rows[1:] if r[ix["Metric Name"]]=="gpu__time_duration.sum"]
for k,v in seq[-14:]: print(f"{k:60s} {v:10.1f}")
PY
