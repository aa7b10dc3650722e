#!/bin/bash
# A/B of tuning variants (cvsteer_b200/variants/*.so): kernel table rows selected by $ONLY for the shipped library and each variant
# Build variant <v> from cvsteer_b200/csrc with: make OBJDIR=build/var_<v> OUT=../variants/libcvsteer_b200_<v>.so EXTRA="-D..."
mkdir -p gpurun_out
ONLY=${ONLY:-g4}
SIZES=${SIZES:-4k}
for v in base $VARIANTS; do
  if [ $v = base ]; then unset CVS_LIB; else export CVS_LIB=$PWD/cvsteer_b200/variants/libcvsteer_b200_$v.so; fi
  timeout 300 python tools/kernel_table.py --only $ONLY --sizes $SIZES --iters 30 > gpurun_out/var_$v.jsonl 2> gpurun_out/var_$v.err
  timeout 300 python tools/kernel_table.py --only $ONLY --sizes $SIZES --iters 30 >> gpurun_out/var_$v.jsonl 2>> gpurun_out/var_$v.err
done
python - <<'PY'
import json,glob,collections
t=collections.defaultdict(dict)
for f in sorted(glob.glob("gpurun_out/var_*.jsonl")):
    v=f.split("var_")[1][:-6]
    for l in open(f):
        try:d=json.loads(l)
        except Exception: continue
        if "Gpix_s" in d: t[(d["kernel"],d["size"])].setdefault(v,[]).append(d["Gpix_s"])
for k,row in t.items(): print(k, {v:[round(x,1) for x in xs] for v,xs in row.items()})
PY
