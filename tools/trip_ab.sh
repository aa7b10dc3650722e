#!/bin/bash
# Alternating A/B of the shipped library against tuning variants: ROUNDS x (base, each variant), kernel-table rows matching $ONLY
# Build variant <v> from cvsteer_b200/csrc with: make OBJDIR=build/var_<v> OUT=../variants/libcvsteer_b200_<v>.so EXTRA="-D..."
ONLY=${ONLY:-M2}; SIZES=${SIZES:-1080p,4k}; ROUNDS=${ROUNDS:-3}; ITERS=${ITERS:-100}
for i in $(seq $ROUNDS); do for v in base $VARIANTS; do
  if [ $v = base ]; then unset CVS_LIB; else export CVS_LIB=$PWD/cvsteer_b200/variants/libcvsteer_b200_$v.so; fi
  echo -n "$v "; python tools/kernel_table.py --only "$ONLY" --sizes $SIZES --iters $ITERS | python -c "
import sys,json
print([(d['kernel'],d['size'],d['Gpix_s']) for d in map(json.loads,sys.stdin)])"
done; done
