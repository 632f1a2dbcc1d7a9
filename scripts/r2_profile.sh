#!/bin/bash
# GPU evidence pass of round 2: in-graph timeline, ncu --set full of the decode kernels, format table.  Outputs -> $OUT
# (default build/r2_profile/, git-ignored; the .ncu-rep files are exported to CSV and removed to keep the directory small)
OUT=${OUT:-build/r2_profile}
mkdir -p $OUT
TIMELINE=2000 TL_ROWS=70 timeout 300 python scripts/probe_model.py "dict()" > $OUT/r2_timeline_q8_0.log 2>&1
WTYPE=q4_0 TIMELINE=2000 TL_ROWS=70 timeout 300 python scripts/probe_model.py > $OUT/r2_timeline_q4_0.log 2>&1
for spec in "q8_0 4096 14336 2 1 w13" "q8_0 14336 4096 1 0 w2" "q4_0 4096 14336 2 1 w13"; do
  set -- $spec
  timeout 200 python scripts/kernel_only.py $1 $2 $3 $4 $5 > $OUT/r2_kernel_$1_$6.txt 2>&1 && \
  timeout 300 ncu --set full --clock-control none --import-source on -k regex:matvec_idp -s 12 -c 1 -f -o /tmp/r2_ncu_$1_$6 python scripts/kernel_only.py $1 $2 $3 $4 $5 > $OUT/r2_ncu_$1_$6.log 2>&1
  ncu -i /tmp/r2_ncu_$1_$6.ncu-rep --page raw --csv > $OUT/r2_ncu_$1_$6_raw.csv 2>/dev/null
  ncu -i /tmp/r2_ncu_$1_$6.ncu-rep --page source --csv > $OUT/r2_ncu_$1_$6_source.csv 2>/dev/null
  ncu -i /tmp/r2_ncu_$1_$6.ncu-rep --page details > $OUT/r2_ncu_$1_$6_details.txt 2>/dev/null
done
timeout 600 python scripts/format_table.py f16 bf16 f8_e4m3 q8_0 q5_1 q5_0 q4_1 q4_0 > $OUT/r2_format_table.md 2>&1
du -sh $OUT
tail -3 $OUT/r2_format_table.md
