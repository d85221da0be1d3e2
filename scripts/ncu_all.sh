#!/bin/bash
# `ncu --set full` capture of every kernel of the library (one launch each, the last of the workload), summaries
# into gpurun_out/ncu_<name>.txt (copied to profiles/<tag>_ncu_<name>.txt by scripts/save_profiles.sh).
# usage: scripts/ncu_all.sh [kernel-name-regex ...]
OUT=gpurun_out
mkdir -p $OUT
KERNELS=${@:-"pool_mean_kernel pool_bins_kernel pool_mean_convert_kernel softmax_rows_reg_kernel resample_kernel consolidate gemm_tf32_kernel cont_attn_tc_kernel attn_tc_combine sticky_hist_rect_kernel cont_attn_fast_kernel cont_attn_kernel sticky_hist_gauss_kernel cont_attn_g16_kernel split_half3_kernel fold_sample_columns_kernel rbf_eval_kernel gather_rows_kernel density_rect_kernel ridge"}
for k in $KERNELS; do
  which=rect
  case $k in sticky_hist_gauss*|rbf_eval*|gather_rows*|ridge*|cont_attn_g16*|split_half3*|fold_sample*) which=gauss;; pool_bins*) which=bins;;
            pool_mean_convert*|softmax_rows*) which=caller;; esac
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:$k -c 3 -f -o $OUT/prof_$k \
      python scripts/ncu_workload.py $which > $OUT/ncu_$k.log 2>&1
  echo "$k rc=$?" >> $OUT/summary.txt
done
