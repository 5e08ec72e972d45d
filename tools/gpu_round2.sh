#!/bin/bash
# Round-2 profiling visit: launch list + DRAM traffic of one eager UNet call, then shape-LABELLED full ncu captures of every
# kernel class (one tools/one_op.py command per capture; each ncu run is preceded by the same command without ncu).
mkdir -p gpurun_out
rm -f gpurun_out/*.ncu-rep
python tools/profile_unet.py --batch 8 > gpurun_out/prof_plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv \
    --log-file gpurun_out/launches_unet_b8.csv python tools/profile_unet.py --batch 8 > gpurun_out/prof_ncu.log 2>&1
echo "ncu launches rc=$?"
ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --profile-from-start off -k regex:tc_contract --csv \
    --log-file gpurun_out/traffic_tc_unet_b8.csv python tools/profile_unet.py --batch 8 > gpurun_out/prof_traffic.log 2>&1
echo "ncu traffic rc=$?"
cap() {   # cap <label> <kernel regex> <one_op args...>
  local label=$1 regex=$2; shift 2
  python tools/one_op.py "$@" > gpurun_out/cap_$label.plain.log 2>&1 && \
  ncu --set full --clock-control none --import-source on -k regex:$regex -s 6 -c 1 -f -o gpurun_out/cap_$label \
      python tools/one_op.py "$@" > gpurun_out/cap_$label.ncu.log 2>&1
  local rc=$?
  # the reports do not travel (64 MiB limit on gpurun_out): export the raw metrics page (and, for the kernels listed in $HOT, the
  # hottest SASS instructions with their stall reasons) here on the box, then drop the report
  if [ -f gpurun_out/cap_$label.ncu-rep ]; then
    ncu -i gpurun_out/cap_$label.ncu-rep --page raw --csv > gpurun_out/cap_$label.raw.csv 2>/dev/null
    case " $HOT " in *" $label "*)
      ncu -i gpurun_out/cap_$label.ncu-rep --page source --print-source sass --csv > gpurun_out/cap_$label.src.csv 2>/dev/null
      python tools/ncu_hot.py gpurun_out/cap_$label.src.csv 45 > gpurun_out/cap_$label.hot.txt 2>&1
      rm -f gpurun_out/cap_$label.src.csv;;
    esac
    rm -f gpurun_out/cap_$label.ncu-rep
  fi
  echo "cap $label rc=$rc :: $(tail -1 gpurun_out/cap_$label.plain.log)"
}
HOT="pair160_f32res_M32768_N320_K320 single160_f32res_M32768_N320_K320 pair256_geglu_M32768_N2560_K320 attn_d40_S4096 attn_d40_S4096_Sk77 attn_wide_d512_S4096 pair128_conv3x3_128_512x512_res"
cap pair256_geglu_M32768_N2560_K320        tc_contract_pair gemm 32768 2560 320 0 1 2 256 1
cap pair256_bf16out_M32768_N960_K320       tc_contract_pair gemm 32768 960 320 0 1 2 256 0
cap pair160_f32res_M2048_N1280_K1280       tc_contract_pair gemm 2048 1280 1280 1 0 2 160 0
cap pair160_f32res_M32768_N320_K320        tc_contract_pair gemm 32768 320 320 1 0 2 160 0
cap single160_f32res_M32768_N320_K320      tc_contract_kernel gemm 32768 320 320 1 0 1 160 0
cap single160_conv3x3_320_64x64_res        tc_contract_kernel conv 8 64 64 320 320 3 1 1 1 160
cap pair256_conv3x3_1280_16x16_res         tc_contract_pair conv 8 16 16 1280 1280 3 1 1 2 256
cap pair128_conv3x3_128_512x512_res        tc_contract_pair conv 2 512 512 128 128 3 1 1 2 128
cap splitk_conv3x3_1280_8x8                splitk_reduce conv 8 8 8 1280 1280 3 1 1 2 256
cap attn_d40_S4096                         tc_attention_kernel attn 8 8 4096 4096 40
cap attn_d80_S1024                         tc_attention_kernel attn 8 8 1024 1024 80
cap attn_d160_S256                         tc_attention_kernel attn 8 8 256 256 160
cap attn_d40_S4096_Sk77                    tc_attention_kv1 attn 8 8 4096 77 40
cap attn_d80_S1024_Sk77                    tc_attention_kv1 attn 8 8 1024 77 80
cap attn_wide_d512_S4096                   tc_attention_wide attnw 8 4096 4096 512
cap gn_cluster_N8_HW4096_C320              gn_ gn 8 4096 320 1
cap layernorm_rows32768_C320               layernorm_kernel ln 32768 320
cap ddim_step_n131072                      sampler_update_kernel ddim 131072
ls gpurun_out/*.raw.csv | wc -l; du -sh gpurun_out
