# ncu --set full captures of the kernels bench.py reports, one launch each, at the shapes of its `roofline` block.
# Report names follow <round>__<bench kernel>__<bench shape key>.ncu-rep: tools/ncu_summary.py turns them into
# profiles/r02b_ncu_summary.json, where bench.py's `ncu_traffic` finds `roofline.traffic` by (kernel, key).
set -x
N="ncu --set full --clock-control none --import-source on -f"
M="python -m guided_attention_b200.microbench"
O=gpurun_out/ncu
mkdir -p $O
timeout 300 $N -k "regex:cross_attn_fwd_tc_(pipe|stream)" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_fwd__N1024_d80_mapsTrue $M --single fwd 256 1024 80 maps > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k "regex:cross_attn_fwd_tc_(pipe|stream)" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_fwd__N256_d160_mapsTrue $M --single fwd 512 256 160 maps > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k "regex:cross_attn_fwd_tc_(pipe|stream)" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_fwd__N4096_d40_mapsFalse $M --single fwd 128 4096 40 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k "regex:cross_attn_bwd_tc_stream" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_bwd__N1024_d80_mapsTrue $M --single bwd 256 1024 80 maps > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k "regex:cross_attn_bwd_tc_stream" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_bwd__N256_d160_mapsTrue $M --single bwd 512 256 160 maps > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k "regex:cross_attn_bwd_tc_stream" --launch-skip 3 --launch-count 1 -o $O/r02b__cross_attn_bwd__N4096_d40_mapsFalse $M --single bwd 128 4096 40 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:tail_fwd --launch-skip 4 --launch-count 2 -o $O/r02b__guidance_tail_fwd__res16 $M --single-tail fwd 16 2048 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:tail_bwd --launch-skip 3 --launch-count 1 -o $O/r02b__guidance_tail_bwd__res16 $M --single-tail bwd 16 2048 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:tail_fwd --launch-skip 4 --launch-count 2 -o $O/r02b__guidance_tail_fwd__res32 $M --single-tail fwd 32 512 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:tail_bwd --launch-skip 3 --launch-count 1 -o $O/r02b__guidance_tail_bwd__res32 $M --single-tail bwd 32 512 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:self_attn_fwd --launch-skip 3 --launch-count 1 -o $O/r02b__self_attn_fwd__B1_H8_N4096_d40 $M --single-self fwd 1 4096 40 > /dev/null 2>&1; echo rc=$?
timeout 300 $N -k regex:self_attn_bwd --launch-skip 4 --launch-count 2 -o $O/r02b__self_attn_bwd__B1_H8_N4096_d40 $M --single-self bwd 1 4096 40 > /dev/null 2>&1; echo rc=$?
ls -la $O
