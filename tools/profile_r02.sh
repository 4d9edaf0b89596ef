#!/bin/bash
# Evidence run for profiles/ (one B200, under gpurun): ncu launch list of one prefill chunk + two decode steps, ncu --set full
# captures of every kernel of a decode step and of one prefill layer (final code), compute-sanitizer logs.
# Numbers printed by the profiled programs are NOT bench values.
set -u
O=gpurun_out; mkdir -p $O
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:'^(add_rmsnorm|argmax|decode_attn|embed_kernel|gemm_|prefill_attn|rope_|activate_rows|gather_|silu_mul|decode_layer)' -c 1200 --csv --log-file $O/r02_launches.csv \
    python tools/profile_step.py --decode-steps 2 > $O/r02_prof_step.log 2>&1
# (-k regex:'^(add_rmsnorm|argmax|decode_attn|embed_kernel|gemm_|prefill_attn|rope_|activate_rows|gather_|silu_mul|decode_layer)' : only this library's kernels count for -s / -c; torch's weight-initialisation kernels do not;
#  launch 0 is rr::rope_table_kernel at engine creation)
# decode step 2 (step 1 warms up), eager launches: embed, norm0, then layer 0 = qkv, attention, o, norm, fused mlp, norm
ncu --set full --clock-control none --import-source on -k regex:'^(add_rmsnorm|argmax|decode_attn|embed_kernel|gemm_|prefill_attn|rope_|activate_rows|gather_|silu_mul|decode_layer)' -s 197 -c 8 -f -o $O/r02_decode_layer0 \
    python tools/profile_step.py --prefill-prompts 0 --decode-steps 2 > $O/r02_ncu_a.log 2>&1
# ... and its last two kernels: lm_head GEMM, argmax
ncu --set full --clock-control none --import-source on -k regex:'^(add_rmsnorm|argmax|decode_attn|embed_kernel|gemm_|prefill_attn|rope_|activate_rows|gather_|silu_mul|decode_layer)' -s 391 -c 2 -f -o $O/r02_decode_head \
    python tools/profile_step.py --prefill-prompts 0 --decode-steps 2 > $O/r02_ncu_b.log 2>&1
# prefill chunk (16 x 512 tokens), layer 0: qkv (2-CTA, RoPE epilogue), attention (tcgen05), o (residual epilogue), gate/up (SiLU), down
ncu --set full --clock-control none --import-source on -k regex:'^(add_rmsnorm|argmax|decode_attn|embed_kernel|gemm_|prefill_attn|rope_|activate_rows|gather_|silu_mul|decode_layer)' -s 3 -c 5 -f -o $O/r02_prefill_layer0 \
    python tools/profile_step.py --decode-steps 0 > $O/r02_ncu_c.log 2>&1
# K1 router kernel + tokenizer kernel
ncu --set full --clock-control none -k regex:'router_kernel|tokenize_kernel' -c 4 -f -o $O/r02_router_tokenizer \
    python -m pytest tests/test_router_gpu.py tests/test_tokenizer_gpu.py -x -q > $O/r02_ncu_d.log 2>&1
ls -la $O/*.ncu-rep
if [ "${1:-}" = "--ncu-only" ]; then exit 0; fi
# compute-sanitizer
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_ops_gpu.py tests/test_tokenizer_gpu.py \
    tests/test_router_gpu.py -x -q > $O/r02_sanitizer_memcheck_ops.log 2>&1; echo "memcheck ops rc=$?" | tee -a $O/r02_sanitizer_memcheck_ops.log
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_engine_gpu.py -x -q \
    -k "tiny or (small and 64) or serving" > $O/r02_sanitizer_memcheck_engine.log 2>&1
echo "memcheck engine rc=$?" | tee -a $O/r02_sanitizer_memcheck_engine.log
timeout 900 compute-sanitizer --tool racecheck --error-exitcode 1 python -m pytest tests/test_ops_gpu.py tests/test_tokenizer_gpu.py -x -q \
    > $O/r02_sanitizer_racecheck_ops.log 2>&1; echo "racecheck ops rc=$?" | tee -a $O/r02_sanitizer_racecheck_ops.log
for f in $O/r02_sanitizer_*.log; do tail -n 3 $f; done
