#!/bin/bash
# compute-sanitizer passes over the hot-path kernels at test sizes (SURVEY §5): memcheck on smoke() (tcgen05 GEMMs,
# prefill attention, the persistent decode kernel at batch 1, sampler, codec kernels) and on a batched decode
# (batch 6: fold-phase variant of the persistent kernel; batch 12 via NT_DECODE_IMPL=perop: the per-op chain with
# attn_decode_mma_kernel), racecheck (shared-memory hazards) on smoke().  Poll loops in the persistent kernel carry
# spin limits, so a sanitizer-induced slowdown shows up as a trap, not a hang.
out=gpurun_out/sanitizer
mkdir -p $out
run() { name=$1; shift; timeout 1500 compute-sanitizer "$@" > $out/$name.log 2>&1; echo "rc=$?" >> $out/$name.log; tail -4 $out/$name.log; }
if [ "$1" = codec_ragged ]; then   # ragged codec batch, tiny config, all three arithmetic modes
  run memcheck_codec_ragged --tool memcheck --print-limit 20 python -m pytest -q -m gpu tests/test_gpu_codec_ragged.py -k tiny_config
  exit 0
fi
run memcheck_smoke --tool memcheck --print-limit 20 python -c "import __graft_entry__ as g; g.smoke()"
run memcheck_batched --tool memcheck --print-limit 20 python profiles/sanitizer_batched.py
run racecheck_smoke --tool racecheck --racecheck-report all --print-limit 20 python -c "import __graft_entry__ as g; g.smoke()"
