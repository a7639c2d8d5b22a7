#!/bin/bash
# Marginal cost of each kernel family INSIDE the replayed training-step graph: run bench.py with one family of
# entry points turned into no-ops (POLUS_ABLATE, polus_b200/_lib.py) and compare ms/step.
# usage: tools/ablate_step.sh [out_file]
out=${1:-gpurun_out/ablate.txt}
: > "$out"
run() {  # label, env...
    label=$1; shift
    line=$(env "$@" python bench.py --steps 20 --warmup 3 --no-cpu-baseline 2>&1 | grep '"metric"' | tail -1)
    ms=$(echo "$line" | python -c 'import sys,json; d=json.loads(sys.stdin.read()); print("%.3f ms/step  %.0f seq/s  gemm_frac %.3f" % (d["ms_per_step"], d["value"], d["roofline"]["frac"]))' 2>/dev/null || echo "FAILED")
    printf "%-44s %s\n" "$label" "$ms" | tee -a "$out"
}
run "full"
run "- layernorm fwd+bwd" POLUS_ABLATE=polus_ln_res_fwd,polus_ln_res_bwd
run "- act_bwd_colsum" POLUS_ABLATE=polus_act_bwd_colsum
run "- attention fwd+bwd" POLUS_ABLATE=polus_attention_fwd,polus_attention_bwd
run "- attention bwd" POLUS_ABLATE=polus_attention_bwd
run "- adam" POLUS_ABLATE=polus_adam
run "- crf nll+decode" POLUS_ABLATE=polus_crf_nll,polus_crf_decode
run "- tcgen05 gemms" POLUS_ABLATE=polus_gemm_tc
run "- everything but gemms" POLUS_ABLATE=polus_ln_res_fwd,polus_ln_res_bwd,polus_act_bwd_colsum,polus_attention_fwd,polus_attention_bwd,polus_adam,polus_crf_nll,polus_crf_decode,polus_embed_ln_fwd,polus_embed_ln_bwd
