#!/bin/bash
# Round 2: quick check of a kernel change -- guarded parity subset, bench, k_tc_gcnt phase trace.
cd "${GRAFT_REPO_ROOT:-/root/repo}"
mkdir -p gpurun_out
rm -f gpurun_out/summary.txt
run() { name=$1; shift; timeout $1 "${@:2}" > gpurun_out/$name.log 2>&1; echo "$name rc=$?" >> gpurun_out/summary.txt; }
run pytest_quick 400 python -m pytest tests/test_gpu_parity.py -x -q -m gpu --timeout 60 -k "${QUICK_K:-channel_major or forward_steps_vs_reference or kinetics or long_run or state_lifecycle}"
if ! grep -q "pytest_quick rc=0" gpurun_out/summary.txt; then tail -40 gpurun_out/pytest_quick.log | cut -c1-400; exit 1; fi
run bench_a 300 python bench.py --steps 200 --warmup 8 --no-cpu-baseline ${BENCH_ARGS}
run bench_b 300 python bench.py --steps 200 --warmup 8 --no-cpu-baseline ${BENCH_ARGS}
cat > /tmp/trace.py <<'PY'
import sys, os, torch
sys.path.insert(0, '.')
import continual_skeletons_b200 as cs
for cin, cout in ((64, 128), (128, 128), (128, 256)):
    st = cs.CoStack([cs.BlockSpec(cin, cout, 1, True)], padding=4)
    N = 4096
    x = torch.rand(N, cin, 25, device='cuda')
    for t in range(6):
        st.forward_step(x)
    torch.cuda.synchronize()
    tr = st.trace_read(16)
    n = max(tr[4], 1)
    print(f"k_tc_gcnt {cin}->{cout} ({st.knobs()['blocks'][0]['gcn']}): per chunk-item (cycles): epilogue wait_acc {tr[0]//n} load+mix {tr[1]//n} store {tr[2]//n} total {tr[3]//n} | "
          f"mma wait_acc_free {tr[8]//n} wait_x {tr[9]//n} wait_w {tr[10]//n} total {tr[11]//n} | producer wait_x_free {tr[12]//n} wait_w_free {tr[13]//n} | chunk-items {n}")
PY
COSK_TRACE=1 run trace_gcnt 120 python /tmp/trace.py
cat gpurun_out/summary.txt
tail -n 3 gpurun_out/pytest_quick.log | cut -c1-300
cat gpurun_out/trace_gcnt.log | cut -c1-420
python - <<'PY'
import json
for f in ('bench_a','bench_b'):
    txt=open(f'gpurun_out/{f}.log').read()
    for line in txt.split('\n'):
        if line.startswith('{'):
            d=json.loads(line)
            pb=d['kernel_time_per_block_ms']
            print(f, round(d['value']), 'e2e', round(d['e2e']['value']), 'ms/step', round(d['ms_per_step'],4), 'p50', round(d.get('p50_ms_per_step'),3), d.get('clocks',{}).get('sm_mhz'))
            print('   gcn/launch', [round(b['gcn_ms']/max(b['gcn_n'],1),4) for b in pb], 'attn', [round(b.get('attn_ms',0)/max(b.get('attn_n',1),1),4) for b in pb])
            print('   tcn/launch', [round(b['tcn_ms']/max(b['tcn_n'],1),4) for b in pb], 'blk', [round(b['block_ms']/max(b['block_n'],1),4) for b in pb], 'head', round(d['kernel_time_ms']['head']['ms']/max(d['kernel_time_ms']['head']['launches'],1),4))
    if 'Traceback' in txt: print(txt[-800:])
PY
