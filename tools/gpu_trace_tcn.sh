#!/bin/bash
# phase timers of the single-CTA temporal-conv kernel (who waits: the TMA producer or the MMA issuer?), printed to stdout.
# It serves the 64-channel layers (COSK_FUSE_BLOCK=0: as its own launch, not inside k_tc_block64); the 128- and
# 256-channel ones run on CTA pairs (k_tc_tcn2), which record no timers.
cd "${GRAFT_REPO_ROOT:-/root/repo}"
cat > /tmp/trace_tcn.py <<'PY'
import sys, torch
sys.path.insert(0, '.')
import continual_skeletons_b200 as cs
for c in (64,):
    st = cs.CoStack([cs.BlockSpec(c, c, 1, True)], padding=4)
    x = torch.rand(8192, c, 25, device='cuda')
    for t in range(12):
        st.forward_step(x)
    torch.cuda.synchronize()
    tr = st.trace_read(32)
    print(f"tcn C={c}: producer wait {tr[24]} of {tr[25]} cycles | mma wait operands {tr[26]} wait accumulator {tr[27]} of {tr[28]} cycles")
PY
COSK_TRACE=1 COSK_FUSE_BLOCK=0 timeout 300 python /tmp/trace_tcn.py 2>&1
