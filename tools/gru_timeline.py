"""Developer tool: per-step timeline (ns) of CTA 0 of the GRU recurrence at north-star width.

    python tools/gru_timeline.py [fwd|bwd]      (TL_B=<batch>, default 64)
"""
import sys
import numpy as np, torch
sys.path.insert(0, ".")
from speech_b200 import _lib, ops
lib = _lib.load()
torch.manual_seed(0)
import os
B, T, In, H = int(os.environ.get('TL_B', '64')), 64, 2048, 1024
rnn = torch.nn.GRU(In, H, 1, batch_first=True, bidirectional=True).cuda()
x = torch.randn(B, T, In, device="cuda")
dbg = torch.zeros(64 * 16 + 512, dtype=torch.int64, device="cuda")
MODE = sys.argv[1] if len(sys.argv) > 1 else "fwd"
if MODE == "fwd":
    with torch.no_grad():
        ops.gru_stack(x, rnn)
        torch.cuda.synchronize()
        lib.sb_debug_gru_timeline(dbg.data_ptr())
        ops.gru_stack(x, rnn)
        torch.cuda.synchronize()
        lib.sb_debug_gru_timeline(None)
else:
    xr = x.clone().requires_grad_(True)
    y = ops.gru_stack(xr, rnn)
    y.sum().backward()
    y = ops.gru_stack(xr, rnn)
    torch.cuda.synchronize()
    lib.sb_debug_gru_timeline(dbg.data_ptr())
    y.sum().backward()
    torch.cuda.synchronize()
    lib.sb_debug_gru_timeline(None)
print("mode:", MODE)
raw = dbg.cpu().numpy()
d = raw[:1024].reshape(64, 16)
names = ["P:grid_wait done", "P:tma issued", "M:all mma committed", "E:accfull",
         "E:tmem loaded (+reduce-scatter)", "E:xn stored", "E:proxy fence", "E:epi barrier", None,
         "E:arrived", "E:offpath done"]
for step in (11, 40):
    base = d[step - 1][9]   # previous step's arrival by this CTA
    print("step %d (ns since this CTA's previous arrive):" % step)
    for i, n in enumerate(names):
        if n is None:
            continue
        print("   %-22s %7d" % (n, d[step][i] - base))
print("cluster size used:", lib.sb_debug_gru_cluster(0))
print("mean step period (ns):", (d[60][9] - d[10][9]) / 50.0)

if MODE == "fwd":
    arr = raw[1024:1024 + 128].astype(np.float64)
    seen = raw[1024 + 256:1024 + 256 + 128].astype(np.float64)
    if arr.min() > 0:
        a0 = arr.min()
        print("skew probe, step 20 -> 21 (ns after the earliest arrive): arrive per CTA (dir 0 | dir 1)")
        for dname, sl in (("dir0", slice(0, 64)), ("dir1", slice(64, 128))):
            a = arr[sl] - a0
            w = seen[sl] - a0
            print("  %s arrive: min %5.0f  p50 %5.0f  p90 %5.0f  max %5.0f | barrier seen: min %5.0f p50 %5.0f max %5.0f"
                  % (dname, a.min(), np.percentile(a, 50), np.percentile(a, 90), a.max(),
                     w.min(), np.percentile(w, 50), w.max()))
        print("  slowest arrivers (cta, ns):", sorted([(int(i), int(arr[i] - a0)) for i in range(128)],
                                                   key=lambda t: -t[1])[:8])
