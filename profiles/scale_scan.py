"""FP32 span scaling at wide spans: how many cfg4 sequences leave the safe range, and on which side, as a function of
kappa = 2^-klog2 (stored Alpha = cA kappa^d x, stored Beta = cB kappa^-d y; DESIGN.md §2.6).
usage: scale_scan.py [W=150] [n=1000] [full | wide]
wide: the same for the wide-span FP64 engine (W > 200, DESIGN.md §2.9): sequences re-run in the exact engine as a
function of PRIB_WIDE_KLOG2 (cA = cB = 1)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r'''
import json, sys
sys.path.insert(0, %r)
from priblast_b200 import Raccess, workloads
W, n = int(sys.argv[1]), int(sys.argv[2])
seqs = workloads.cfg4(first=n)
with Raccess(W, 5) as r:
    r.stage(seqs); r.compute(); r.sync()
    c = r.counters()
print(json.dumps({"flagged": c["fp32_flagged"], "rerun": c["fp64_rerun_sequences"],
                  "exact_rerun": c["exact_rerun_sequences"], "ms": round(c["kernel_ms"], 1)}))
''' % ROOT
W = sys.argv[1] if len(sys.argv) > 1 else "150"
n = sys.argv[2] if len(sys.argv) > 2 else "1000"
full = len(sys.argv) > 3 and sys.argv[3] == "full"
if len(sys.argv) > 3 and sys.argv[3] == "wide":
    for k in (0.30, 0.45, 0.60, 0.75):
        env = dict(os.environ, PRIB_WIDE_KLOG2=str(k))
        p = subprocess.run([sys.executable, "-c", CHILD, W, n], env=env, capture_output=True, text=True)
        print(f"W={W} wide klog2={k:.2f}:", p.stdout.strip().splitlines()[-1] if p.stdout.strip() else p.stderr[-300:], flush=True)
    sys.exit(0)
for k in ((0.20, 0.25, 0.30, 0.35, 0.40, 0.45, 0.50) if full else (0.30, 0.35, 0.40, 0.45, 0.50, 0.55)):
    for a, b in (((4.0, 16.0), (0.0, 16.0), (-8.0, 24.0), (12.0, 8.0)) if full else ((4.0, 16.0), (12.0, 8.0))):
        env = dict(os.environ, PRIB_KLOG2=str(k), PRIB_ALOG2=str(a), PRIB_BLOG2=str(b))
        p = subprocess.run([sys.executable, "-c", CHILD, W, n], env=env, capture_output=True, text=True)
        print(f"W={W} klog2={k:.2f} alog2={a:5.1f} blog2={b:5.1f}:", p.stdout.strip().splitlines()[-1] if p.stdout.strip() else p.stderr[-300:], flush=True)
