"""Developer tool: compare the per-kernel tables of two bench.py runs (A/B of a kernel change).
    python bench.py > a.json 2>&1; ...; python tools/cmp_bench.py a.json b.json [threshold_ms]"""
import json
import sys


def load(p):
    """The result line (stdout) merged with the per-kernel tables bench.py prints on stderr."""
    d = {}
    for line in open(p):
        if line.startswith("{"):
            d.update(json.loads(line))
    return d


a, b = load(sys.argv[1]), load(sys.argv[2])
thr = float(sys.argv[3]) if len(sys.argv) > 3 else 0.03
print(f"value {a['value']:.3f} -> {b['value']:.3f}   ms/step {a['ms_per_step']:.2f} -> {b['ms_per_step']:.2f}   "
      f"e2e {a['e2e']['value']:.3f} -> {b['e2e']['value']:.3f}   clocks {a['clocks']['sm_mhz']} -> {b['clocks']['sm_mhz']}")
ka, kb = a["kernels"], b["kernels"]
ta = sum(v["ms"] for v in ka.values())
tb = sum(v["ms"] for v in kb.values())
print(f"instrumented frame: {ta:.2f} -> {tb:.2f} ms")
for k in sorted(set(ka) | set(kb), key=lambda k: -max(ka.get(k, {}).get("ms", 0), kb.get(k, {}).get("ms", 0))):
    x, y = ka.get(k, {}).get("ms", 0.0), kb.get(k, {}).get("ms", 0.0)
    if abs(x - y) >= thr:
        print(f"  {k:40s} {x:8.3f} -> {y:8.3f}  ({y - x:+.3f})")
