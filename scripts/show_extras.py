import json, sys
# bench.py prints the result line on stdout and `extras` / `roofline_by_kernel` on stderr: pass both files (or one with both)
d = {}
for path in sys.argv[1:]:
    for l in open(path):
        if l.startswith("{"):
            d.update(json.loads(l))
print(f"headline {d['value']/1e9:.1f} Gpts/s  {d['roofline']['achieved']:.0f} GB/s frac {d['roofline']['frac']:.3f} clocks {d['clocks']}")
for k, v in d["extras"]["linearize_100M"].items():
    print(f"  linearize {k:28s} {v['ms']:.3f} ms {v['gb_s']:.0f} GB/s")
for k, v in d["extras"]["project_unproject_100M_f64"].items():
    print(f"  {k:16s} project {v['project_ms']:.3f} ms {v['project_gb_s']:.0f} GB/s   unproject {v['unproject_ms']:.3f} ms {v['unproject_gb_s']:.0f} GB/s   fused round trip {v.get('round_trip_fused_ms', 0):.3f} ms {v.get('round_trip_fused_gb_s', 0):.0f} GB/s")
print("  undistort", d.get("undistort_batch") or d["extras"].get("undistort_4096x4096_kb_bilinear"))
if d.get("lm_conversion"): print("  lm", {k: d["lm_conversion"][k] for k in ("ms", "iterations", "passes", "us_per_pass")})
if d.get("e2e"): print("  e2e", d["e2e"]["value"] / 1e9, "Gpts/s")
