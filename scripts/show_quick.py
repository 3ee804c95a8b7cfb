"""Summary of the bench lines a scripts/gpu_quick.sh call left behind: python scripts/show_quick.py TAG [SUFFIX...]"""
import json, sys
tag = sys.argv[1]
sfxs = sys.argv[2:] or [""]
for w in ["ml10m", "ml1m", "jester", "ml20m", "netflix"]:
    for sfx in sfxs:
        try:
            d = json.load(open("gpurun_out/%s_bench_%s%s.json" % (tag, w, sfx)))
        except Exception as e:
            print(w, sfx, "ERR", e); continue
        r = d.get("roofline") or {}
        print("%-8s%-9s value %7.1fM e2e %7.1fM ms/step %.4f e2e_ms %.4f launches/step %.1f  %s frac %.3f share %.2f" % (
            w, sfx, d["value"] / 1e6, d["e2e"]["value"] / 1e6, d["ms_per_step"], d["e2e"]["ms_per_step"], d["gpu_launches"] / d["steps"],
            (r.get("kernel") or "?")[:14], r.get("frac") or 0, r.get("share_of_step") or 0))
        if sfx == sfxs[0]:
            for k, v in (d.get("kernels") or {}).items():
                print("     %-22s %.4f ms  %s GB/s" % (k, v["ms"], None if v.get("GB/s") is None else round(v["GB/s"])))
