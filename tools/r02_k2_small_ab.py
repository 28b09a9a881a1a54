"""A/B of the votes kernel on sparse tiles (P <= 1024 tracked points per query) in ONE process on one GPU:
python tools/r02_k2_small_ab.py > gpurun_out/r02_k2_small_ab.json
Per workload (the C1 video, a 32-video slice of the C4 mixture, three 1 k-track points of the C5 sweep) and per kernel
(s2d_point_votes_variant: 4 = one warp per tile for every frame size, 3 = label-table kernel, 2 = one CTA per tile):
K2 time, fraction of the measured HBM copy peak, frames/s, and the digest of the results (must not depend on the kernel)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from s2d_b200 import _lib                                            # noqa: E402
from s2d_b200 import workloads as wl                                # noqa: E402
from s2d_b200.pipeline import Params                                # noqa: E402

PEAK = 6548.2
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def main():
    dev = torch.device("cuda:0")
    lists = {
        "c1": [wl.VideoSpec("c1", 2024, 24, 480, 854, 10, 1000)],
        "c4_32": wl.c4_specs(512)[:32],
        "c5_m10_t8": wl.c5_specs(10, 1024, 8),
        "c5_m50_t32": wl.c5_specs(50, 1024, 32),
        "c5_m100_t64": wl.c5_specs(100, 1024, 64),
    }
    configs = [("table", 3), ("warp_per_tile", 4), ("cta_per_tile", 2)]
    out = {"peak_gbs": PEAK, "rows": []}
    runner = wl.DeviceRunner(dev, Params())
    runner.run_list([wl.VideoSpec(f"warm{i}", 7 + i, 16, 240, 426, 8, 1024) for i in range(2)])
    for lname, specs in lists.items():
        ref = None
        for cname, variant in configs:
            _lib.call("s2d_point_votes_variant", variant)
            res, st, _ = runner.run_list(specs, warm=2)
            dig = wl.list_digest(res)
            ref = ref or dig
            k2ms = st["k2_ms"]                                       # of the last repetition
            row = {"list": lname, "kernel": cname, "k2_ms": round(k2ms, 4), "k2_frac": round(st["k2_bytes"] / (k2ms / 1e3) / 1e9 / PEAK, 4),
                   "device_ms": round(st["device_ms"], 3), "frames_per_s": round(st["frames"] / (st["device_ms"] / 1e3)),
                   "tiles": st["k2_tiles"], "same_results": dig == ref}
            out["rows"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
    _lib.call("s2d_point_votes_variant", 0)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
