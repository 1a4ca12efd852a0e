"""Measured deviations of the tensor-core forward from oracle/emulate.py over the cases of
tests/test_tc_emulated_parity_gpu.py: one line per case, then the maximum per check and path (the figures of DESIGN.md
section 5 and the measured maxima next to the thresholds in tests/util.py).

    python tools/emu_parity_report.py [--json OUT]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tests.test_tc_emulated_parity_gpu import CASES, FUSED, _ids, run_case  # noqa: E402

CHECKS = ("occ_biteq_min", "occ_worst", "feat", "sim", "logits", "cos_push", "cos_fwd")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    print(torch.cuda.get_device_name(0))
    rows = []
    t0 = time.time()
    for c in CASES:
        r = run_case(c)
        r["case"] = _ids(c)
        r["family"] = "fused" if c[0] == FUSED else "tiled"
        rows.append(r)
        print(r["case"], " ".join(f"{k}={r[k]:.3g}" for k in CHECKS), flush=True)
    print(f"{len(rows)} cases in {time.time() - t0:.1f} s")
    for fam in ("fused", "tiled"):
        for order in ("pool_first", "w2_first"):
            rs = [r for r in rows if r["family"] == fam and r["order"] == order]
            if rs:
                agg = {k: (min if k == "occ_biteq_min" else max)(r[k] for r in rs) for k in CHECKS}
                print(f"{fam} {order}: " + " ".join(f"{k}={v:.3g}" for k, v in agg.items()))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
