"""Measured deviations of pasn_head_backward from float64 autograd over the runs of tests/test_backward_parity_gpu.py: one
line per run (conditioning margin, then max |got - ref| / max |ref| per gradient), then the worst value per family (the
figures next to BWD_TILED_MAX / BWD_GENERIC_MAX in tests/util.py and in DESIGN.md section 2.5).

    python tools/bwd_parity_report.py [--seed S] [--lib PATH] [--only tiled|generic] [--json OUT]

--lib measures another build of the library (e.g. of an older commit) against the same references; a run that fails
with an error is reported as such and the sweep goes on.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from protoasnet_b200 import _lib  # noqa: E402
from tests import test_backward_parity_gpu as t  # noqa: E402
from tests.bwd_reference import KEYS  # noqa: E402

SHORT = dict(zip(KEYS, ["W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4", "W5", "V", "Wl"]), grad_feat="gX")


def sweep(seed=t.SEED, only=None, chunked=True):
    rows = []
    runs = t.RUNS + ([(t.CHUNKED_CASE, "chunked-all"), (t.CHUNKED_CASE, "chunked-occ_only")] if chunked else [])
    for case, combo in runs:
        fam = "tiled" if case[0] == t.TILED else "generic"
        if only and fam != only:
            continue
        r = {"case": t.case_id(case, combo), "family": fam}
        try:
            if combo.startswith("chunked-"):   # PASN_TILED_CHUNK = 3, in a process of its own
                r.update(t.run_chunked(seed)[combo[len("chunked-"):]])
            else:
                r.update(t.run_case(case, combo, seed))
            r["limit"] = t.threshold(case)
            r["pass"] = not r["untouched"] and all(v <= r["limit"] for v in r["dev"].values()) and r["margin"] >= t.TAU and r["fe_margin"] >= t.TAU_FE
        except Exception as e:   # noqa: BLE001 -- a failing build is what this reports
            r.update(error=f"{type(e).__name__}: {str(e)[:300]}", **{"pass": False})
        rows.append(r)
        if "error" in r:
            print(f"{r['case']}: ERROR {r['error']}", flush=True)
        else:
            devs = " ".join(f"{SHORT[k]}={v:.2g}" for k, v in r["dev"].items())
            extra = f" untouched-violated={r['untouched']}" if r["untouched"] else ""
            print(f"{r['case']}: margin={r['margin']:.3g} fe_margin={r['fe_margin']:.3g} rounds={r['rounds']} {devs}{extra} {'ok' if r['pass'] else 'FAIL'}",
                  flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=t.SEED)
    ap.add_argument("--lib", default=None, help="another build of libpasn_b200.so")
    ap.add_argument("--only", choices=("tiled", "generic"), default=None)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if a.lib:
        _lib.LIB_PATH = os.path.abspath(a.lib)
    print(torch.cuda.get_device_name(0), _lib.LIB_PATH)
    t0 = time.time()
    rows = sweep(a.seed, a.only)
    print(f"{len(rows)} runs in {time.time() - t0:.1f} s, {sum(not r['pass'] for r in rows)} failing")
    for fam in ("tiled", "generic"):
        rs = [r for r in rows if r["family"] == fam and "dev" in r]
        if rs:
            worst = max((v, k, r["case"]) for r in rs for k, v in r["dev"].items())
            wnorm = max(v for r in rs for v in r["norm"].values())
            print(f"{fam}: worst max-deviation {worst[0]:.3g} ({SHORT[worst[1]]}, {worst[2]}), worst normwise {wnorm:.3g}, "
                  f"smallest margin {min(r['margin'] for r in rs):.3g}")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
