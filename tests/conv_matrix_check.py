"""The conv kernel matrix of tests/test_gpu_conv_matrix.py under the kernel switches of the calling environment (DT_CONV_MMA, DT_CONV_WS,
DT_CONV_SLOTS, DT_CONV_NARROW1, DT_CONV_HALO, DT_CONV_RES_RING, DT_CONV_PDL: read once per process).  Prints one JSON line per case and a
last line {"rows": [instantiation rows reached], "failed": [...]}.  Run by test_gpu_conv_matrix.py::test_conv_matrix_under_switch;
`--dynamic-range` adds the input-scale sweep."""
import json
import os
import sys
import traceback

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_conv_matrix as M  # noqa: E402


def main():
    dev = torch.device("cuda:0")
    rows, failed = set(), []

    def attempt(name, fn):
        try:
            return fn()
        except Exception as e:          # noqa: BLE001 -- report every failing case, not just the first
            failed.append("%s: %s" % (name, e))
            traceback.print_exc()
            return None

    for c in M.matrix_cases():
        r = attempt(c["name"], lambda: M.run_case(c, dev))
        if r is None:
            continue
        rows.add(r["plan"]["instantiation"])
        if "rows2" in r:
            rows.add(r["rows2"])
        print(json.dumps({"case": c["name"], "kind": c["kind"], "ratio": r["ratio"], "rel": r["rel"], "row": r["plan"]["instantiation"]}), flush=True)
        attempt(c["name"], lambda: M.check_result(c, r))
    attempt("range_flag", lambda: M.range_flag_checks(dev))
    if os.environ.get("DT_CONV_PDL") == "1":
        attempt("pdl chain", lambda: M.pdl_chain_check(dev))
    if "--dynamic-range" in sys.argv:
        for r in M.dynamic_range(dev):
            print(json.dumps({"dyn": r["exp"], "kind": r["kind"], "x_multiplier": r["x_multiplier"], "ratio": r["ratio"],
                              "rel_maxabs": r["rel_maxabs"]}), flush=True)
    print(json.dumps({"rows": sorted(rows), "failed": failed}))
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main())
