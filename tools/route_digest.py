"""Seeded digest of the routing matrix of tests/test_gpu_routes.py: for every case, the kernels one call launched, the launch and
replay counts, the integer counters and sum_err2 / sum_ref2 / sum_evm_lin as hex doubles.  Two builds that route and compute
alike write byte-identical files:
    python tools/route_digest.py OUT.json                 (OFDM_B200_LIB=<other build> for the other arm)"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import __graft_entry__ as e  # noqa: E402
import test_gpu_routes as routes  # noqa: E402

pkg = e.load_pkg()
o = pkg.Ofdm(0)
out = {}
for c in routes.cases():
    kernels, launches, replayed, counters, _ = routes.run_case(o, pkg, c)
    out[routes.case_id(c)] = {
        "kernels": kernels, "launches": launches, "replayed": replayed,
        "counters": [[int(x.bit_errors), int(x.bits), int(x.frames_in_error), int(x.rail_errors), int(x.frames),
                      float(x.sum_err2).hex(), float(x.sum_ref2).hex(), float(x.sum_evm_lin).hex()] for x in counters]}
o.close()
with open(sys.argv[1], "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
    f.write("\n")
print("%d cases -> %s" % (len(out), sys.argv[1]))
