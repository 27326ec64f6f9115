"""Regenerates tests/golden/ref_ikdtree.json: what the reference's own ikd-Tree (compiled unmodified into oracle/_ref by
`make -C oracle REF=<reference source tree>`) returns on the call sequences of the tests that compare a map with it
(tests/test_oracle_map.py, tests/test_gpu_api.py).  Those tests replay the same calls on the map under test and compare
call by call, so they need neither the reference source nor oracle/_ref.

    python tests/golden/make_golden_ref.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import pyoracle as po  # noqa: E402
from tests import test_gpu_api as api, test_oracle_map as om  # noqa: E402
from tests.helpers import REF_GOLDEN, RecordedMap  # noqa: E402


def main():
    assert po.have_ref(), "build oracle/_ref first"
    scene = api.api_scene()
    cases = {"port_knn": lambda m: om.knn_calls(m),
             "port_add_delete": lambda m: om.add_delete_calls(m),
             "properties": lambda m: om.properties_calls(m),
             "nearest_search_other_k_and_max_dist": lambda m: api.nearest_search_calls(m, scene),
             "delete_points": lambda m: api.delete_points_calls(m, scene),
             "intensity": lambda m: api.intensity_calls(m, scene)}
    out = {}
    for name, run in cases.items():
        m = RecordedMap(po.RefIkdTree(ds=0.2))
        run(m)
        out[name] = m.calls
        m.close()
        print(name, len(m.calls), "calls")
    with open(REF_GOLDEN, "w") as f:      # one call per line
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: [\n  " + ",\n  ".join(json.dumps(c) for c in v) + "]"
                                     for k, v in out.items()) + "\n}\n")


if __name__ == "__main__":
    main()
