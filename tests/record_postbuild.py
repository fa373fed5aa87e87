"""Record the digests of tests/golden/postbuild.json from the drop-in class:

    python -m tests.record_postbuild OUT.json          # read-only scans and statistics, on the C-oracle test double
    python -m tests.record_postbuild OUT.json --gpu    # the node removals, the k sweep and the lazy rebuild, on cuda:0

Entries already in OUT.json and not recorded by this run are kept.  A recording is only as good as the code it
ran: record from a commit whose results are known to equal upstream's."""
import json
import os
import sys
import tempfile

from amira_b200 import construct_graph
from tests import test_host_mirror_cpu, test_postbuild
from tests.fake_device import OracleBackedDevice
from tests.helpers import digest


def record(gpu):
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        if gpu:
            for name, k in test_postbuild.CASES:
                ours, vocab, _ = test_postbuild.readonly_values(name, k, tmp)
                out["edits/%s_k%d" % (name, k)] = test_postbuild.edit_values(ours, vocab)
            out["k_sweep/fixture_four"] = test_postbuild.k_sweep_values()
            out["lazy_rebuild/fixture_eight"] = test_postbuild.lazy_rebuild_values()
        else:
            construct_graph._HANDLES.clear()
            construct_graph.DeviceGraph = OracleBackedDevice
            for name, k in test_postbuild.CASES:
                out["scans/%s_k%d" % (name, k)] = test_postbuild.readonly_values(name, k, tmp)[2]
            out["statistics/c3_400"] = test_host_mirror_cpu.statistics_values()
    return {key: {label: digest(v) for label, v in values.items()} for key, values in out.items()}


if __name__ == "__main__":
    path = sys.argv[1]
    gold = {}
    if os.path.exists(path):
        with open(path) as f:
            gold = json.load(f)
    gold.update(record("--gpu" in sys.argv))
    with open(path, "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
        f.write("\n")
