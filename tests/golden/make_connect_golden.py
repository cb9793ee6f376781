#!/usr/bin/env python
"""Generate tests/golden/connect_labels.npz: what LabelConnected (lib/visfd/connect.hpp:171, the arguments HandleTV
passes) gives for the inputs tests/test_gpu_connect.py builds -- labels, cluster counts and, for the membrane cases,
the standardised directions of the clustered voxels -- with a SHA-256 of each case's inputs.  The inputs come from
the CPU restatement (oracle/visfd_oracle.cpp), as in the tests; no GPU is needed.

    python tests/golden/make_connect_golden.py [OUT.npz]

The labels come from the unmodified reference (oracle/_ref) where it has been built, otherwise from the restatement,
which tests/test_oracle_golden.py::test_label_connected_restatement_is_the_reference pins to the reference's labels
and directions.  tests/golden/README.md says where the committed file came from."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    from oracle.pyoracle import Oracle, have
    import test_gpu_connect as tc
    from util import sha256_of
    port = Oracle("port")
    ref = Oracle("reference") if have("reference") else port
    out = {}
    for seed, shape, angle, quant in tc.MEMBRANE_CASES:
        sal, tensor, thr = tc.membrane_case(port, seed, shape, quant)
        labels, n, direction = ref.label_connected(sal, tensor, thr, angle_deg=angle, want_direction=True)
        key = "membrane_%d_" % seed
        out[key + "inputs_sha256"] = np.array(sha256_of(sal, tensor, np.float32(thr)))
        out[key + "labels"], out[key + "n_clusters"] = labels.astype(np.int16), np.int64(n)
        out[key + "direction_inside"] = direction[labels >= 1]
    for seed in range(6):
        sal, tensor, mask, thr = tc.random_field_case(port, seed)
        out["random_%d_inputs_sha256" % seed] = np.array(sha256_of(sal, tensor, mask, np.float32(thr)))
        for angle in tc.RANDOM_FIELD_ANGLES:
            labels, n = ref.label_connected(sal, tensor, thr, angle_deg=angle, mask=mask)
            key = "random_%d_%g_" % (seed, angle)
            out[key + "labels"], out[key + "n_clusters"] = labels.astype(np.int16), np.int64(n)
    sal, tensor = tc.plateau_case(port)
    labels, n = ref.label_connected(sal, tensor, tc.PLATEAU_THRESHOLD, thresholds=(-np.inf,) * 4)
    out["plateau_inputs_sha256"] = np.array(sha256_of(sal, tensor))
    out["plateau_labels"], out["plateau_n_clusters"] = labels.astype(np.int16), np.int64(n)
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "connect_labels.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "(labels of the %s)" % ref.kind, "%.1f KiB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
