"""Generates tests/golden/ref_pickle_digests.npz: what the reference's pretrained pickles hold, in a form small enough
to keep in the repository.  For every leaf of pretrained/<Env>/gcbf+/models/1000/{actor,cbf}.pkl it records the shape,
the SHA-256 of its float32 bytes and a seeded sample of its values; tests/test_oracle.py checks params_<Env>.npz
against them.
Usage: python tests/golden/make_pickle_digests.py --reference <gcbfplus checkout>
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from oracle.nn import flatten_params, load_ref_pickle  # noqa: E402

ENVS = ["SingleIntegrator", "DoubleIntegrator", "DubinsCar", "LinearDrone"]
N_SAMPLE = 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of MIT-REALM/gcbfplus")
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    meta, index, value = {}, [], []
    for env in ENVS:
        meta[env] = {}
        for net in ["actor", "cbf"]:
            tree = load_ref_pickle(os.path.join(args.reference, "pretrained", env, "gcbf+", "models", "1000", f"{net}.pkl"))
            for k, v in flatten_params(tree).items():
                assert v.dtype == np.float32, (env, net, k, v.dtype)
                v = np.ascontiguousarray(v)
                idx = np.sort(rng.choice(v.size, size=min(N_SAMPLE, v.size), replace=False))
                start = sum(len(i) for i in index)
                index.append(idx)
                value.append(v.ravel()[idx])
                meta[env][f"{net}:{k}"] = {"shape": list(v.shape), "sha256": hashlib.sha256(v.tobytes()).hexdigest(),
                                           "sample": [start, start + len(idx)]}
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_pickle_digests.npz")
    np.savez_compressed(out, meta=np.asarray(json.dumps(meta, sort_keys=True)), index=np.concatenate(index),
                        value=np.concatenate(value))
    print(out, os.path.getsize(out), "bytes,", len(index), "leaves")


if __name__ == "__main__":
    main()
