"""Generates tests/golden/sdfgen/sdf_from_points_reference.npz (run from the repo root, on a CUDA device).

The reference's GT-SDF generator, compiled unmodified into oracle/_ref/nksr_sdfgen_ref.so by oracle/Makefile.ref, is
run on the inputs of tests/test_gpu_sdfgen.py with each of its argument sets; its output is stored at the test's fixed
sample of the queries, next to those queries (so that the test notices when the seeded inputs change).

    python tests/golden/make_sdfgen_golden.py [out.npz]
"""
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import test_gpu_sdfgen as T  # noqa: E402

REF_SO = os.path.join(ROOT, "oracle", "_ref", "nksr_sdfgen_ref.so")

if __name__ == "__main__":
    spec = importlib.util.spec_from_file_location("nksr_sdfgen_ref", REF_SO)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = {}
    for case in T.CASES:
        xyz, nrm, q = T._case(case)
        i = T.sample_indices(q.shape[0])
        out[f"{case}_q"] = q[i]
        for aid, kw in zip(T.ARG_IDS, T.ARGS):
            r = ref.sdf_from_points(t(q), t(xyz), t(nrm), kw["nb_points"], kw["stdv"], True, kw["imls"],
                                    kw["adaptive_knn"])
            out[f"{case}_{aid}_sdf"] = r[0].cpu().numpy()[i]
            out[f"{case}_{aid}_grad"] = r[1].cpu().numpy()[i]
    path = sys.argv[1] if len(sys.argv) > 1 else T.GOLDEN
    np.savez_compressed(path, **out)
    print(path, {k: v.shape for k, v in out.items()})
