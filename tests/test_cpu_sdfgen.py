"""oracle/sdfgen.py (restatement of ext/sdfgen/sdf_from_points.cu) on the CPU: analytic checks of the rule itself.
The comparison with the reference BINARY's stored output needs a GPU: tests/test_gpu_sdfgen.py."""
import os

import numpy as np

from oracle import sdfgen as OS
from tests import clouds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sdf_of_a_sphere():
    xyz, nrm = clouds.sphere(20_000, noise=0.0)
    rng = np.random.default_rng(0)
    q = rng.uniform(-0.7, 0.7, size=(5000, 3)).astype(np.float32)
    r = np.linalg.norm(q, axis=1)
    for kw in (dict(nb_points=8, stdv=0.02), dict(nb_points=8, stdv=3.0, adaptive_knn=8),
               dict(nb_points=16, stdv=0.05, imls=True)):
        sdf, grad = OS.sdf_from_points(q, xyz, nrm, compute_grad=True, **kw)
        far = np.abs(r - 0.35) > 0.02
        assert (np.sign(sdf[far]) == np.sign(r[far] - 0.35)).all()            # positive outside (outward normals)
        assert np.abs(np.abs(sdf) - np.abs(r - 0.35)).max() < 0.02
        radial = q / r[:, None]
        assert (np.sum(grad * radial, axis=1)[far] > 0.9).all()


def test_reference_build_recipe_exists_and_copies_nothing():
    """oracle/Makefile.ref compiles the reference sources WHERE THEY LIE (no copy in the repo) into oracle/_ref/"""
    mk = open(os.path.join(ROOT, "oracle", "Makefile.ref")).read()
    assert "/root/reference/ext" in mk and "_ref/nksr_sdfgen_ref.so" in mk
    for dirpath, _, files in os.walk(ROOT):
        if "/.git" in dirpath or "/oracle/_ref" in dirpath or "gpurun_out" in dirpath:
            continue
        assert "kdtree_cuda.cu" not in files and "sdf_from_points.cu" not in files
    assert "oracle/_ref/" in open(os.path.join(ROOT, ".gitignore")).read()
