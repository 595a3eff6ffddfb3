"""Generate tests/golden/ref_boundary_sampling.npz: what the reference's own boundary stage returns.

For every case of tests/boundary_oracle.py (seeded dental arches of 30 000, 100 000 and 200 000 vertices with 24 000
labelled sampled points, and a 24 000-vertex single-label mesh) this imports the reference's
``inference_pipelines.inference_pipeline_tgn`` on CPU (I/O packages stubbed as oracle/ref_models.py does, its
``gen_utils.fps`` served by the oracle's C restatement of the reference FPS kernel, which is pinned bitwise against the
verbatim kernel), builds an ``InferencePipeLine`` without its networks (``__new__`` + the ``boundary_sampling_info`` of
inference_pipeline_maker.py:56-60), and calls ``get_boundary_sampled_feats`` under ``np.random.seed(SEEDS[case])``.

Stored per case: the four outputs through ``oracle.golden.pack`` (digests of large arrays), the number of boundary
vertices ``n_bd`` (before the 20 000 cap), one ``np.random.random()`` drawn after the call (pins the RNG consumption),
or ``raises = 1`` when the method raised TypeError (the FPS refusal of gen_utils.fps).

    python tests/golden/make_ref_boundary_golden.py
"""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import boundary_oracle as B  # noqa: E402
from oracle import golden, ref_models  # noqa: E402

OUT_KEYS = ("results_feat", "results_label", "bd_feat", "bd_label")


def main():
    world = ref_models.World("reference", cpu_dry_run=True)
    out = {}
    with world:
        tgn = importlib.import_module("inference_pipelines.inference_pipeline_tgn")
        gu = world.mod("gen_utils")
        gu.fps = B._fps
        pipe = tgn.InferencePipeLine.__new__(tgn.InferencePipeLine)
        pipe.config = {"boundary_sampling_info": dict(B.BOUNDARY_INFO)}
        for name in B.CASES:
            labels, org, sampled = B.boundary_case(name)
            tree = tgn.KDTree(sampled[:, :3].copy(), leaf_size=40)          # n_bd as the method computes it (:293-300)
            near = tree.query(org[:, :3], k=40, return_distance=False)
            n_bd = int((gu.count_unique_by_row(labels[near])[:, 0] / 40. < B.BOUNDARY_INFO["bdl_ratio"]).sum())
            out[f"{name}.n_bd"] = np.asarray(n_bd, np.int64)
            np.random.seed(B.SEEDS[name])
            try:
                res = pipe.get_boundary_sampled_feats(labels, org, sampled, None)
            except TypeError:
                out[f"{name}.raises"] = np.asarray(1, np.int64)
            else:
                for key, a in zip(OUT_KEYS, res):
                    out.update(golden.pack(f"{name}.{key}", a))
            out[f"{name}.post_random"] = np.asarray(np.random.random(), np.float64)
            print(name, "n_bd", n_bd, "taken", None if f"{name}.raises" in out else res[2].shape[0])
    for name in list(sys.modules):
        if name.split(".")[0] == "inference_pipelines":
            del sys.modules[name]
    np.savez_compressed(os.path.join(HERE, "ref_boundary_sampling.npz"), **out)


if __name__ == "__main__":
    main()
