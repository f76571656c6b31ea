"""Generates tests/golden/ds_utils_vectors.npz by running the original project's lib/datasets/ds_utils.py
(importable on its own: numpy only) on seeded boxes with duplicates.  tests/test_datasets.py compares this
repo's datasets.ds_utils against the stored outputs.

    python tests/golden/make_ds_utils_golden.py <checkout of the original tf-faster-rcnn>
"""
import importlib.util
import os
import sys

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ds_utils_vectors.npz")


def main(ref_root):
    spec = importlib.util.spec_from_file_location("ref_ds_utils", os.path.join(ref_root, "lib", "datasets", "ds_utils.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    rng = np.random.default_rng(5)
    b = rng.integers(0, 40, (200, 4)).astype(np.float64)
    b[:, 2:] += b[:, :2]
    b = np.vstack([b, b[:50]])
    out = {"boxes": b,
           "unique": np.asarray(ref.unique_boxes(b)), "unique_0.25": np.asarray(ref.unique_boxes(b, 0.25)),
           "xywh_to_xyxy": ref.xywh_to_xyxy(b), "xyxy_to_xywh": ref.xyxy_to_xywh(b),
           "filter_small_12": np.asarray(ref.filter_small_boxes(b, 12))}
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
