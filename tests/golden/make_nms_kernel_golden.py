"""Generates tests/golden/nms_kernel_vectors.npz: the keep lists of the original project's CUDA NMS
(lib/nms/nms_kernel.cu, entry `_nms`, compiled unmodified into oracle/_ref/ by oracle.build.build_ref)
on the score-sorted proposal sets of tests/test_stages_gpu.py.  Needs a GPU and the compiled kernel;
test_stages_gpu.py::test_nms_host_vs_reference_kernel compares this repo's NMS against the stored lists.

    python tests/golden/make_nms_kernel_golden.py [out.npz]
"""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import build as OBUILD  # noqa: E402
from oracle import nms as ONMS  # noqa: E402
from test_stages_gpu import _proposal_case  # noqa: E402

SIZES = (1, 64, 65, 300, 2000, 6000)
THRESHOLDS = (0.3, 0.7)


def main(out):
    path = OBUILD.build_ref()
    if path is None or not os.path.exists(path):
        sys.exit("oracle/_ref/libref_gpu_nms.so not built")
    fn = getattr(ctypes.CDLL(path), "_Z4_nmsPiS_PKfiifi")
    ip, fp = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_float)
    fn.argtypes = [ip, ip, fp, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int]
    fn.restype = None
    rng = np.random.default_rng(99)
    vec = {}
    for n in SIZES:
        props, scores = _proposal_case(rng, n)
        dets = np.hstack([props, scores[:, None]]).astype(np.float32)
        sd = np.ascontiguousarray(dets[ONMS.argsort_desc(scores)])
        vec["dets_%d" % n] = sd
        for thr in THRESHOLDS:
            keep = np.empty(n, np.int32); num = ctypes.c_int(0)
            fn(keep.ctypes.data_as(ip), ctypes.byref(num), sd.ctypes.data_as(fp), n, 5, thr, 0)
            vec["keep_%d_%g" % (n, thr)] = keep[:num.value].copy()
    np.savez_compressed(out, **vec)
    print("wrote", out, {k: v.shape for k, v in vec.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "nms_kernel_vectors.npz"))
