"""Generates tests/golden/reference_kernels.npz by RUNNING the reference's CUDA kernels (roi_align_kernel.cu,
nms_kernel.cu, highway_lstm_kernel.cu, compiled unmodified for sm_100a into oracle/_ref by oracle/Makefile) on the
inputs of the comparisons in tests/test_ops_gpu.py. Needs a CUDA device and oracle/_ref/libref_kernels.so; the tests
then compare against the stored results and need neither.
Outputs too large to store whole are kept as seeded samples (tests/test_ops_gpu.py:golden_sample), plus the SHA-256 of
the bit-exact RoIAlign forward and the per-plane sums of the RoIAlign backward.

    python tests/golden/make_golden_kernels.py [OUT_DIR]
"""
import ctypes
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "neural-motifs_b200")):
    sys.path.insert(0, p)

import torch  # noqa: E402

from oracle import ref_loader  # noqa: E402
from tests import test_ops_gpu as T  # noqa: E402


def main(out_dir):
    ref = ref_loader.ref_kernels()
    assert ref is not None, "run `make -C oracle` first"
    assert torch.cuda.is_available(), "the reference kernels need a CUDA device"
    cuda = torch.device("cuda:0")
    g = {}
    fwd, bwd = T.roi_align_launch(ref, *T.roi_align_reference_case(cuda))
    g["roi_fwd_sha256"] = np.array(hashlib.sha256(fwd.tobytes()).hexdigest())
    g["roi_fwd_sample"] = fwd.reshape(-1)[T.golden_sample(fwd.size, 4096, 1)]
    g["roi_bwd_sample"] = bwd.reshape(-1)[T.golden_sample(bwd.size, 8192, 2)]
    planes = bwd.reshape(bwd.shape[0] * bwd.shape[1], -1).astype(np.float64)
    g["roi_bwd_plane_sums"] = planes.sum(1)
    g["roi_bwd_plane_abs_sums"] = np.abs(planes).sum(1).astype(np.float32)
    for n, thr, boxes in T.nms_reference_cases():
        g["nms_keep_%d" % n] = T.nms_launch(ref, boxes, thr, cuda).astype(np.int32)
    cublas = ctypes.CDLL("libcublas.so.12")     # same SONAME the reference .so links: one instance
    handle = ctypes.c_void_p()
    assert cublas.cublasCreate_v2(ctypes.byref(handle)) == 0
    h, c, gates = T.lstm_launch(ref, handle, *T.lstm_reference_case(cuda))
    g["lstm_h"], g["lstm_c"] = h, c
    cg = T.lstm_covered_gates(gates)
    g["lstm_gates_sample"] = cg[T.golden_sample(cg.size, 8192, 3)]
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "reference_kernels.npz")
    np.savez_compressed(path, **g)
    print("wrote", path, {k: v.shape for k, v in g.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__)))
