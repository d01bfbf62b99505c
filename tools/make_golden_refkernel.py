"""Golden outputs of the REFERENCE's own MSDeformAttn CUDA kernel (oracle/_ref/libref_msda.so, built by oracle/Makefile
from the reference tree) on the problems of tests/test_gpu_msda.py::test_msda_vs_reference_kernel.  Needs a GPU and the
built library; writes a fixed sample of each output (oracle.cases.sample), the sum of every output row (over the M x D
channels of one query, so that every element is covered) and the largest magnitude, so that the test compares the B200
kernel with the reference kernel without the reference kernel being present.

    python tools/make_golden_refkernel.py [OUT]        # default OUT: tests/golden/refkernel_msda.pt
"""
import os
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import cases, refmsda  # noqa: E402
import test_gpu_msda as T  # noqa: E402

SAMPLE = 6144                      # elements kept of each output, besides its row sums


@torch.no_grad()
def main(out):
    assert refmsda.available(), "oracle/_ref/libref_msda.so not built"
    dev = torch.device("cuda:0")
    samples, row_sums, absmax = [], [], []
    for cfg in T.REFKERNEL_CASES:
        value, ss, lsi, loc, aw = (t.to(dev) for t in T._problem(**cfg))
        want = refmsda.forward(value, ss, lsi, loc, aw, 128)
        torch.cuda.synchronize()
        samples.append(cases.sample(want, SAMPLE).cpu())
        row_sums.append(want.double().sum(-1).float().cpu())
        absmax.append(want.abs().max().item())
        print(cfg, tuple(want.shape), absmax[-1])
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    torch.save(dict(samples=samples, row_sums=row_sums, absmax=absmax), out)
    print(out, os.path.getsize(out))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "refkernel_msda.pt"))
