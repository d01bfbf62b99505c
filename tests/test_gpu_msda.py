"""GPU parity of odise_msda_forward_f32 / odise_msda_fused_f32 against the CPU oracle (oracle/msda.py) and the
committed golden vectors, mirroring the reference's own test (ops/test.py:24-63: kernel vs PyTorch restatement,
fp32 rtol 1e-2 / atol 1e-3 -- we hold 1e-5 absolute on O(1) data)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _problem(seed, N, M, D, shapes, Lq, P, spread=1.0):
    g = torch.Generator().manual_seed(seed)
    ss = torch.as_tensor(shapes, dtype=torch.long)
    lsi = torch.cat((ss.new_zeros((1,)), ss.prod(1).cumsum(0)[:-1]))
    S = int(ss.prod(1).sum())
    L = len(shapes)
    value = torch.rand(N, S, M, D, generator=g) * 0.01 if spread == 1.0 else torch.randn(N, S, M, D, generator=g)
    loc = torch.rand(N, Lq, M, L, P, 2, generator=g) * spread - (spread - 1) / 2
    aw = torch.rand(N, Lq, M, L, P, generator=g) + 1e-5
    aw = aw / aw.sum(-1, keepdim=True).sum(-2, keepdim=True)
    return value, ss, lsi, loc, aw


@pytest.mark.parametrize("cfg", [
    dict(seed=3, N=1, M=2, D=2, shapes=[(6, 4), (3, 2)], Lq=2, P=2),                 # ops/test.py:24-31
    dict(seed=4, N=2, M=8, D=32, shapes=[(16, 16), (32, 32), (64, 64)], Lq=5376, P=4, spread=1.5),  # 512^2 release
    dict(seed=5, N=1, M=8, D=32, shapes=[(32, 32), (64, 64), (128, 128)], Lq=21504, P=4, spread=1.2),  # 1024^2
    dict(seed=6, N=3, M=4, D=64, shapes=[(7, 5), (3, 9)], Lq=11, P=3, spread=2.0),
    dict(seed=8, N=2, M=8, D=32, shapes=[(16, 16), (32, 32), (64, 64), (128, 128)], Lq=300, P=4, spread=1.4),  # C4: L = 4
    dict(seed=9, N=1, M=8, D=32, shapes=[(9, 7), (5, 3)], Lq=37, P=3, spread=2.5),   # L*P = 6: ragged sub-warp, tail block
    dict(seed=10, N=2, M=5, D=32, shapes=[(4, 4)] * 8, Lq=19, P=4, spread=1.1),       # L*P = 32: a full warp per pair
    dict(seed=7, N=1, M=3, D=30, shapes=[(5, 5)], Lq=4, P=1),                          # scalar path (D % 4 != 0)
])
def test_msda_vs_oracle(cuda, cfg):
    from odise_b200 import lib
    from oracle.msda import msda_forward
    value, ss, lsi, loc, aw = _problem(**cfg)
    ref = msda_forward(value, ss, lsi, loc, aw)
    out = lib.msda_forward(value.to(cuda), ss.to(cuda), lsi.to(cuda), loc.to(cuda), aw.to(cuda), 128)
    assert out.shape == ref.shape
    err = (out.cpu() - ref).abs().max().item()
    assert err < 1e-5 * max(1.0, ref.abs().max().item()), err


def test_msda_fused_vs_oracle(cuda):
    """odise_msda_fused_f32 (raw sampling_offsets / attention logits + reference points, ms_deform_attn.py:98-113) on the
    D = 32 shared-memory kernel, L = 3 (ODISE pixel decoder) and L = 4 (C4 microbench / the op's default)."""
    from odise_b200 import ops
    from oracle.msda import msda_forward
    for seed, shapes in ((11, [(8, 8), (16, 16), (32, 32)]), (12, [(4, 6), (8, 12), (16, 24), (32, 48)])):
        g = torch.Generator().manual_seed(seed)
        N, M, D, P, L = 2, 8, 32, 4, len(shapes)
        ss = torch.as_tensor(shapes, dtype=torch.long)
        lsi = torch.cat((ss.new_zeros((1,)), ss.prod(1).cumsum(0)[:-1]))
        S = int(ss.prod(1).sum())
        value = torch.randn(N, S, M, D, generator=g)
        offs = torch.randn(N, S, M, L, P, 2, generator=g) * 3
        logits = torch.randn(N, S, M, L * P, generator=g) * 2
        ref_pts = torch.rand(N, S, L, 2, generator=g)
        norm = torch.stack([ss[:, 1], ss[:, 0]], -1).float()                           # (W, H)
        loc = ref_pts[:, :, None, :, None, :] + offs / norm[None, None, None, :, None, :]
        aw = logits.softmax(-1).view(N, S, M, L, P)
        want = msda_forward(value, ss, lsi, loc, aw)
        o32, pl = ops.msda_fused(value.to(cuda), ss.to(cuda), lsi.to(cuda), ref_pts.to(cuda), offs.to(cuda).contiguous(),
                                 logits.to(cuda), N, S, M, D, L, S, P, want_f32=True)
        assert (o32.view(N, S, -1).cpu() - want).abs().max().item() < 2e-5 * max(1.0, want.abs().max().item())
        assert (pl.float().view(N, S, -1).cpu() - want).abs().max().item() < 1e-4 * max(1.0, want.abs().max().item())


REFKERNEL_CASES = (dict(seed=4, N=2, M=8, D=32, shapes=[(16, 16), (32, 32), (64, 64)], Lq=5376, P=4, spread=1.5),
                   dict(seed=8, N=2, M=8, D=32, shapes=[(16, 16), (32, 32), (64, 64), (128, 128)], Lq=300, P=4, spread=1.4),
                   dict(seed=6, N=3, M=4, D=64, shapes=[(7, 5), (3, 9)], Lq=11, P=3, spread=2.0))


def test_msda_vs_reference_kernel(cuda):
    """Same inputs as the REFERENCE's own CUDA kernel compiled for sm_100a (ops/src/cuda/ms_deform_im2col_cuda.cuh behind
    oracle/ref_msda_host.cu) was given by tools/make_golden_refkernel.py, which stored a fixed sample of its outputs and
    the sum of every output row in tests/golden/refkernel_msda.pt: fp32, only the summation order differs.  A row sum
    holds M x D elements, so its bound is M x D times the element bound."""
    from odise_b200 import lib
    from oracle import cases
    gold = torch.load(os.path.join(GOLD, "refkernel_msda.pt"), weights_only=True)
    assert len(gold["samples"]) == len(REFKERNEL_CASES)
    for cfg, want, rows, amax in zip(REFKERNEL_CASES, gold["samples"], gold["row_sums"], gold["absmax"]):
        value, ss, lsi, loc, aw = (t.to(cuda) for t in _problem(**cfg))
        got = lib.msda_forward(value, ss, lsi, loc, aw, 128)
        torch.cuda.synchronize()
        assert abs(got.abs().max().item() - amax) < 1e-5 * max(1.0, amax)
        tol = 1e-5 * max(1.0, amax)
        assert (cases.sample(got, want.numel()).cpu() - want).abs().max().item() < tol
        assert rows.shape == got.shape[:-1]
        assert (got.double().sum(-1).cpu() - rows.double()).abs().max().item() < tol * got.shape[-1]


def test_msda_golden(cuda):
    from odise_b200 import lib
    for name in sorted(os.listdir(GOLD)):
        if not name.startswith("msda_"):
            continue
        d = torch.load(os.path.join(GOLD, name))
        out = lib.msda_forward(d["value"].to(cuda), d["spatial_shapes"].to(cuda), d["level_start_index"].to(cuda),
                               d["sampling_locations"].to(cuda), d["attention_weights"].to(cuda), 128)
        assert torch.allclose(out.cpu(), d["output"], rtol=1e-4, atol=1e-6), name


def test_msda_errors(cuda):
    from odise_b200 import lib
    value, ss, lsi, loc, aw = _problem(3, 1, 2, 4, [(6, 4)], 2, 2)
    with pytest.raises(RuntimeError):   # CPU tensors: reference raises "Not implemented on the CPU"
        lib.msda_forward(value, ss, lsi, loc, aw, 128)
    with pytest.raises(RuntimeError):   # non-contiguous (reference .cu:33)
        lib.msda_forward(value.to(cuda).transpose(2, 3), ss, lsi, loc.to(cuda), aw.to(cuda), 128)
