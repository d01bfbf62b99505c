"""Seeded inputs of the golden-vector cases (TEST INFRASTRUCTURE ONLY): shared by tools/make_golden_ref.py, which runs
the REFERENCE's own code on them in the build container (/root/reference present) and commits the outputs under
tests/golden/ref_*.pt, and by tests/test_golden_cpu.py, which replays the oracle on the same inputs wherever the suite
runs (the GPU box has no /root/reference)."""
import contextlib

import torch

from odise_b200 import spec

# torch splits CPU reductions (convolutions, GEMMs, norms) over its intra-op threads, so the bits of a result depend on
# the thread count.  The golden files were written with this many threads; comparisons that must be bit-exact run with
# the same count (whatever the machine's core count).
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def sample(t, n=1024, seed=0):
    """A fixed, seeded sample of n elements of t, flattened (all of t when it has at most n): golden files keep this
    instead of a whole large tensor, and the tests take the same sample of what they compute."""
    flat = t.reshape(-1)
    if flat.numel() <= n:
        return flat.clone()
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n]
    return flat[idx.to(flat.device)]


def head_case():
    sd = spec.synth_state_dict(spec.head_params(), 1)
    g = torch.Generator().manual_seed(5)
    feats = {f"s{i}": torch.randn(1, 512, 64 // 2 ** i, 64 // 2 ** i, generator=g) for i in (2, 3, 4, 5)}
    sizes = [1, 3, 2, 1, 4] * 4
    te, ne = torch.randn(sum(sizes), 256, generator=g), torch.randn(1, 256, generator=g)
    return sd, feats, sizes, te, ne


def _init(module, seed, std):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * std)
    return module.eval()


def clip_case():
    from oracle import clip as oclip
    vis = _init(oclip.VisionTransformer(image_size=56, patch=14, width=128, layers=2, heads=2, out_dim=32), 11, 0.1)
    txt = _init(oclip.TextTransformer(vocab=50, ctx=9, width=64, layers=2, heads=2, out_dim=32), 12, 0.1)
    g = torch.Generator().manual_seed(13)
    img = torch.rand(2, 3, 96, 96, generator=g)
    crop = torch.randn(2, 3, 56, 56, generator=g)
    masks = torch.randn(2, 5, 24, 24, generator=g) * 3
    masks[0, 0] = -5.0
    text = torch.randn(7, 32, generator=g)
    labels = [["a", "b"], ["c"], ["d", "e", "f"], ["g"]]
    ids = torch.randint(1, 40, (3, 9), generator=g)
    ids[0, 4], ids[1, 8], ids[2, 2] = 49, 49, 49
    cat_logits, clip_logits = torch.randn(2, 6, 4, generator=g) * 4, torch.randn(2, 6, 4, generator=g) * 4
    return dict(vis=vis, txt=txt, img=img, crop=crop, masks=masks, text=text, labels=labels, ids=ids,
                cat_logits=cat_logits, clip_logits=clip_logits,
                test_labels=[["cat", "kitty"], ["unicorn"], ["dog"], ["spaceship", "rocket"]],
                train_labels=[["cat"], ["dog", "puppy"], ["tree"]], overlap=torch.tensor([1, 0, 1, 0]))


def postprocess_case():
    g = torch.Generator().manual_seed(4)
    Q, K, H, W = 30, 9, 40, 56
    cls = torch.randn(Q, K + 1, generator=g) * 3
    cls[:, -1] -= 2
    yy, xx = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    pred = torch.stack([(6 + 10 * torch.rand(1, generator=g) - ((yy - torch.rand(1, generator=g) * H) ** 2 +
                                                               (xx - torch.rand(1, generator=g) * W) ** 2).sqrt()) * 2
                        for _ in range(Q)])
    return cls, pred, K, [0, 2, 4]


def ldm_case():
    from oracle import ldm as oldm
    unet = _init(oldm.UNetModel(model_channels=64, num_heads=8, context_dim=48), 21, 0.05)
    vae = _init(oldm.AutoencoderKL(), 22, 0.03)
    g = torch.Generator().manual_seed(23)
    return dict(unet=unet, vae=vae, x=torch.randn(2, 4, 16, 16, generator=g), ctx=torch.randn(2, 5, 48, generator=g),
                cond=torch.randn(2, 256, generator=g), img=torch.randn(1, 3, 64, 64, generator=g))
