"""Golden data for tests/test_oracle_cpu.py and tests/test_vocab_cpu.py, produced by the REFERENCE'S OWN CODE (run where
the reference tree is present, see oracle/refshim.py).  Each of those tests once imported the reference and compared
with it live; this runs the reference side of every such comparison on the tests' own seeded inputs and keeps what they
compare against in tests/golden/ref_pins.pt, so the comparisons run anywhere:

  * state-dict shapes, constructor keywords and prompt defaults of the reference modules, and facts read off its
    model configs (which keywords they pass);
  * reference outputs of the head, position embedding, LdmExtractor drivers and CLIP glue (large tensors as a fixed
    sample, oracle.cases.sample);
  * the label files the vocabulary is read from (copied to tests/golden/openseg_labels/) with SHA-256 digests of the
    reference's parse of them and of its prompt expansion.

    python tools/make_golden_pins.py
"""
import importlib
import inspect
import os
import re
import shutil
import sys
import types

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import cases, refshim  # noqa: E402
from oracle import clip as oclip  # noqa: E402
from oracle import ldm as oldm  # noqa: E402
import test_oracle_cpu as T  # noqa: E402  (the tests' seeded inputs)
import test_vocab_cpu as V  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
h = lambda t: t.detach().clone().to(torch.float32)
sample = lambda t, n=512: cases.sample(h(t), n)       # what the tests compare of a large output


def head(m, gold):
    pd, dec = refshim.ref_head(m)
    gold["head_state_shapes"] = {
        **{"sem_seg_head.pixel_decoder." + k: tuple(v.shape) for k, v in pd.state_dict().items()},
        **{"sem_seg_head.predictor." + k: tuple(v.shape) for k, v in dec.state_dict().items()}}
    sd, feats, (ms, mf), (me, te, ne, sizes) = T.head_inputs()
    pd.load_state_dict(refshim.strip(sd, "sem_seg_head.pixel_decoder."))
    dec.load_state_dict(refshim.strip(sd, "sem_seg_head.predictor."))
    mf_r, _, ms_r = pd.forward_features(feats)
    out = dec(ms, mf)
    logits = m.CategoryODISE.cal_pred_logits(None, dict(mask_embed=me, text_embed=te, null_embed=ne,
                                                        labels=[["x"] * n for n in sizes], logit_scale=out["logit_scale"]))
    gold["head"] = dict(mask_features=sample(mf_r), multi_scale=[sample(x) for x in ms_r],
                        **{k: sample(out[k]) for k in ("pred_masks", "mask_embed", "mask_pooled_features")},
                        logit_scale=h(out["logit_scale"]),
                        aux_pred_masks=[sample(a["pred_masks"]) for a in out["aux_outputs"]],
                        pred_logits=h(logits))
    gold["position_embedding"] = sample(m.PositionEmbeddingSine(128, normalize=True)(torch.zeros(2, 256, 7, 9)), 1024)
    kw = {}
    for name in ("MSDeformAttnPixelDecoder", "ODISEMultiScaleMaskedTransformerDecoder", "PooledMaskEmbed", "PseudoClassEmbed"):
        ref = getattr(m, name)
        kw[name] = [p for c in ref.__mro__ if c.__module__.startswith(("odise", "mask2former"))
                    for p in inspect.signature(c.__init__).parameters if p not in ("self", "kwargs", "args")]
    gold["constructor_keywords"] = kw
    od = m.odise_module
    gold["prompt_defaults"] = {c: inspect.signature(getattr(od, c).__init__).parameters["prompt"].default
                               for c in ("CategoryEmbed", "PoolingCLIPHead")}


def ldm_driver(gold):
    rl = importlib.import_module("odise.modeling.meta_arch.ldm")
    rl.timestep_embedding = oldm.timestep_embedding
    rl.DiagonalGaussianDistribution = oldm.DiagonalGaussianDistribution
    unet, x, ctx, cond, vae, img = T.ldm_driver_inputs()
    fake = types.SimpleNamespace(ldm=types.SimpleNamespace(unet=unet),
                                 unet_blocks=[unet.output_blocks[i] for i in oldm.UNET_TAP_BLOCKS])
    _, uf = rl.LdmExtractor.unet_forward(fake, x, torch.zeros(2, dtype=torch.long), ctx, cond_emb=cond.clone())
    enc_blocks = [vae.encoder.down[i].block[j] for i in range(4) for j in range(2)]
    dec_blocks = [vae.decoder.up[i].block[j] for i in reversed(range(4)) for j in range(3)]
    fake = types.SimpleNamespace(
        ldm=types.SimpleNamespace(encoder=vae.encoder, decoder=vae.decoder,
                                  ldm=types.SimpleNamespace(first_stage_model=vae, scale_factor=oldm.SCALE_FACTOR)),
        encoder_blocks=[enc_blocks[i] for i in oldm.ENC_TAP_BLOCKS],
        decoder_blocks=[dec_blocks[i] for i in oldm.DEC_TAP_BLOCKS])
    fake.encoder_forward = lambda im: rl.LdmExtractor.encoder_forward(fake, im)
    fake.decoder_forward = lambda z: rl.LdmExtractor.decoder_forward(fake, z)
    lat, ef = rl.LdmExtractor.encode_to_latent(fake, img)
    _, df = rl.LdmExtractor.decode_to_image(fake, lat)
    gold["ldm_driver"] = dict(unet_feats=[sample(t) for t in uf], latent=sample(lat),
                              enc_feats=[sample(t) for t in ef], dec_feats=[sample(t) for t in df])


def clip_glue(gold):
    rc = importlib.import_module("odise.modeling.meta_arch.clip")
    ro = importlib.import_module("odise.modeling.meta_arch.odise")
    import einops
    rc.rearrange = einops.rearrange
    v, img = T.clip_glue_inputs()
    emb, _ = rc.ClipAdapter._encode_image(types.SimpleNamespace(clip=types.SimpleNamespace(visual=v)), img)
    gold["clip_image_embed"] = h(emb)
    v, img, masks, text, labels = T.maskclip_inputs()
    fake = types.SimpleNamespace(clip=types.SimpleNamespace(visual=v), image_size=(56, 56),
                                 clip_preprocess=lambda im: oclip.preprocess(im, 56), logit_scale=torch.tensor(37.0))
    fake._mask_clip_forward = lambda *a: rc.MaskCLIP._mask_clip_forward(fake, *a)
    fake.encode_image_with_mask = lambda *a: rc.MaskCLIP.encode_image_with_mask(fake, *a)
    me = rc.MaskCLIP.get_mask_embed(fake, img, masks)
    gold["maskclip"] = dict(mask_embed=h(me), logits=h(rc.MaskCLIP.pred_logits(fake, me, text, labels)))
    test_labels, train_labels, cat_logits, clip_logits = T.ensemble_inputs()
    fake = types.SimpleNamespace(training=False, test_labels=test_labels, train_labels=train_labels, prompt="photo",
                                 with_bg=False, bg_labels=None, alpha=0.3, beta=0.7, normalize_logits=True,
                                 get_and_cache_test_text_embed=lambda labels: None,
                                 clip=lambda im, mk, t, l: {"mask_pred_open_logits": clip_logits})
    gold["ensemble"] = h(ro.PoolingCLIPHead.forward(fake, {"pred_open_logits": cat_logits.clone(), "images": torch.zeros(1),
                                                           "pred_masks": None})["pred_open_logits"])
    m, ids = T.encode_text_inputs()
    emb, enc = rc.ClipAdapter._encode_text(types.SimpleNamespace(clip=m), ids)
    gold["text_tower"] = dict(embed=h(emb), encodings=h(enc))


def configs(gold):
    def kwargs(name):
        return sorted(set(re.findall(r"(\w+)=", open(os.path.join(refshim.REF, "configs/common/models", name)).read())))
    gold["odise_with_label_keywords"] = kwargs("odise_with_label.py")
    cfg = open(os.path.join(refshim.REF, "configs/common/models/mask_generator_with_label.py")).read()
    gold["label_config"] = dict(category_head_sets_prompt="prompt=" in cfg.split("category_head=")[1].split("clip_head=")[0],
                                clip_head_is_default_pooling_clip_head="clip_head=L(PoolingCLIPHead)()" in cfg)


def labels(gold):
    rb = importlib.import_module("odise.data.build")
    od = importlib.import_module("odise.modeling.meta_arch.odise")
    src = os.path.join(refshim.REF, "odise", "data", "datasets", "openseg_labels")
    os.makedirs(V.LABELS, exist_ok=True)
    digests = {}
    for name, prompted in V.LABEL_FILES:
        shutil.copyfile(os.path.join(src, V.label_file(name, prompted)), os.path.join(V.LABELS, V.label_file(name, prompted)))
        ref = rb.get_openseg_labels(name, prompt_engineered=prompted)
        digests[V.label_file(name, prompted)] = V.digest(ref)
        if prompted:
            for p in V.PROMPTS:
                digests[f"{V.label_file(name, prompted)}:{p}"] = V.digest(rb.prompt_labels(ref, p))
    ade = rb.get_openseg_labels("ade20k_150", prompt_engineered=True)
    for c in ("CategoryEmbed", "PoolingCLIPHead"):
        p = gold["prompt_defaults"][c]
        digests[f"odise.prompt_labels:{c}"] = V.digest([s for group in od.prompt_labels(ade, p) for s in group])
    gold["label_digests"] = digests


@torch.no_grad()
def main():
    assert refshim.available(), "needs the reference tree (see oracle/refshim.py)"
    torch.set_num_threads(cases.GOLDEN_THREADS)                  # the bits of CPU reductions depend on it
    m = refshim.modules()
    gold = {}
    head(m, gold)
    ldm_driver(gold)
    clip_glue(gold)
    configs(gold)
    labels(gold)
    path = os.path.join(OUT, "ref_pins.pt")
    torch.save(gold, path)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
