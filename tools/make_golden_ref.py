"""Golden vectors from the REFERENCE ITSELF (run in the build container, where /root/reference is mounted):
the reference's Mask2Former pixel decoder / ODISE decoder / cal_pred_logits, ClipAdapter / MaskCLIP / PoolingCLIPHead
glue, MaskFormer post-processing and LdmExtractor drivers are executed on the seeded inputs of oracle/cases.py and their
outputs written to tests/golden/ref_*.pt.  tests/test_golden_cpu.py replays the ORACLE against these files anywhere.

    python tools/make_golden_ref.py
"""
import importlib
import os
import sys
import types

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import cases, refshim  # noqa: E402
from oracle import ldm as oldm  # noqa: E402
from oracle import clip as oclip  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
h = lambda t: t.detach().clone().to(torch.float32)


@torch.no_grad()
def main():
    assert refshim.available(), "needs /root/reference"
    torch.set_num_threads(cases.GOLDEN_THREADS)                  # the bits of CPU reductions depend on it
    m = refshim.modules()
    # ---- Mask2Former pixel decoder + ODISE decoder + scoring
    sd, feats, sizes, te, ne = cases.head_case()
    pd, dec = refshim.ref_head(m)
    pd.load_state_dict(refshim.strip(sd, "sem_seg_head.pixel_decoder."))
    dec.load_state_dict(refshim.strip(sd, "sem_seg_head.predictor."))
    mf, _, ms = pd.forward_features(feats)
    out = dec(ms, mf)
    logits = m.CategoryODISE.cal_pred_logits(None, dict(mask_embed=out["mask_embed"], text_embed=te, null_embed=ne,
                                                        labels=[["x"] * n for n in sizes], logit_scale=out["logit_scale"]))
    torch.save(dict(mask_features=h(mf), multi_scale=[h(x) for x in ms], pred_masks=h(out["pred_masks"]),
                    mask_embed=h(out["mask_embed"]), mask_pooled_features=h(out["mask_pooled_features"]),
                    logit_scale=h(out["logit_scale"]), aux0_pred_masks=h(out["aux_outputs"][0]["pred_masks"]),
                    pred_logits=h(logits)), os.path.join(OUT, "ref_head.pt"))
    # ---- CLIP glue: image embed, MaskCLIP, text tower, PoolingCLIPHead
    rc = importlib.import_module("odise.modeling.meta_arch.clip")
    ro = importlib.import_module("odise.modeling.meta_arch.odise")
    import einops
    rc.rearrange = einops.rearrange
    c = cases.clip_case()
    fake = types.SimpleNamespace(clip=types.SimpleNamespace(visual=c["vis"]), image_size=(56, 56),
                                 clip_preprocess=lambda im: oclip.preprocess(im, 56), logit_scale=torch.tensor(37.0))
    fake._mask_clip_forward = lambda *a: rc.MaskCLIP._mask_clip_forward(fake, *a)
    fake.encode_image_with_mask = lambda *a: rc.MaskCLIP.encode_image_with_mask(fake, *a)
    img_emb, _ = rc.ClipAdapter._encode_image(fake, c["crop"])
    mask_emb = rc.MaskCLIP.get_mask_embed(fake, c["img"], c["masks"])
    mask_lg = rc.MaskCLIP.pred_logits(fake, mask_emb, c["text"], c["labels"])
    text_emb, text_enc = rc.ClipAdapter._encode_text(types.SimpleNamespace(clip=c["txt"]), c["ids"])
    fh = types.SimpleNamespace(training=False, test_labels=c["test_labels"], train_labels=c["train_labels"], prompt="photo",
                               with_bg=False, bg_labels=None, alpha=0.3, beta=0.7, normalize_logits=True,
                               get_and_cache_test_text_embed=lambda labels: None,
                               clip=lambda im, mk, t, l: {"mask_pred_open_logits": c["clip_logits"]})
    ens = ro.PoolingCLIPHead.forward(fh, {"pred_open_logits": c["cat_logits"].clone(), "images": torch.zeros(1),
                                          "pred_masks": None})["pred_open_logits"]
    torch.save(dict(image_embed=h(img_emb), mask_embed=h(mask_emb), mask_logits=h(mask_lg), text_embed=h(text_emb),
                    text_encodings=h(text_enc), ensemble=h(ens)), os.path.join(OUT, "ref_clip.pt"))
    # ---- MaskFormer post-processing
    MF = importlib.import_module("mask2former.maskformer_model").MaskFormer
    cls, pred, K, things = cases.postprocess_case()
    fk = types.SimpleNamespace(sem_seg_head=types.SimpleNamespace(num_classes=K), object_mask_threshold=0.0,
                               overlap_threshold=0.8, num_queries=cls.shape[0], test_topk_per_image=10, panoptic_on=True,
                               metadata=types.SimpleNamespace(thing_dataset_id_to_contiguous_id={i: t for i, t in enumerate(things)}))
    pan, info = MF.panoptic_inference(fk, cls, pred)
    torch.save(dict(sem_seg=h(MF.semantic_inference(fk, cls, pred)), panoptic_seg=pan.to(torch.int32), segments_info=info),
               os.path.join(OUT, "ref_postprocess.pt"))
    # ---- LdmExtractor drivers on the oracle UNet / VAE modules
    rl = importlib.import_module("odise.modeling.meta_arch.ldm")
    rl.timestep_embedding = oldm.timestep_embedding
    rl.DiagonalGaussianDistribution = oldm.DiagonalGaussianDistribution
    d = cases.ldm_case()
    unet, vae = d["unet"], d["vae"]
    fu = types.SimpleNamespace(ldm=types.SimpleNamespace(unet=unet),
                               unet_blocks=[unet.output_blocks[i] for i in oldm.UNET_TAP_BLOCKS])
    _, uf = rl.LdmExtractor.unet_forward(fu, d["x"], torch.zeros(2, dtype=torch.long), d["ctx"], cond_emb=d["cond"].clone())
    enc_blocks = [vae.encoder.down[i].block[j] for i in range(4) for j in range(2)]
    dec_blocks = [vae.decoder.up[i].block[j] for i in reversed(range(4)) for j in range(3)]
    fv = types.SimpleNamespace(
        ldm=types.SimpleNamespace(encoder=vae.encoder, decoder=vae.decoder,
                                  ldm=types.SimpleNamespace(first_stage_model=vae, scale_factor=oldm.SCALE_FACTOR)),
        encoder_blocks=[enc_blocks[i] for i in oldm.ENC_TAP_BLOCKS], decoder_blocks=[dec_blocks[i] for i in oldm.DEC_TAP_BLOCKS])
    fv.encoder_forward = lambda im: rl.LdmExtractor.encoder_forward(fv, im)
    fv.decoder_forward = lambda z: rl.LdmExtractor.decoder_forward(fv, z)
    lat, ef = rl.LdmExtractor.encode_to_latent(fv, d["img"])
    _, df = rl.LdmExtractor.decode_to_image(fv, lat)
    torch.save(dict(unet_feats=[h(x) for x in uf], latent=h(lat), enc_feats=[h(x) for x in ef], dec_feats=[h(x) for x in df]),
               os.path.join(OUT, "ref_ldm_driver.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
