"""Oracle vs golden vectors produced by the REFERENCE'S OWN CODE (tools/make_golden_ref.py, run where /root/reference is
mounted; fixtures committed under tests/golden/ref_*.pt).  Unlike tests/test_oracle_cpu.py these need no reference tree,
so the oracle stays pinned on the GPU box too.  Inputs: oracle/cases.py (seeded)."""
import os

import torch

from oracle import cases
from oracle import clip as oclip
from oracle import ldm as oldm
from oracle import m2f
from oracle import postprocess as opp

G = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return torch.load(os.path.join(G, name), map_location="cpu", weights_only=True)


def _close(a, b, rtol=1e-4, atol=1e-5):
    assert a.shape == b.shape
    assert torch.allclose(a.float(), b, rtol=rtol, atol=atol), (a.float() - b).abs().max().item()


@torch.no_grad()
def test_head_matches_reference_golden():
    ref = _load("ref_head.pt")
    sd, feats, sizes, te, ne = cases.head_case()
    mf, _, ms = m2f.pixel_decoder(sd, feats, "sem_seg_head.pixel_decoder.")
    _close(mf, ref["mask_features"])
    for a, b in zip(ms, ref["multi_scale"]):
        _close(a, b)
    # decoder from the REFERENCE's pixel-decoder outputs (isolates it; thresholds make it discontinuous otherwise)
    out, _ = m2f.transformer_decoder(sd, ref["multi_scale"], ref["mask_features"], "sem_seg_head.predictor.")
    for k in ("pred_masks", "mask_embed", "mask_pooled_features"):
        _close(out[k], ref[k], rtol=1e-3, atol=1e-4)
    _close(out["aux_outputs"][0]["pred_masks"], ref["aux0_pred_masks"], rtol=1e-3, atol=1e-4)
    assert torch.equal(out["logit_scale"].float(), ref["logit_scale"])
    _close(m2f.cal_pred_logits(ref["mask_embed"], te, ne, ref["logit_scale"], sizes), ref["pred_logits"], 1e-5, 1e-5)


@torch.no_grad()
def test_clip_glue_matches_reference_golden():
    ref = _load("ref_clip.pt")
    c = cases.clip_case()
    _close(oclip.encode_image(c["vis"], c["crop"]), ref["image_embed"], 1e-5, 1e-6)
    me = oclip.get_mask_embed(c["vis"], c["img"], c["masks"])
    _close(me, ref["mask_embed"], 1e-5, 1e-6)
    _close(oclip.maskclip_pred_logits(ref["mask_embed"], c["text"], [len(l) for l in c["labels"]], 37.0),
           ref["mask_logits"], 1e-5, 1e-5)
    emb, enc = oclip.encode_text(c["txt"], c["ids"])
    _close(emb, ref["text_embed"], 1e-5, 1e-6)
    _close(enc, ref["text_encodings"], 1e-5, 1e-6)
    _close(oclip.pooling_clip_ensemble(c["cat_logits"], c["clip_logits"], c["overlap"], 0.3, 0.7), ref["ensemble"], 1e-6, 1e-6)


@torch.no_grad()
def test_postprocess_matches_reference_golden():
    ref = _load("ref_postprocess.pt")
    cls, pred, K, things = cases.postprocess_case()
    assert torch.equal(opp.semantic_inference(cls, pred), ref["sem_seg"])
    pan, info = opp.panoptic_inference(cls, pred, K, things)
    assert torch.equal(pan, ref["panoptic_seg"]) and info == ref["segments_info"] and len(info) > 0


@torch.no_grad()
def test_ldm_drivers_match_reference_golden():
    ref = _load("ref_ldm_driver.pt")
    d = cases.ldm_case()
    with cases.golden_threads():                       # bit-exact: same reduction order as when the file was written
        feats = oldm.unet_features(d["unet"], d["x"], d["ctx"], d["cond"])
        lat, ef = oldm.encoder_features(d["vae"], d["img"])
        df = oldm.decoder_features(d["vae"], ref["latent"])
    for a, b in zip(feats, ref["unet_feats"]):
        assert torch.equal(a, b)
    assert torch.equal(lat, ref["latent"]) and all(torch.equal(a, b) for a, b in zip(ef, ref["enc_feats"]))
    assert len(df) == 2 and all(torch.equal(a, b) for a, b in zip(df, ref["dec_feats"]))
