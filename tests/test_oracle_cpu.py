"""CPU tests that PIN the oracle (oracle/) against the reference's own code, and check the parameter inventory of
odise_b200/spec.py.  What the reference computed on these tests' inputs (see the *_inputs functions) is stored in
tests/golden/ref_pins.pt by tools/make_golden_pins.py, so the tests need no reference tree."""
import os

import torch

from odise_b200 import spec
from oracle import cases
from oracle import ldm as oldm
from oracle import m2f


def _pins():
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", "ref_pins.pt"), weights_only=True)


def _shapes(params, prefix):
    return {n[len(prefix):]: tuple(s) for n, s, _ in params}


def test_unet_and_vae_inventory_matches_oracle_modules():
    with torch.device("meta"):
        unet, vae = oldm.UNetModel(), oldm.AutoencoderKL()
    assert _shapes(spec.unet_params(), spec.UNET_PREFIX) == {k: tuple(v.shape) for k, v in unet.state_dict().items()}
    assert _shapes(spec.vae_params(), spec.VAE_PREFIX) == {k: tuple(v.shape) for k, v in vae.state_dict().items()}
    n = sum(torch.Size(s).numel() for _, s, _ in spec.unet_params())
    assert n == 859_520_964          # the published SD-v1 UNet parameter count
    assert sum(torch.Size(s).numel() for _, s, _ in spec.vae_params()) == 83_653_863


def test_tap_table():
    """reset_dim_stride expectations of the reference (ldm.py:284-346): tap channels / strides."""
    inp, mid, out = spec.unet_blocks()
    assert [out[i][0][1] for i in (2, 5, 8, 11)] == [2560, 1920, 960, 640]
    assert spec.FEATURE_DIMS == (512, 512, 2560, 1920, 960, 640, 512, 512)


def _head_sd(seed=0):
    return spec.synth_state_dict(spec.head_params(), seed)


def test_head_inventory_matches_reference_modules():
    got = {n: tuple(s) for n, s, _ in spec.pixel_decoder_params() + spec.decoder_params()}
    assert got == _pins()["head_state_shapes"]


def head_inputs():
    """Seeded inputs of the head check: weights, backbone features for the pixel decoder, inputs of the decoder (drawn
    on their own, so the decoder check does not ride on the pixel decoder's rounding: its mask thresholds make it
    discontinuous) and of the scoring."""
    sd = _head_sd(1)
    g = torch.Generator().manual_seed(5)
    feats = {f"s{i}": torch.randn(2, 512, 128 // 2 ** i, 128 // 2 ** i, generator=g) for i in (2, 3, 4, 5)}
    ms = [torch.randn(2, 256, 128 // s, 128 // s, generator=g) for s in (32, 16, 8)]
    mf = torch.randn(2, 256, 32, 32, generator=g)
    sizes = [1, 3, 2, 1, 4] * 4
    me = torch.randn(2, 100, 256, generator=g)
    te = torch.randn(sum(sizes), 256, generator=g)
    ne = torch.randn(1, 256, generator=g)
    return sd, feats, (ms, mf), (me, te, ne, sizes)


def _close(a, b, rtol, atol):
    a = cases.sample(a, b.numel())
    assert a.shape == b.shape and torch.allclose(a, b, rtol=rtol, atol=atol), (a - b).abs().max().item()


@torch.no_grad()
def test_head_oracle_equals_reference():
    """Pixel decoder, decoder and CategoryODISE.cal_pred_logits against the reference's outputs (fixed samples)."""
    ref = _pins()["head"]
    sd, feats, (ms, mf), (me, te, ne, sizes) = head_inputs()
    mf_o, t_o, ms_o = m2f.pixel_decoder(sd, feats, "sem_seg_head.pixel_decoder.")
    _close(mf_o, ref["mask_features"], 1e-4, 1e-5)
    assert len(ms_o) == len(ref["multi_scale"])
    for a, b in zip(ms_o, ref["multi_scale"]):
        _close(a, b, 1e-4, 1e-5)
    out_o, _ = m2f.transformer_decoder(sd, ms, mf, "sem_seg_head.predictor.")
    for k in ("pred_masks", "mask_embed", "mask_pooled_features"):
        _close(out_o[k], ref[k], 1e-3, 1e-4)
    assert torch.equal(out_o["logit_scale"], ref["logit_scale"])
    assert len(out_o["aux_outputs"]) == len(ref["aux_pred_masks"])
    for a, b in zip(out_o["aux_outputs"], ref["aux_pred_masks"]):
        _close(a["pred_masks"], b, 1e-3, 1e-4)
    mine = m2f.cal_pred_logits(me, te, ne, out_o["logit_scale"], sizes)
    assert torch.allclose(mine, ref["pred_logits"], rtol=1e-5, atol=1e-5)


@torch.no_grad()
def test_position_embedding_and_msdeformattn_equal_reference():
    _close(m2f.position_embedding_sine(2, 7, 9), _pins()["position_embedding"], 0, 1e-6)


def ldm_driver_inputs():
    torch.manual_seed(0)
    unet = oldm.UNetModel(model_channels=64, num_heads=8, context_dim=48).eval()
    for p in unet.parameters():
        torch.nn.init.normal_(p, std=0.05)
    x, ctx = torch.randn(2, 4, 16, 16), torch.randn(2, 5, 48)
    cond = torch.randn(2, 256)
    vae = oldm.AutoencoderKL().eval()
    img = torch.randn(1, 3, 64, 64)
    return unet, x, ctx, cond, vae, img


@torch.no_grad()
def test_reference_ldm_driver_runs_on_oracle_unet():
    """The reference's LdmExtractor.unet_forward / encoder_forward / decoder_forward (ldm.py:424-533) executed
    VERBATIM on the oracle modules == oracle.ldm.unet_features / encoder_features / decoder_features (fixed samples)."""
    ref = _pins()["ldm_driver"]
    unet, x, ctx, cond, vae, img = ldm_driver_inputs()
    with cases.golden_threads():                       # bit-exact: same reduction order as when the file was written
        mine = oldm.unet_features(unet, x, ctx, cond)
        lat_o, ef_o = oldm.encoder_features(vae, img)
        df_o = oldm.decoder_features(vae, lat_o)
    assert len(mine) == len(ref["unet_feats"]) == 4
    for a, b in zip(mine, ref["unet_feats"]):
        assert torch.equal(cases.sample(a, b.numel()), b)
    assert len(ef_o) == len(ref["enc_feats"])
    assert torch.equal(cases.sample(lat_o, ref["latent"].numel()), ref["latent"])
    assert all(torch.equal(cases.sample(a, b.numel()), b) for a, b in zip(ef_o, ref["enc_feats"]))
    assert len(df_o) == len(ref["dec_feats"]) == 2
    assert all(torch.equal(cases.sample(a, b.numel()), b) for a, b in zip(df_o, ref["dec_feats"]))


def test_q_sample_constants():
    a, b = oldm.SQRT_ALPHA_BAR_0, oldm.SQRT_ONE_MINUS_ALPHA_BAR_0
    assert abs(a - 0.999575) < 1e-6 and abs(b - 0.029155) < 1e-6   # SURVEY.md §8a row a6
    n = oldm.shared_noise()
    assert n.shape == (1, 4, 64, 64)


def test_clip_inventory_matches_oracle_module():
    from oracle import clip as oclip
    with torch.device("meta"):
        v = oclip.VisionTransformer()
    got = {n[len(spec.CLIP_PREFIX):]: tuple(s) for n, s, _ in spec.clip_visual_params()}
    assert got == {k: tuple(t.shape) for k, t in v.state_dict().items()}
    assert 303e6 < sum(torch.Size(s).numel() for s in got.values()) < 305e6      # ViT-L/14-336 image tower


def clip_glue_inputs():
    from oracle import clip as oclip
    torch.manual_seed(0)
    v = oclip.VisionTransformer(image_size=56, patch=14, width=64, layers=2, heads=4, out_dim=32).eval()
    for p in v.parameters():
        torch.nn.init.normal_(p, std=0.1)
    return v, torch.randn(2, 3, 56, 56)


@torch.no_grad()
def test_reference_clip_glue_runs_on_oracle_visual():
    """ClipAdapter._encode_image (clip.py:177-222) executed verbatim on the oracle VisionTransformer == oracle.encode_image."""
    from oracle import clip as oclip
    v, img = clip_glue_inputs()
    emb_ref = _pins()["clip_image_embed"]
    assert torch.allclose(emb_ref, oclip.encode_image(v, img), rtol=1e-5, atol=1e-6)


def maskclip_inputs():
    from oracle import clip as oclip
    torch.manual_seed(1)
    v = oclip.VisionTransformer(image_size=56, patch=14, width=128, layers=2, heads=2, out_dim=32).eval()
    for p in v.parameters():
        torch.nn.init.normal_(p, std=0.1)
    img = torch.rand(2, 3, 96, 96)
    masks = torch.randn(2, 5, 24, 24) * 3
    masks[0, 0] = -5.0                                         # a query whose mask touches no patch at all
    text = torch.randn(7, 32)
    labels = [["a", "b"], ["c"], ["d", "e", "f"], ["g"]]
    return v, img, masks, text, labels


@torch.no_grad()
def test_reference_maskclip_runs_on_oracle_visual():
    """MaskCLIP.get_mask_embed / pred_logits (clip.py:252-351, logit scale 37) executed verbatim on the oracle
    VisionTransformer."""
    from oracle import clip as oclip
    v, img, masks, text, labels = maskclip_inputs()
    ref = _pins()["maskclip"]
    got = oclip.get_mask_embed(v, img, masks)
    assert ref["mask_embed"].shape == (2, 5, 32) and torch.allclose(ref["mask_embed"], got, rtol=1e-5, atol=1e-6)
    lo = oclip.maskclip_pred_logits(got, text, [len(l) for l in labels], torch.tensor(37.0))
    assert torch.allclose(ref["logits"], lo, rtol=1e-5, atol=1e-5)


def ensemble_inputs():
    torch.manual_seed(2)
    test_labels = [["cat", "kitty"], ["unicorn"], ["dog"], ["spaceship", "rocket"]]
    train_labels = [["cat"], ["dog", "puppy"], ["tree"]]
    cat_logits, clip_logits = torch.randn(2, 6, 4) * 4, torch.randn(2, 6, 4) * 4
    return test_labels, train_labels, cat_logits, clip_logits


@torch.no_grad()
def test_reference_pooling_clip_head_ensemble():
    """PoolingCLIPHead.forward (odise.py:1469-1542, alpha 0.3, beta 0.7, prompt "photo") run verbatim with a stubbed
    MaskCLIP == oracle ensemble."""
    from oracle import clip as oclip
    test_labels, train_labels, cat_logits, clip_logits = ensemble_inputs()
    ov = torch.tensor([1, 0, 1, 0])
    got = oclip.pooling_clip_ensemble(cat_logits, clip_logits, ov, 0.3, 0.7)
    assert torch.allclose(_pins()["ensemble"], got, rtol=1e-6, atol=1e-6)
    full = torch.randn(2, 6, 5)
    merged = oclip.merge_with_void(full, got)
    assert torch.allclose(merged.exp().sum(-1), torch.ones(2, 6) + 5e-8, atol=1e-5)


def test_clip_text_inventory_matches_oracle_module():
    from oracle import clip as oclip
    with torch.device("meta"):
        t = oclip.TextTransformer()
    got = {n[len(spec.CLIP_TEXT_PREFIX):]: tuple(s) for n, s, _ in spec.clip_text_params()}
    assert got == {k: tuple(v.shape) for k, v in t.state_dict().items()}
    # the SD-v1 cond_stage_model (HF names) maps onto the same module minus projection / logit_scale
    hf = spec.synth_state_dict(spec.sd_text_params(width=64, layers=2, vocab=100), 0)
    conv = spec.hf_text_to_openai(hf, dst_prefix="")
    small = oclip.TextTransformer(vocab=100, width=64, layers=2, heads=2, out_dim=64)
    missing = set(small.state_dict()) - set(conv)
    assert missing == {"text_projection", "logit_scale"} and not (set(conv) - set(small.state_dict()))


def encode_text_inputs():
    from oracle import clip as oclip
    torch.manual_seed(3)
    m = oclip.TextTransformer(vocab=50, ctx=9, width=64, layers=2, heads=2, out_dim=32).eval()
    for p in m.parameters():
        torch.nn.init.normal_(p, std=0.1)
    ids = torch.randint(1, 40, (3, 9))
    ids[0, 4], ids[1, 8], ids[2, 2] = 49, 49, 49                          # EOT = highest id
    return m, ids


@torch.no_grad()
def test_reference_encode_text_runs_on_oracle_text_tower():
    """ClipAdapter._encode_text (clip.py:138-152) executed verbatim on the oracle TextTransformer == oracle.encode_text."""
    from oracle import clip as oclip
    m, ids = encode_text_inputs()
    ref = _pins()["text_tower"]
    emb_ref, enc_ref = ref["embed"], ref["encodings"]
    emb, enc = oclip.encode_text(m, ids)
    assert torch.allclose(emb_ref, emb, rtol=1e-5, atol=1e-6) and torch.allclose(enc_ref, enc, rtol=1e-5, atol=1e-6)


def test_plugin_surface_matches_reference_modules():
    """SURVEY §8b B-1 / B-2: the B200 plugin classes take the constructor keywords the LazyConfigs pass
    (configs/common/models/odise_with_label.py:16-29, mask_generator_with_label.py:29-66) and expect exactly the state-dict
    keys of the reference modules they replace."""
    import inspect
    from odise_b200 import plugin
    pins = _pins()
    head = plugin.B200MaskFormerHead(num_classes=133, device="cpu")
    want = {k[len("sem_seg_head."):] for k in pins["head_state_shapes"]}
    assert set(head.expected_keys()) == want
    for mine, ref in ((plugin.B200MSDeformAttnPixelDecoder, "MSDeformAttnPixelDecoder"),
                      (plugin.B200ODISEMultiScaleMaskedTransformerDecoder, "ODISEMultiScaleMaskedTransformerDecoder"),
                      (plugin.B200PooledMaskEmbed, "PooledMaskEmbed"), (plugin.B200PseudoClassEmbed, "PseudoClassEmbed")):
        ref_kw = pins["constructor_keywords"][ref]
        mine_kw = set(inspect.signature(mine.__init__).parameters)
        assert set(ref_kw) <= mine_kw, (mine.__name__, set(ref_kw) - mine_kw)
    # the keywords the label model's config passes (odise_with_label.py), as read from the file
    cfg = set(pins["odise_with_label_keywords"])
    bb_kw = {"feature_extractor", "out_features", "use_checkpoint", "slide_training"}
    assert bb_kw <= cfg
    assert bb_kw <= set(inspect.signature(plugin.B200FeatureExtractorBackbone.__init__).parameters)
    fe_kw = {"encoder_block_indices", "unet_block_indices", "decoder_block_indices", "steps", "learnable_time_embed",
             "num_timesteps", "clip_model_name"}
    assert fe_kw <= cfg
    assert fe_kw <= set(inspect.signature(plugin.B200LdmImplicitCaptionerExtractor.__init__).parameters)
    fe = plugin.B200LdmImplicitCaptionerExtractor(frozen_state_dict={}, device="cpu")
    bb = plugin.B200FeatureExtractorBackbone(fe, ["s2", "s3", "s4", "s5"], use_checkpoint=True, slide_training=True)
    got = set(bb.expected_keys())
    assert {k for k in got if k.startswith("feature_extractor.")} == {
        "feature_extractor." + k for k in ("clip_project.linear.weight", "clip_project.linear.bias",
                                           "clip_project.positional_embedding", "alpha_cond",
                                           "time_embed_project.linear.weight", "time_embed_project.linear.bias",
                                           "time_embed_project.positional_embedding", "alpha_cond_time_embed")}
    assert len([k for k in got if k.startswith("feature_projections.")]) == 8 * 9 + 4 * 3   # 4 of 8 blocks have a shortcut
