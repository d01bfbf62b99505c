"""Import scaffolding that lets the REFERENCE's own Python (vendored Mask2Former + odise/modeling/meta_arch/odise.py)
run on CPU where detectron2 / fvcore / open_clip / ldm / ... are not installed.
TEST INFRASTRUCTURE ONLY — used by tools/make_golden_ref.py and tools/make_golden_pins.py, which store what the
reference computes under tests/golden/; no test imports it.  The arithmetic executed is the reference's; only third-party
registry / config decorators and the tiny detectron2 layer helpers are stubbed (SURVEY.md Appendix C):

  detectron2.layers.Conv2d     = nn.Conv2d with optional .norm / .activation applied in forward  (d2 wrappers.py)
  detectron2.layers.get_norm   = "GN" -> GroupNorm(32, C)                                          (d2 batch_norm.py)
  fvcore c2_xavier_fill        = kaiming_uniform_(a=1) + zero bias
"""
import importlib
import importlib.abc
import importlib.machinery
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

REF = os.environ.get("ODISE_REFERENCE", "/root/reference")
M2F = os.path.join(REF, "third_party", "Mask2Former")


def available():
    return os.path.isdir(os.path.join(REF, "odise")) and os.path.isdir(os.path.join(M2F, "mask2former"))


class _Anything:
    """Permissive stand-in: callable as an identity decorator / factory, attribute access returns itself."""

    def __init__(self, name="stub"):
        self._name = name

    def __call__(self, *a, **k):
        if len(a) == 1 and not k and (isinstance(a[0], type) or callable(a[0])):
            return a[0]
        return self

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        return _Anything(self._name + "." + item)

    def __iter__(self):
        return iter(())

    def __mro_entries__(self, bases):
        return (object,)


class _StubModule(types.ModuleType):
    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        v = _Anything(self.__name__ + "." + item)
        setattr(self, item, v)
        return v


_STUB_ROOTS = ("detectron2", "fvcore", "open_clip", "diffdist", "nltk", "iopath", "omegaconf", "ldm", "timm",
               "panopticapi", "pycocotools", "lvis", "wandb", "xformers")


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] in _STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _StubModule(spec.name)
        m.__path__ = []
        return m

    def exec_module(self, module):
        pass


class Conv2d(nn.Conv2d):
    """detectron2.layers.Conv2d: conv -> optional norm -> optional activation."""

    def __init__(self, *args, **kwargs):
        norm = kwargs.pop("norm", None)
        activation = kwargs.pop("activation", None)
        super().__init__(*args, **kwargs)
        self.norm = norm
        self.activation = activation

    def forward(self, x):
        x = F.conv2d(x, self.weight, self.bias, self.stride, self.padding, self.dilation, self.groups)
        if self.norm is not None:
            x = self.norm(x)
        if self.activation is not None:
            x = self.activation(x)
        return x


def get_norm(norm, out_channels):
    if norm is None or norm == "":
        return None
    assert norm == "GN", norm
    return nn.GroupNorm(32, out_channels)


class ShapeSpec:
    def __init__(self, channels=None, height=None, width=None, stride=None):
        self.channels, self.height, self.width, self.stride = channels, height, width, stride


def c2_xavier_fill(module):
    nn.init.kaiming_uniform_(module.weight, a=1)
    if module.bias is not None:
        nn.init.constant_(module.bias, 0)


_installed = False


def install():
    """Make `mask2former.modeling...` and `odise.modeling.meta_arch.odise` importable. Idempotent."""
    global _installed
    if _installed:
        return
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF)
    sys.meta_path.insert(0, _StubFinder())
    d2l = importlib.import_module("detectron2.layers")
    d2l.Conv2d, d2l.get_norm, d2l.ShapeSpec = Conv2d, get_norm, ShapeSpec
    importlib.import_module("detectron2.modeling").ShapeSpec = ShapeSpec
    bb = importlib.import_module("detectron2.modeling.backbone")
    bb.Backbone = nn.Module
    importlib.import_module("detectron2.modeling.backbone.backbone").Backbone = nn.Module
    comm = importlib.import_module("detectron2.utils.comm")
    comm.get_world_size = lambda: 1
    comm.get_rank = lambda: 0
    comm.get_local_rank = lambda: 0
    importlib.import_module("detectron2.utils").comm = comm
    wi = importlib.import_module("fvcore.nn.weight_init")
    wi.c2_xavier_fill = c2_xavier_fill
    importlib.import_module("fvcore.nn").weight_init = wi
    cfgm = importlib.import_module("detectron2.config")
    cfgm.configurable = lambda f=None, **kw: (f if f is not None else (lambda g: g))

    # packages whose __init__ would import datasets / detectron2 internals: pre-register bare packages
    def pkg(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
        return m

    pkg("mask2former", os.path.join(M2F, "mask2former"))
    pkg("mask2former.modeling", os.path.join(M2F, "mask2former", "modeling"))
    pkg("mask2former.modeling.pixel_decoder", os.path.join(M2F, "mask2former", "modeling", "pixel_decoder"))
    pkg("mask2former.modeling.transformer_decoder", os.path.join(M2F, "mask2former", "modeling", "transformer_decoder"))
    pkg("mask2former.modeling.meta_arch", os.path.join(M2F, "mask2former", "modeling", "meta_arch"))
    pkg("mask2former.utils", os.path.join(M2F, "mask2former", "utils"))
    pkg("odise", os.path.join(REF, "odise"))
    pkg("odise.modeling", os.path.join(REF, "odise", "modeling"))
    pkg("odise.modeling.meta_arch", os.path.join(REF, "odise", "modeling", "meta_arch"))
    pkg("odise.modeling.backbone", os.path.join(REF, "odise", "modeling", "backbone"))
    pkg("odise.data", os.path.join(REF, "odise", "data"))
    pkg("odise.utils", os.path.join(REF, "odise", "utils"))
    pkg("odise.checkpoint", os.path.join(REF, "odise", "checkpoint"))
    _installed = True


def ref_head(m):
    """The reference's pixel decoder and ODISE decoder (m = modules()) in the configuration of the label model."""
    S = m.ShapeSpec
    shape = {f"s{i}": S(channels=512, stride=2 ** i) for i in (2, 3, 4, 5)}
    pd = m.MSDeformAttnPixelDecoder(shape, transformer_dropout=0.0, transformer_nheads=8,
                                    transformer_dim_feedforward=1024, transformer_enc_layers=6, conv_dim=256,
                                    mask_dim=256, norm="GN", transformer_in_features=["s3", "s4", "s5"],
                                    common_stride=4).eval()
    dec = m.ODISEMultiScaleMaskedTransformerDecoder(
        class_embed=m.PseudoClassEmbed(133), post_mask_embed=m.PooledMaskEmbed(256, 256, 256), in_channels=256,
        mask_classification=True, num_classes=133, hidden_dim=256, num_queries=100, nheads=8, dim_feedforward=2048,
        dec_layers=9, pre_norm=False, enforce_input_project=False, mask_dim=256).eval()
    return pd, dec


def strip(sd, prefix):
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def modules():
    """Returns the reference classes on the hot path."""
    install()
    msd = importlib.import_module("mask2former.modeling.pixel_decoder.msdeformattn")
    dec = importlib.import_module("mask2former.modeling.transformer_decoder.mask2former_transformer_decoder")
    pe = importlib.import_module("mask2former.modeling.transformer_decoder.position_encoding")
    od = importlib.import_module("odise.modeling.meta_arch.odise")
    hp = importlib.import_module("odise.modeling.meta_arch.helper")
    return types.SimpleNamespace(
        MSDeformAttnPixelDecoder=msd.MSDeformAttnPixelDecoder,
        MSDeformAttn=importlib.import_module("mask2former.modeling.pixel_decoder.ops.modules.ms_deform_attn").MSDeformAttn,
        ms_deform_attn_core_pytorch=importlib.import_module(
            "mask2former.modeling.pixel_decoder.ops.functions.ms_deform_attn_func").ms_deform_attn_core_pytorch,
        MultiScaleMaskedTransformerDecoder=dec.MultiScaleMaskedTransformerDecoder,
        PositionEmbeddingSine=pe.PositionEmbeddingSine,
        ODISEMultiScaleMaskedTransformerDecoder=od.ODISEMultiScaleMaskedTransformerDecoder,
        PooledMaskEmbed=od.PooledMaskEmbed, PseudoClassEmbed=od.PseudoClassEmbed, MaskPooling=od.MaskPooling,
        CategoryODISE=od.CategoryODISE, ensemble_logits_with_labels=hp.ensemble_logits_with_labels,
        ShapeSpec=ShapeSpec, odise_module=od)
