"""Vocabulary front end (odise_b200/vocab.py): label files / prompts / overlap rule pinned against the reference's own
functions and data, the BPE tokenizer checked on a hand-built merge table.  The reference's label files are kept under
tests/golden/openseg_labels/, and digests of what its own functions make of them in tests/golden/ref_pins.pt
(tools/make_golden_pins.py)."""
import hashlib
import json
import os

import pytest
import torch

from odise_b200 import vocab

GOLD = os.path.join(os.path.dirname(__file__), "golden")
LABELS = os.path.join(GOLD, "openseg_labels")
LABEL_FILES = (("ade20k_150", True), ("coco_panoptic", True), ("ade20k_847", True), ("ade20k_150", False))
PROMPTS = (None, "a", "photo", "scene")


def label_file(name, prompt_engineered):
    return f"{name}_with_prompt_eng.txt" if prompt_engineered else f"{name}.txt"


def digest(labels):
    """SHA-256 of a (nested) list of strings: equal digests <=> equal lists."""
    return hashlib.sha256(json.dumps(labels).encode()).hexdigest()


def _digests():
    return torch.load(os.path.join(GOLD, "ref_pins.pt"), weights_only=True)["label_digests"]


def test_label_files_and_prompts_match_reference():
    d = _digests()
    for name, n_cls, n_prompts in (("ade20k_150", 150, 403), ("coco_panoptic", 133, 254), ("ade20k_847", 847, 1342)):
        f = label_file(name, True)
        mine = vocab.read_label_file(os.path.join(LABELS, f))
        assert digest(mine) == d[f] and len(mine) == n_cls and sum(len(s) for s in mine) == n_prompts     # SURVEY.md §8 K' counts
        for p in PROMPTS:
            assert digest(vocab.prompt_labels(mine, p)) == d[f"{f}:{p}"], (f, p)
    f = label_file("ade20k_150", False)
    assert digest(vocab.read_label_file(os.path.join(LABELS, f))) == d[f]


def test_overlap_rule():
    test_labels = [["cat", "kitty"], ["unicorn"], ["dog"], ["spaceship", "rocket"]]
    train_labels = [["cat"], ["dog", "puppy"], ["tree"]]
    assert vocab.overlapping_mask(test_labels, train_labels) == [True, False, True, False]      # as pinned in ref_clip.pt
    with pytest.raises(ValueError):
        vocab.prompt_labels(test_labels, "poem")
    assert vocab.prompt_labels([["wall"]], "photo") == [["a photo of a wall."]]


def test_bpe_tokenizer_mechanics():
    """merge table: 'c a' -> 'ca', 'ca t</w>' -> 'cat</w>', 'd o' -> 'do', 'p h' -> 'ph'.  Ranks decide the merge order;
    unmerged characters stay single tokens; the last character carries '</w>'."""
    tk = vocab.SimpleTokenizer(merges=["c a", "ca t</w>", "d o", "p h"])
    e = tk.encoder
    assert len(e) == 256 + 256 + 4 + 2 and tk.sot_id == len(e) - 2 and tk.eot_id == len(e) - 1
    assert tk.encode("cat") == [e["cat</w>"]]
    assert tk.encode("Cat  ") == [e["cat</w>"]]                                  # lower-cased, whitespace cleaned
    assert tk.encode("cats") == [e["ca"], e["t"], e["s</w>"]]                     # 'ca t</w>' needs the word-final t
    assert tk.encode("dog") == [e["do"], e["g</w>"]]
    assert tk.encode("a photo.") == [e["a</w>"], e["ph"], e["o"], e["t"], e["o</w>"], e[".</w>"]]
    assert tk.encode("it's 42") == [e["i"], e["t</w>"], e["'"], e["s</w>"], e["4</w>"], e["2</w>"]]   # 's split, digits single
    assert tk.encode("&amp;") == [e["&</w>"]]                                    # html unescape
    ids = tk.tokenize(["cat", "dog dog dog dog"], context_length=6)
    assert ids.dtype == torch.int64 and ids.shape == (2, 6)
    assert ids[0].tolist() == [tk.sot_id, e["cat</w>"], tk.eot_id, 0, 0, 0]
    assert ids[1].tolist() == [tk.sot_id, e["do"], e["g</w>"], e["do"], e["g</w>"], tk.eot_id]   # truncated, EOT kept
    assert (ids.argmax(-1) == torch.tensor([2, 5])).all()                        # the EOT position clip.py:150 reads
    full = vocab.SimpleTokenizer(merges=[])
    assert full.tokenize("")[0, :2].tolist() == [full.sot_id, full.eot_id]


def test_open_state_dict_protocol_swaps_vocabularies():
    """OpenPanopticInference (pano_wrapper.py:36-68) saves the model's open state, loads its own, runs, restores: the
    plugin must round-trip the same keys, build a vocabulary once per label tuple and re-activate cached ones."""
    import types
    from collections import OrderedDict
    from odise_b200.plugin import B200CategoryODISE

    class FakeEngine:                                           # records what the plugin asks of the engine
        dev = "cpu"

        def __init__(self):
            self.vocabs, self.active, self.built = {}, None, []

        def has_vocabulary(self, key):
            return key in self.vocabs

        def use_vocabulary(self, key):
            self.active = key

        clip_head = object()                                    # the engine has a MaskCLIP head

        def set_vocabulary_from_tokens(self, key, ids, sizes, thing_ids=None, overlapping=None, clip_token_ids=None):
            self.vocabs[key] = dict(ids=ids, sizes=sizes, things=thing_ids, ov=overlapping, clip_ids=clip_token_ids)
            self.built.append(key)
            self.active = key

    eng = FakeEngine()
    tk = vocab.SimpleTokenizer(merges=["c a", "ca t</w>"])
    meta_a = types.SimpleNamespace(thing_dataset_id_to_contiguous_id={7: 0, 9: 2})
    model = B200CategoryODISE(eng, tokenizer=tk, train_labels=[["cat"], ["tree"]])
    assert list(model.open_state_dict()) == ["sem_seg_head.num_classes", "metadata", "test_topk_per_image", "semantic_on",
                                             "panoptic_on", "instance_on", "category_head.test_labels",
                                             "clip_head.test_labels"]
    la = [["cat", "kitty"], ["sky"], ["dog"]]
    lb = [["tree"], ["car", "automobile"]]
    wrap_a = OrderedDict([("sem_seg_head.num_classes", 3), ("metadata", meta_a), ("test_topk_per_image", 50),
                          ("semantic_on", True), ("panoptic_on", True), ("instance_on", False),
                          ("category_head.test_labels", la), ("clip_head.test_labels", la)])
    saved = model.open_state_dict()
    model.load_open_state_dict(wrap_a)
    ka = tuple(tuple(s) for s in la)
    assert eng.active == ka and eng.built == [ka]
    v = eng.vocabs[ka]
    assert v["sizes"] == [2, 1, 1] and v["things"] == [0, 2] and v["ov"] == [True, False, False]
    assert v["ids"].shape == (4, 77) and v["ids"][0, 0] == tk.sot_id
    # category bank = raw class names (CategoryEmbed prompt=None), MaskCLIP bank = "a photo of a {}." (PoolingCLIPHead)
    assert v["ids"][0].tolist()[:3] == [tk.sot_id, tk.encoder["cat</w>"], tk.eot_id]
    assert v["clip_ids"].shape == (4, 77) and torch.equal(v["clip_ids"], tk.tokenize(
        ["a photo of a cat.", "a photo of a kitty.", "a photo of a sky.", "a photo of a dog."]))
    assert model.test_topk_per_image == 50 and model.instance_on is False and model.num_classes == 3
    model.load_open_state_dict(OrderedDict([("sem_seg_head.num_classes", 2), ("category_head.test_labels", lb),
                                            ("clip_head.test_labels", lb)]))
    kb = tuple(tuple(s) for s in lb)
    assert eng.active == kb and eng.built == [ka, kb] and eng.vocabs[kb]["ov"] == [True, False]
    model.load_open_state_dict(wrap_a)                                         # cached: no rebuild
    assert eng.active == ka and eng.built == [ka, kb]
    with pytest.raises(KeyError):
        model.load_open_state_dict({"backbone.whatever": 1})
    with pytest.raises(ValueError):
        model.load_open_state_dict({"sem_seg_head.num_classes": 5, "category_head.test_labels": [["x"]],
                                    "clip_head.test_labels": [["x"]]})
    assert saved["category_head.test_labels"] is None
    # no silent defaults: a new vocabulary without train_labels / metadata is an error, not an alternating pattern
    bare = B200CategoryODISE(FakeEngine(), tokenizer=tk)
    with pytest.raises(RuntimeError):
        bare.load_open_state_dict({"category_head.test_labels": la, "clip_head.test_labels": la})
    bare.metadata = meta_a
    with pytest.raises(RuntimeError):
        bare.load_open_state_dict({"category_head.test_labels": la, "clip_head.test_labels": la})


def test_prompts_of_the_two_heads_match_reference():
    """ADVICE r1 (high): in the label model the category head scores against the RAW class names (CategoryEmbed
    prompt=None, odise.py:1225; configs/common/models/mask_generator_with_label.py passes none) and only PoolingCLIPHead
    uses "a photo of a {}." (odise.py:1428).  Pinned on the reference's own defaults, config and prompt function."""
    pins = torch.load(os.path.join(GOLD, "ref_pins.pt"), weights_only=True)
    assert pins["prompt_defaults"] == {"CategoryEmbed": None, "PoolingCLIPHead": "photo"}
    assert not pins["label_config"]["category_head_sets_prompt"]
    assert pins["label_config"]["clip_head_is_default_pooling_clip_head"]
    labels = vocab.read_label_file(os.path.join(LABELS, "ade20k_150_with_prompt_eng.txt"))
    cat, clip, sizes = vocab.vocabulary_prompts(labels)
    d = pins["label_digests"]
    assert digest(cat) == d["odise.prompt_labels:CategoryEmbed"] and digest(clip) == d["odise.prompt_labels:PoolingCLIPHead"]
    assert sizes == [len(s_) for s_ in labels] and len(cat) == len(clip) == 403 and cat != clip
