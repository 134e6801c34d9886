"""CPU: INTEGRATION.md section A, checked against what the UNMODIFIED reference does at the seams a maintainer touches.

tests/golden/reference_seams.json (written by oracle/pin_against_reference.py from the reference itself) records, for
the reference's own factories and helpers:
  * which decoder class, with which constructor call, ``network_constructors.make_depth_decoder``
    (KITTI/networks/network_constructors.py:30-40) and ``Model`` (NYUv2/model.py:47-71) build for each option set -
    after the three-line swap the same names resolve to OUR classes, so the same calls must build them;
  * the ``.convs`` keys and the parameter groups ``pyt_utils.group_weight`` forms over them (KITTI/trainer.py:74-75,
    KITTI/pyt_utils.py:12-29; its assert fails if a module carries a parameter that is not a Conv/Linear weight or bias);
  * the decoders' state-dict keys and shapes, in order, so checkpoints load STRICTLY in both directions
    (KITTI/test_simple.py:101-102) and survive the save / load code paths on disk (KITTI/trainer.py:733-773 pattern,
    NYUv2/load_save_utils.py:10-39);
  * the parameter names of the hot-path functions of KITTI/layers.py.
Without CUDA the swapped-in decoders fail loudly (no silent CPU path).
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from wavelet_monodepth_b200 import kitti_decoders as kd
from wavelet_monodepth_b200 import kitti_layers as kl
from wavelet_monodepth_b200 import nyu_decoders as nd

from helpers import GOLDEN

SEAMS = json.load(open(os.path.join(GOLDEN, "reference_seams.json")))
STATE_DICTS = json.load(open(os.path.join(GOLDEN, "state_dict_keys.json")))


def _arg(v):
    """Inverse of the pinning script's tagging: {"ndarray": [...]} -> np.array, {"range": [a, b, s]} -> range."""
    if isinstance(v, dict) and set(v) == {"ndarray"}:
        return np.array(v["ndarray"])
    if isinstance(v, dict) and set(v) == {"range"}:
        return range(*v["range"])
    return v


def _build(module, call):
    """The constructor call the reference's factory made, with the class name resolved in `module` (ours)."""
    cls = getattr(module, call["class"])
    return cls(*[_arg(a) for a in call["args"]], **{k: _arg(v) for k, v in call["kwargs"].items()})


def _keys_shapes(module):
    return [[k, list(v.shape)] for k, v in module.state_dict().items()]


def _checkpoint_from(keys_shapes, seed):
    """A state dict with the reference module's keys and shapes (in its order) and seeded values."""
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(*shape, generator=g) for k, shape in keys_shapes}


def _group_counts(module):
    """(decay, no_decay) as pyt_utils.group_weight splits a module: Conv/Linear weights, then their biases; the
    parameters it would leave out make its assert fail, so they are checked here too."""
    decay, no_decay = [], []
    for m in module.modules():
        if isinstance(m, (nn.Linear, nn.Conv2d, nn.Conv3d)):
            decay.append(m.weight)
            if m.bias is not None:
                no_decay.append(m.bias)
    assert len(list(module.parameters())) == len(decay) + len(no_decay)
    return len(decay), len(no_decay)


def test_kitti_factory_builds_our_decoders_and_trainer_param_groups_accept_them():
    assert [c["class"] for c in SEAMS["kitti"]["factory"]] == \
        ["DepthWaveProgressiveDecoder", "SparseDepthWaveProgressiveDecoder", "DepthDecoder"]
    for k, call in enumerate(SEAMS["kitti"]["factory"]):
        dec = _build(kd, call)
        want = SEAMS["kitti"]["decoders"][call["class"]]
        decay = no_decay = groups = 0
        for _, weights in dec.convs.items():                          # KITTI/trainer.py:74-75
            d, nd_ = _group_counts(weights)
            decay, no_decay, groups = decay + d, no_decay + nd_, groups + 2
        assert {"decay": decay, "no_decay": no_decay, "groups": groups} == want["group_weight"]
        assert decay + no_decay == len(list(dec.parameters())) > 0   # every parameter is reachable through .convs
        assert [list(key) for key in dec.convs.keys()] == want["convs"]
        assert _keys_shapes(dec) == want["state_dict"]
        assert [[k_, s] for k_, s in STATE_DICTS["kitti." + call["class"]].items()] == want["state_dict"]
        # strict loading both ways (KITTI/test_simple.py:101-102): the reference's keys and shapes, our module
        theirs = _checkpoint_from(want["state_dict"], seed=k)
        dec.load_state_dict(theirs, strict=True)
        for key, v in dec.state_dict().items():
            assert torch.equal(v, theirs[key]), key


def test_kitti_checkpoints_round_trip_on_disk_through_the_trainers_code_path(tmp_path):
    ours = _build(kd, next(c for c in SEAMS["kitti"]["factory"] if c["opts"]["use_sparse"]))
    assert type(ours) is kd.SparseDepthWaveProgressiveDecoder
    theirs_keys = SEAMS["kitti"]["decoders"]["SparseDepthWaveProgressiveDecoder"]["state_dict"]
    # trainer.save_model (:733-751): torch.save(model.state_dict(), "<name>.pth")
    torch.save(ours.state_dict(), tmp_path / "depth.pth")
    torch.save(_checkpoint_from(theirs_keys, seed=5), tmp_path / "depth_ref.pth")
    # what a reference module loading depth.pth strictly requires: exactly its keys, in its order, with its shapes
    mine = torch.load(tmp_path / "depth.pth", map_location="cpu")
    assert [[k, list(v.shape)] for k, v in mine.items()] == theirs_keys
    for k, v in ours.state_dict().items():
        assert torch.equal(mine[k], v), k
    # trainer.load_model (:753-773): filter by key, update, load
    model_dict = ours.state_dict()
    pretrained = {k: v for k, v in torch.load(tmp_path / "depth_ref.pth").items() if k in model_dict}
    assert set(pretrained) == set(model_dict)
    model_dict.update(pretrained)
    ours.load_state_dict(model_dict)
    for k, v in torch.load(tmp_path / "depth_ref.pth").items():      # what the reference module had saved
        assert torch.equal(ours.state_dict()[k], v), k
    # evaluate_depth.py:130 loads non-strictly
    ours.load_state_dict(torch.load(tmp_path / "depth_ref.pth"), strict=False)


def test_swapped_kitti_decoder_fails_loudly_without_cuda():
    """Host tensors are refused whether or not a device is present: there is no CPU path to fall back to."""
    from wavelet_monodepth_b200._lib import WmdError
    call = next(c for c in SEAMS["kitti"]["factory"] if c["opts"]["use_sparse"])
    dec = _build(kd, call)
    num_ch_enc = _arg(call["args"][0])
    feats = [torch.rand(1, c, 6 << (4 - k), 20 << (4 - k)) for k, c in enumerate(num_ch_enc)]
    with pytest.raises(WmdError):
        dec(feats, 0.05)


class _Model(nn.Module):
    """Stand-in for NYUv2/model.py's Model: the decoder under `decoder.`, beside an encoder."""

    def __init__(self, decoder):
        super().__init__()
        self.encoder = nn.Conv2d(3, 4, 3)
        self.decoder = decoder


def test_nyu_model_builds_our_decoders_and_load_save_utils_round_trip(tmp_path):
    cases = SEAMS["nyu"]["model"]
    assert [c["class"] for c in cases] == ["DecoderWave", "SparseDecoderWave", "DecoderWave224", "Decoder", "Decoder224"]
    for k, call in enumerate(cases):
        dec = _build(nd, call)                                       # INTEGRATION.md A, line 2
        want = SEAMS["nyu"]["decoders"][call["class"]]["state_dict"]
        assert _keys_shapes(dec) == want, call["class"]
        theirs = _checkpoint_from(want, seed=k)
        dec.load_state_dict(theirs, strict=True)
        for key, v in dec.state_dict().items():
            assert torch.equal(v, theirs[key]), key
        if "nyu." + call["class"] in STATE_DICTS:
            assert [[k_, s] for k_, s in STATE_DICTS["nyu." + call["class"]].items()] == want
    # load_save_utils.save_model writes Model.state_dict() to <log>/models/weights_<epoch>/model.pth and load_model
    # filters a checkpoint by the model's keys, updates and loads it: a model carrying our decoder, then a reference twin
    save = SEAMS["nyu_save_model"]
    assert save["files"] == ["models/weights_%d/model.pth" % save["epoch"]]
    sparse = next(c for c in cases if c["class"] == "SparseDecoderWave")
    m = _Model(_build(nd, sparse))
    path = tmp_path / save["files"][0]
    path.parent.mkdir(parents=True)
    torch.save(m.state_dict(), path)
    prefix = SEAMS["nyu"]["decoders"]["SparseDecoderWave"]["model_prefix"]
    saved = torch.load(path)
    theirs_keys = SEAMS["nyu"]["decoders"]["SparseDecoderWave"]["state_dict"]
    assert [[k[len(prefix):], list(v.shape)] for k, v in saved.items() if k.startswith(prefix)] == theirs_keys
    twin = {prefix + k: v for k, v in _checkpoint_from(theirs_keys, seed=9).items()}
    torch.save(twin, tmp_path / "twin.pth")
    model_dict = m.state_dict()
    pretrained = {k: v for k, v in torch.load(tmp_path / "twin.pth").items() if k in model_dict}
    assert set(pretrained) == {k for k in model_dict if k.startswith(prefix)}
    model_dict.update(pretrained)
    m.load_state_dict(model_dict)
    for k, v in twin.items():
        assert torch.equal(m.state_dict()[k], v), k


def test_functional_api_names_match_the_reference_layers():
    """Every public name of the hot path in KITTI/layers.py exists with the same parameter names here."""
    import inspect
    sigs = SEAMS["kitti"]["layer_signatures"]
    assert sorted(sigs) == sorted(("Conv3x3", "Conv1x1", "ConvBlock", "upsample", "sparse_select", "make_result", "mask2yx",
                                   "mask2idxmap", "sparse_conv1x1", "sparse_conv3x3", "sparse_upsample"))
    for name, want in sigs.items():
        b = getattr(kl, name)
        if want["class"]:
            assert inspect.isclass(b) and issubclass(b, nn.Module), name
            b = b.__init__
        pa, pb = want["params"], list(inspect.signature(b).parameters)
        assert pa == pb[:len(pa)], (name, pa, pb)
