"""CPU: the oracle restatement reproduces every golden vector the unmodified reference produced.

(The fixtures under tests/golden/ were written by oracle/pin_against_reference.py from the reference
itself; /root/reference is not needed here.)
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import GOLDEN_THREADS, haar, kitti as okitti, nyu as onyu, sparse_ops as osp
from wavelet_monodepth_b200 import synth
from wavelet_monodepth_b200.kitti_decoders import DepthWaveProgressiveDecoder
from wavelet_monodepth_b200.nyu_decoders import DecoderWave

from helpers import (compare_outputs, golden_names, kitti_features, load_golden, nyu_features, seeded_params)


@pytest.fixture(autouse=True)
def _golden_arithmetic():
    """No autograd, and the thread count the fixtures were written with: on a host with more cores the default count
    changes how the GEMMs split their sums, and the 1e-6 bar below is a same-summation-order statement."""
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        with torch.no_grad():
            yield
    finally:
        torch.set_num_threads(threads)




def test_kitti_dense_matches_reference_golden():
    want, meta = load_golden("kitti_tiny_dense")
    mod = DepthWaveProgressiveDecoder(np.array(meta["num_ch_enc"]))
    sd = seeded_params(mod, meta)
    got = okitti.dense_forward(sd, kitti_features(meta))
    assert compare_outputs(got, want, "kitti dense", float_tol=1e-6) <= 1e-6


@pytest.mark.parametrize("name", golden_names("kitti_tiny_sparse"))
def test_kitti_sparse_matches_reference_golden(name):
    want, meta = load_golden(name)
    mod = DepthWaveProgressiveDecoder(np.array(meta["num_ch_enc"]))
    sd = seeded_params(mod, meta)
    got = okitti.sparse_forward(sd, kitti_features(meta), meta["thresh_ratio"])
    compare_outputs(got, want, name, float_tol=1e-6)


def test_nyu_dense_matches_reference_golden():
    want, meta = load_golden("nyu_tiny_dense")
    mod = DecoderWave(enc_features=list(meta["enc_features"]))
    got = onyu.dense_forward(seeded_params(mod, meta), nyu_features(meta))
    compare_outputs(got, want, "nyu dense", float_tol=1e-6)


@pytest.mark.parametrize("name", golden_names("nyu_tiny_sparse"))
def test_nyu_sparse_matches_reference_golden(name):
    want, meta = load_golden(name)
    mod = DecoderWave(enc_features=list(meta["enc_features"]))
    got = onyu.sparse_forward(seeded_params(mod, meta), nyu_features(meta), meta["thresh_ratio"])
    compare_outputs(got, want, name, float_tol=1e-6)


def test_sparse_thr_negative_equals_dense():
    """Reference invariant (SURVEY 4): with all masks full the sparse decoder equals the dense one."""
    want, meta = load_golden("kitti_tiny_sparse_thr-1_s0")
    dense, _ = load_golden("kitti_tiny_dense")
    for s in range(4):
        np.testing.assert_allclose(want["disp_%d" % s], dense["disp_%d" % s][:1], atol=1e-6)


def test_haar_perfect_reconstruction_and_closed_form():
    g = torch.Generator().manual_seed(0)
    x = torch.rand(2, 1, 240, 320, generator=g) * 10
    dwt, idwt = haar.DWTForward(J=4, wave="haar", mode="reflect"), haar.DWTInverse(wave="haar", mode="zero")
    yl, yh = dwt(x)
    assert yl.shape == (2, 1, 15, 20) and [tuple(h.shape) for h in yh] == [
        (2, 1, 3, 120, 160), (2, 1, 3, 60, 80), (2, 1, 3, 30, 40), (2, 1, 3, 15, 20)]
    assert float((idwt((yl, yh)) - x).abs().max()) < 5e-6
    ll, h = torch.rand(2, 1, 6, 8, generator=g), torch.rand(2, 1, 3, 6, 8, generator=g)
    assert float((idwt((ll, [h])) - haar.closed_form_idwt(ll, h)).abs().max()) < 1e-6
    # an image varying only along the height puts all detail energy in LH (band 0)
    ramp = torch.arange(8.0).reshape(1, 1, 8, 1).expand(1, 1, 8, 8).contiguous()
    _, (hh,) = haar.DWTForward(J=1, wave="haar")(ramp)
    assert float(hh[:, :, 0].abs().max()) > 0.5 and float(hh[:, :, 1:].abs().max()) < 1e-6


def test_sparse_ops_match_reference_golden():
    want, meta = load_golden("sparse_ops")
    cin, cout = meta["cin"], meta["cout"]
    shapes = {"conv.weight": (cout, cin, 3, 3), "conv.bias": (cout,)}
    sd = synth.random_state_dict(shapes, seed=meta["param_seed"])
    for a in ("dense", "half", "few", "empty"):
        in_mask = torch.from_numpy(want["in_%s_mask" % a])
        xvals = torch.from_numpy(want["in_%s_xvals" % a])
        idxmap, _ = osp.index_map(in_mask)
        for b in ("dense", "half", "few", "empty"):
            out_mask = torch.from_numpy(want["in_%s_mask" % b])
            for pad in ("reflect", "constant", "replicate"):
                flat, c, ops = osp.conv3x3(sd["conv.weight"], sd["conv.bias"], xvals, idxmap, out_mask,
                                           padding=pad, make_result=False)
                np.testing.assert_array_equal(flat.numpy(), want["conv_%s_%s_%s" % (a, b, pad)])
                assert ops == int(want["conv_%s_%s_%s_ops" % (a, b, pad)])
            np.testing.assert_array_equal(osp.select(xvals, cin, idxmap, out_mask, pad=True).numpy(),
                                          want["select_%s_%s" % (a, b)])


def test_sparse_output_is_zero_outside_wavelet_mask():
    want, _ = load_golden("kitti_tiny_sparse_thr0.25_s0")
    for s in (2, 1, 0):
        m = want["wavelet_mask_%d" % s].astype(bool)
        for band in ("LH", "HL", "HH"):
            assert np.all(want["wavelets_%d_%s" % (s, band)][~m] == 0)
