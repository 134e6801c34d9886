"""Pin the oracle against the UNMODIFIED reference and write the golden vectors.

Runs only in the build container (needs /root/reference).  It
  1. imports the reference's KITTI and NYUv2 trees as they are, with
     ``oracle.haar`` registered as the (absent) ``pytorch_wavelets`` dependency,
  2. runs reference modules and the oracle's restatement on the same seeded
     weights / features and asserts they agree (floats <= 1e-6 abs, masks and
     op counts exactly),
  3. checks the Haar synthesis against the reference's own closed form
     ``my_iwt_once`` (depth_decoder.py:225-239),
  4. reproduces the two notebook known-answer op counts
     (KITTI/sparsity_test_notebook.ipynb:1345, NYUv2/sparsity_test_notebook.ipynb:1344),
  5. stores the *reference's* outputs as ``tests/golden/*.npz`` (the fixtures the
     CPU and GPU tests compare against; /root/reference does not exist on the
     GPU box).

Usage:  python -m oracle.pin_against_reference [--skip-kat]
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from oracle import GOLDEN_THREADS, haar, kitti as okitti, nyu as onyu, sparse_ops as osp   # noqa: E402
from wavelet_monodepth_b200 import synth                                   # noqa: E402

REF = "/root/reference"
GOLDEN = os.path.join(REPO, "tests", "golden")

KITTI_TINY_CH = (8, 8, 16, 32, 64)
NYU_TINY_CH = (8, 8, 16, 32, 64)
# thresholds chosen so the tiny configs hit full, partial (clustered) and empty masks at every scale
KITTI_THRESHOLDS = (-1.0, 0.0, 0.15, 0.2, 0.25, 0.3, 0.42, 5.0)
NYU_THRESHOLDS = (-10.0, 0.0, 0.1, 0.2, 0.3, 0.4, 5.0)
HEAD_GAIN_KITTI = {".2.conv.": 8.0}
HEAD_GAIN_NYU = {"wave1.": 6.0, "wave2.": 6.0, "wave3.": 6.0}


def import_reference(tree):
    """Import the reference's ``tree`` (KITTI | NYUv2) unmodified, Haar stand-in registered."""
    for name in list(sys.modules):
        if name == "layers" or name == "networks" or name.startswith("networks."):
            del sys.modules[name]
    sys.path[:] = [p for p in sys.path if not p.startswith(REF)]
    sys.path.insert(0, os.path.join(REF, tree))
    sys.modules["pytorch_wavelets"] = haar
    importlib.invalidate_caches()
    if tree == "KITTI":
        layers = importlib.import_module("layers")
        dec = importlib.import_module("networks.decoders.depth_decoder")
    else:
        layers = importlib.import_module("networks.layers")
        dec = importlib.import_module("networks.decoders.densedepth_decoder")
    return layers, dec


def key_str(k):
    return k if isinstance(k, str) else "_".join(str(v) for v in k)


def to_npz_dict(outputs, prefix=""):
    d = {}
    for k, v in outputs.items():
        name = prefix + key_str(k)
        if torch.is_tensor(v):
            d[name] = v.detach().cpu().numpy()
        else:
            d[name] = np.asarray(v, dtype=np.int64)
    return d


def compare(ref_out, ora_out, what, atol=1e-6):
    assert set(map(key_str, ref_out)) == set(map(key_str, ora_out)), \
        (what, sorted(map(key_str, ref_out)), sorted(map(key_str, ora_out)))
    worst = 0.0
    for k, rv in ref_out.items():
        ov = ora_out[k]
        if torch.is_tensor(rv):
            assert rv.shape == ov.shape, (what, k, rv.shape, ov.shape)
            if rv.dtype == torch.bool or "mask" in key_str(k):
                assert torch.equal(rv.float(), ov.float()), (what, k, "mask mismatch")
            else:
                err = float((rv - ov).abs().max()) if rv.numel() else 0.0
                worst = max(worst, err)
                assert err <= atol, (what, k, err)
        else:
            assert int(rv) == int(ov), (what, k, rv, ov)
    print("  pinned %-46s max|diff| = %.2e" % (what, worst))


def silence(fn, *a, **kw):
    """The reference prints 'sparse: i' per level (depth_decoder.py:342); keep the log readable."""
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def density(out, name, s):
    m = out[(name, s)]
    return float(m.float().mean())


# --------------------------------------------------------------------------- KITTI
def pin_kitti(save):
    layers, dec = import_reference("KITTI")
    torch.manual_seed(0)
    ref_dense = dec.DepthWaveProgressiveDecoder(np.array(KITTI_TINY_CH)).eval()
    ref_sparse = dec.SparseDepthWaveProgressiveDecoder(np.array(KITTI_TINY_CH)).eval()
    sd = synth.random_state_dict(synth.module_shapes(ref_dense), seed=11, gains=HEAD_GAIN_KITTI)
    ref_dense.load_state_dict(sd, strict=False)
    ref_sparse.load_state_dict(sd, strict=False)
    # state-dict contract (SURVEY 8b): 17 conv modules + the IDWT buffers
    keys = list(ref_dense.state_dict().keys())
    assert [k for k in keys if k.startswith("inverse_wt.")] == \
        ["inverse_wt.g0_col", "inverse_wt.g1_col", "inverse_wt.g0_row", "inverse_wt.g1_row"]

    feats2 = synth.blocky_features(synth.kitti_feature_shapes(2, 64, 96, KITTI_TINY_CH), seed=5, cell=4)
    with torch.no_grad():
        r = ref_dense(feats2)
        o = okitti.dense_forward(sd, feats2)
        compare(r, o, "KITTI dense decoder (N=2)")
        save("kitti_tiny_dense", to_npz_dict(r), dict(num_ch_enc=KITTI_TINY_CH, n=2, height=64, width=96,
                                                     param_seed=11, feat_seed=5, cell=4, gains=HEAD_GAIN_KITTI))
        # closed form == stand-in (depth_decoder.py:225-239)
        yl = r[("wavelets", 0, "LL")]
        yh = torch.stack([r[("wavelets", 0, b)] for b in ("LH", "HL", "HH")], 2)
        a = ref_sparse.my_iwt_once((yl, [yh]))
        b = haar.DWTInverse("haar", "zero")((yl, [yh]))
        c = haar.closed_form_idwt(yl, yh)
        assert float((a - b).abs().max()) <= 2e-6 and torch.equal(a, c)
        print("  pinned my_iwt_once vs Haar stand-in                    max|diff| = %.2e" % float((a - b).abs().max()))

        for thr in KITTI_THRESHOLDS:
            for b_idx in range(2):
                f1 = [f[b_idx:b_idx + 1] for f in feats2]
                r = silence(ref_sparse, f1, thr)
                o = okitti.sparse_forward(sd, f1, thr)
                tag = "KITTI sparse thr=%g sample %d" % (thr, b_idx)
                compare(r, o, tag)
                dens = [round(density(r, "wavelet_mask", s), 3) for s in (3, 2, 1, 0)]
                print("      wavelet_mask density scales 3..0:", dens, " total_ops", r["total_ops"])
                save("kitti_tiny_sparse_thr%g_s%d" % (thr, b_idx), to_npz_dict(r),
                     dict(num_ch_enc=KITTI_TINY_CH, n=1, sample=b_idx, height=64, width=96, thresh_ratio=thr,
                          param_seed=11, feat_seed=5, cell=4, gains=HEAD_GAIN_KITTI))
    return layers


def pin_sparse_ops(layers, save):
    """Functional ops, random masks (incl. empty), all three index-map paddings."""
    rs = np.random.RandomState(3)
    h, w, cin, cout, cs = 10, 14, 6, 5, 3
    full = torch.ones(1, 1, h, w)
    cases = {}
    for name, p in (("dense", 1.0), ("half", 0.5), ("few", 0.08), ("empty", 0.0)):
        cases[name] = torch.from_numpy((rs.uniform(size=(1, 1, h, w)) < p).astype(np.float32)) if p < 1 else full
    conv = layers.Conv3x3(cin, cout)
    block = layers.ConvBlock(cin, cout, use_refl=True)
    seq = nn.Sequential(layers.Conv1x1(cin, cin), nn.LeakyReLU(0.1, inplace=True), layers.Conv3x3(cin, 3))
    for m in (conv, block, seq):
        m.load_state_dict(synth.random_state_dict(synth.module_shapes(m), seed=21), strict=False)
    store = {}
    with torch.no_grad():
        for in_name, in_mask in cases.items():
            m_in = int(in_mask.sum())
            xvals = torch.from_numpy(rs.uniform(-1, 1, size=(cin * m_in,)).astype(np.float32))
            idxmap, ops = layers.mask2idxmap(in_mask)
            oi, oo = osp.index_map(in_mask)
            assert torch.equal(idxmap, oi) and ops == oo
            if m_in:
                assert torch.equal(layers.mask2yx(in_mask), osp.active_coords(in_mask))
            store["in_%s_mask" % in_name] = in_mask.numpy()
            store["in_%s_xvals" % in_name] = xvals.numpy()
            for out_name, out_mask in cases.items():
                for pad in ("reflect", "constant", "replicate"):
                    r_flat, r_c, r_ops = layers.sparse_conv3x3(conv, xvals, idxmap, out_mask, padding=pad,
                                                               make_result=False)
                    o_flat, o_c, o_ops = osp.conv3x3(conv.conv.weight, conv.conv.bias, xvals, idxmap, out_mask,
                                                     padding=pad, make_result=False)
                    assert r_ops == o_ops and r_c == o_c
                    assert torch.equal(r_flat, o_flat), (in_name, out_name, pad)
                    store["conv_%s_%s_%s" % (in_name, out_name, pad)] = r_flat.numpy()
                    store["conv_%s_%s_%s_ops" % (in_name, out_name, pad)] = np.int64(r_ops)
                # ConvBlock branch (its ELU overrides nonlin, layers.py:419-421), dense result
                r_d, r_ops = layers.sparse_conv3x3(block, xvals, idxmap, out_mask)
                o_d, o_ops = osp.conv3x3(block.conv.conv.weight, block.conv.conv.bias, xvals, idxmap, out_mask,
                                         nonlin=torch.nn.functional.elu)
                assert torch.equal(r_d, o_d) and r_ops == o_ops
                store["block_%s_%s" % (in_name, out_name)] = r_d.numpy()
                # Sequential head branch (layers.py:426-431)
                r_d, r_ops = layers.sparse_conv3x3(seq, xvals, idxmap, out_mask, nonlin=torch.sigmoid)
                o_d, o_ops = osp.head3x3(seq[0].conv.weight, seq[0].conv.bias, seq[2].conv.weight,
                                         seq[2].conv.bias, xvals, idxmap, out_mask, torch.sigmoid)
                assert torch.equal(r_d, o_d) and r_ops == o_ops
                store["head_%s_%s" % (in_name, out_name)] = r_d.numpy()
                store["head_%s_%s_ops" % (in_name, out_name)] = np.int64(r_ops)
                # select with pad
                r_s = layers.sparse_select(xvals, cin, idxmap, out_mask, pad=True)
                o_s = osp.select(xvals, cin, idxmap, out_mask, pad=True)
                assert torch.equal(r_s, o_s)
                store["select_%s_%s" % (in_name, out_name)] = r_s.numpy()
        # upsample + skip concat: low-res active set must cover (y//2, x//2) of the hi-res set
        lo_mask = cases["half"]
        lo_idx, _ = layers.mask2idxmap(lo_mask)
        m_lo = int(lo_mask.sum())
        lo_vals = torch.from_numpy(rs.uniform(-1, 1, size=(cin * m_lo,)).astype(np.float32))
        up = torch.nn.functional.interpolate(lo_mask, scale_factor=2, mode="nearest")
        hi_mask = up * torch.from_numpy((rs.uniform(size=up.shape) < 0.6).astype(np.float32))
        skip = torch.from_numpy(rs.uniform(-1, 1, size=(1, cs, 2 * h, 2 * w)).astype(np.float32))
        r_v, r_c = layers.sparse_upsample(lo_vals, cin, lo_idx, skip, hi_mask, make_result=False)
        o_v, o_c = osp.upsample_concat(lo_vals, cin, lo_idx, skip, hi_mask, make_result=False)
        assert torch.equal(r_v, o_v) and r_c == o_c
        store.update(up_lo_vals=lo_vals.numpy(), up_hi_mask=hi_mask.numpy(), up_skip=skip.numpy(), up_out=r_v.numpy())
        r_sel = layers.sparse_select(lo_vals, cin, lo_idx, hi_mask, ufactor=2)
        assert torch.equal(r_sel, osp.select(lo_vals, cin, lo_idx, hi_mask, ufactor=2))
        store["up_select2"] = r_sel.numpy()
    print("  pinned functional sparse ops (4x4 mask pairs x 3 paddings, block, head, select, upsample): exact")
    save("sparse_ops", store, dict(h=h, w=w, cin=cin, cout=cout, cskip=cs, param_seed=21,
                                   modules=["Conv3x3", "ConvBlock(use_refl)", "Sequential(Conv1x1,LReLU,Conv3x3(3))"]))


# --------------------------------------------------------------------------- NYUv2
def pin_nyu(save):
    _, dec = import_reference("NYUv2")
    ref_dense = dec.DecoderWave(enc_features=list(NYU_TINY_CH), decoder_width=0.5).eval()
    ref_sparse = silence(dec.SparseDecoderWave, enc_features=list(NYU_TINY_CH), decoder_width=0.5).eval()
    sd = synth.random_state_dict(synth.module_shapes(ref_dense), seed=13, gains=HEAD_GAIN_NYU)
    ref_dense.load_state_dict(sd, strict=False)
    ref_sparse.load_state_dict(sd, strict=False)
    feats2 = synth.blocky_features(synth.nyu_feature_shapes(2, 96, 128, NYU_TINY_CH), seed=7, cell=4)
    with torch.no_grad():
        r = ref_dense(feats2)
        o = onyu.dense_forward(sd, feats2)
        compare(r, o, "NYU dense decoder (N=2)")
        save("nyu_tiny_dense", to_npz_dict(r), dict(enc_features=NYU_TINY_CH, n=2, height=96, width=128,
                                                   param_seed=13, feat_seed=7, cell=4, gains=HEAD_GAIN_NYU))
        for thr in NYU_THRESHOLDS:
            for b_idx in range(2):
                f1 = [f[b_idx:b_idx + 1] for f in feats2]
                r = ref_sparse(f1, thr)
                o = onyu.sparse_forward(sd, f1, thr)
                compare(r, o, "NYU sparse thr=%g sample %d" % (thr, b_idx))
                dens = [round(density(r, "wavelet_mask", s), 3) for s in (2, 1, 0)]
                print("      wavelet_mask density scales 2..0:", dens, " total_ops", r["total_ops"])
                save("nyu_tiny_sparse_thr%g_s%d" % (thr, b_idx), to_npz_dict(r),
                     dict(enc_features=NYU_TINY_CH, n=1, sample=b_idx, height=96, width=128, thresh_ratio=thr,
                          param_seed=13, feat_seed=7, cell=4, gains=HEAD_GAIN_NYU))


# --------------------------------------------------------------------------- KATs
def pin_known_answers(save):
    """Weight-independent op counts recorded in the reference's notebooks (SURVEY 4)."""
    kat = {}
    _, dec = import_reference("KITTI")
    d = dec.SparseDepthWaveProgressiveDecoder(np.array(synth.RESNET50_CH)).eval()
    feats = [torch.rand(s) for s in synth.kitti_feature_shapes(1, 320, 1024, synth.RESNET50_CH)]
    with torch.no_grad():
        r = silence(d, feats, -1.0)
    assert r["total_ops"] == 17473692295, r["total_ops"]
    kat["kitti_r50_1024x320_total_ops"] = r["total_ops"]
    for s in range(4):
        kat["kitti_r50_1024x320_total_ops_s%d" % s] = r[("total_ops", s)]
    sd = {k: v for k, v in d.state_dict().items()}
    o = okitti.sparse_forward(sd, feats, -1.0)
    assert o["total_ops"] == r["total_ops"]
    print("  KAT KITTI R50 1024x320 thr<0 total_ops = %d  (notebook: 17.474 G)" % r["total_ops"])

    _, dec = import_reference("NYUv2")
    d = silence(dec.SparseDecoderWave, enc_features=list(synth.DENSENET161_CH), decoder_width=0.5).eval()
    feats = [torch.rand(s) for s in synth.nyu_feature_shapes(1, 480, 640, synth.DENSENET161_CH)]
    with torch.no_grad():
        r = d(feats, -10)
    assert r["total_ops"] == 33463546800, r["total_ops"]
    kat["nyu_d161_640x480_total_ops"] = r["total_ops"]
    o = onyu.sparse_forward(dict(d.state_dict()), feats, -10)
    assert o["total_ops"] == r["total_ops"]
    print("  KAT NYU DenseNet161 640x480 thr=-10 total_ops = %d  (notebook: 33.464 G)" % r["total_ops"])
    with open(os.path.join(GOLDEN, "known_answers.json"), "w") as f:
        json.dump(kat, f, indent=1, sort_keys=True)


def pin_full_size(only_check=True):
    """BASELINE configs[0]/[1] size (ResNet18 pyramid, 640x192, one frame) with the bench's synthetic weights / features:
    the restatement against the reference's dense decoder and its sparse decoder at thr 0 and 0.05.  Nothing is stored
    except a small summary (op counts, mask pixel counts, plane checksums) - the point is that the pin also holds at a
    full-size configuration with non-degenerate masks, not only on the tiny fixtures."""
    import bench
    _, dec = import_reference("KITTI")
    ch = synth.RESNET18_CH
    ref_dense = dec.DepthWaveProgressiveDecoder(np.array(ch)).eval()
    ref_sparse = dec.SparseDepthWaveProgressiveDecoder(np.array(ch)).eval()
    sd = synth.random_state_dict(synth.module_shapes(ref_dense), seed=bench.SYNTH["param_seed"],
                                 gains={k: bench.SYNTH["head_gain"] for k in bench.HEAD_KEYS}, highpass=bench.HEAD_KEYS)
    ref_dense.load_state_dict(sd, strict=False)
    ref_sparse.load_state_dict(sd, strict=False)
    feats = synth.blocky_features(synth.kitti_feature_shapes(1, 192, 640, ch), seed=bench.SYNTH["feat_seed"],
                                  cell=bench.SYNTH["cell"], texture=bench.SYNTH["texture"])
    summary = {}
    with torch.no_grad():
        compare(ref_dense(feats), okitti.dense_forward(sd, feats), "KITTI R18 640x192 dense decoder (full size)")
        for thr in (0.0, 0.05):
            r = silence(ref_sparse, feats, thr)
            o = okitti.sparse_forward(sd, feats, thr)
            compare(r, o, "KITTI R18 640x192 sparse thr=%g (full size)" % thr)
            summary["thr%g" % thr] = {
                "total_ops": int(r["total_ops"]),
                "wavelet_mask_pixels": [int(r[("wavelet_mask", s)].sum()) for s in range(4)],
                "disp_sum": [float(r[("disp", s)].double().sum()) for s in range(4)],
                "disp_sumsq": [float((r[("disp", s)].double() ** 2).sum()) for s in range(4)]}
            print("      wavelet_mask density scales 3..0:", [round(density(r, "wavelet_mask", s), 3) for s in (3, 2, 1, 0)],
                  " total_ops", r["total_ops"])
    with open(os.path.join(GOLDEN, "kitti_r18_640x192_summary.json"), "w") as f:
        json.dump({"config": "ResNet18 pyramid 640x192, 1 frame, bench.py synthetic weights/features (param_seed %d, "
                             "feat_seed %d)" % (bench.SYNTH["param_seed"], bench.SYNTH["feat_seed"]),
                   "reference_outputs": summary}, f, indent=1, sort_keys=True)


def pin_state_dicts():
    """Record the reference modules' state-dict keys/shapes: the checkpoint-compatibility contract (SURVEY 8b)."""
    rec = {}
    _, dec = import_reference("KITTI")
    for name in ("DepthDecoder", "DepthWaveProgressiveDecoder", "SparseDepthWaveProgressiveDecoder"):
        m = getattr(dec, name)(np.array(synth.RESNET18_CH))
        rec["kitti." + name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    _, dec = import_reference("NYUv2")
    for name in ("DecoderWave", "SparseDecoderWave"):
        m = silence(getattr(dec, name), enc_features=list(synth.DENSENET161_CH), decoder_width=0.5)
        rec["nyu." + name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(GOLDEN, "state_dict_keys.json"), "w") as f:
        json.dump(rec, f, indent=0, sort_keys=False)
    print("  recorded state-dict contracts of %d reference modules" % len(rec))


def _jsonable(v):
    """Constructor arguments as JSON: arrays and ranges tagged so tests can rebuild the same call."""
    if isinstance(v, np.ndarray):
        return {"ndarray": v.tolist()}
    if isinstance(v, range):
        return {"range": [v.start, v.stop, v.step]}
    if isinstance(v, (list, tuple)):
        return [_jsonable(x) for x in v]
    if isinstance(v, np.integer):
        return int(v)
    return v


def _keys_shapes(module):
    return [[k, list(v.shape)] for k, v in module.state_dict().items()]


def pin_integration_seams():
    """Record what a maintainer of the reference meets when they swap in this package's decoders (INTEGRATION.md A):
    which class and constructor call the reference's factories make for each option set, the decoders' ``.convs`` keys,
    the parameter groups ``pyt_utils.group_weight`` forms from them, the NYUv2 decoders' state dicts, where
    ``load_save_utils.save_model`` writes, and the parameter names of the KITTI layer functions."""
    import argparse as _ap
    import contextlib
    import inspect
    import io
    import tempfile
    rec = {}

    def recorders(module, names):
        calls, orig = [], {n: getattr(module, n) for n in names}

        def make(n):
            def build(*args, **kw):
                calls.append({"class": n, "args": _jsonable(list(args)), "kwargs": {k: _jsonable(v) for k, v in kw.items()}})
                return orig[n](*args, **kw)
            return build
        for n in names:
            setattr(module, n, make(n))
        return calls, orig

    # KITTI: networks.network_constructors.make_depth_decoder, pyt_utils.group_weight, layers.py signatures
    layers, _ = import_reference("KITTI")
    decs = importlib.import_module("networks.decoders")
    ctor = importlib.import_module("networks.network_constructors")
    pyt_utils = importlib.import_module("pyt_utils")
    kitti_names = ("DepthDecoder", "DepthWaveProgressiveDecoder", "SparseDepthWaveProgressiveDecoder")
    calls, orig = recorders(decs, kitti_names)

    class _Encoder:
        num_ch_enc = np.array(synth.RESNET18_CH)

    factory, modules = [], {}
    for use_wavelets, use_sparse in ((True, False), (True, True), (False, False)):
        opts = _ap.Namespace(use_wavelets=use_wavelets, use_sparse=use_sparse, scales=range(4))
        with contextlib.redirect_stdout(io.StringIO()):
            m = ctor.make_depth_decoder(_Encoder(), opts)
        call = dict(calls.pop())
        call["opts"] = {"use_wavelets": use_wavelets, "use_sparse": use_sparse, "scales": _jsonable(opts.scales)}
        factory.append(call)
        groups = []
        for _, weights in m.convs.items():
            pyt_utils.group_weight(groups, weights, 1e-4)
        modules[call["class"]] = {
            "convs": [list(k) for k in m.convs.keys()],
            "group_weight": {"decay": sum(len(g["params"]) for g in groups[0::2]),
                             "no_decay": sum(len(g["params"]) for g in groups[1::2]), "groups": len(groups)},
            "state_dict": _keys_shapes(m)}
    for n, cls in orig.items():
        setattr(decs, n, cls)
    rec["kitti"] = {"factory": factory, "decoders": modules}
    sigs = {}
    for name in ("Conv3x3", "Conv1x1", "ConvBlock", "upsample", "sparse_select", "make_result", "mask2yx", "mask2idxmap",
                 "sparse_conv1x1", "sparse_conv3x3", "sparse_upsample"):
        a = getattr(layers, name)
        is_class = inspect.isclass(a)
        sigs[name] = {"class": is_class, "params": list(inspect.signature(a.__init__ if is_class else a).parameters)}
    rec["kitti"]["layer_signatures"] = sigs

    # NYUv2: model.Model and load_save_utils.save_model
    import_reference("NYUv2")
    decs = importlib.import_module("networks.decoders")
    nyu_names = ("Decoder", "DecoderWave", "Decoder224", "DecoderWave224", "SparseDecoderWave")
    for name in ("model", "load_save_utils"):
        sys.modules.pop(name, None)
    calls, orig = recorders(decs, nyu_names)
    model_mod = importlib.import_module("model")
    load_save_utils = importlib.import_module("load_save_utils")
    cases, modules = [], {}
    for kw in ({}, {"use_sparse": True}, {"use_224": True}, {"use_wavelets": False},
               {"use_wavelets": False, "use_224": True}):
        o = dict(encoder_type="densenet", normalize_input=False, pretrained_encoder=False, num_layers=18,
                 use_wavelets=True, use_sparse=False, use_224=False, dw_waveconv=False, dw_upconv=False)
        o.update(kw)
        with contextlib.redirect_stdout(io.StringIO()):
            m = model_mod.Model(_ap.Namespace(**o))
        call = dict(calls.pop())
        call["opts"] = o
        cases.append(call)
        sd = m.state_dict()
        dec_keys = [k for k in sd if k.startswith("decoder.")]
        assert [k[len("decoder."):] for k in dec_keys] == list(m.decoder.state_dict())
        modules[call["class"]] = {"state_dict": _keys_shapes(m.decoder), "model_prefix": "decoder."}
        if kw == {"use_sparse": True}:
            with tempfile.TemporaryDirectory() as tmp, contextlib.redirect_stdout(io.StringIO()):
                load_save_utils.save_model(m, tmp, 3)
                written = sorted(os.path.relpath(os.path.join(d, f), tmp) for d, _, fs in os.walk(tmp) for f in fs)
                saved = torch.load(os.path.join(tmp, written[0]))
            assert list(saved) == list(sd)
            rec["nyu_save_model"] = {"epoch": 3, "files": written, "content": "Model.state_dict()"}
    for n, cls in orig.items():
        setattr(decs, n, cls)
    rec["nyu"] = {"model": cases, "decoders": modules}
    with open(os.path.join(GOLDEN, "reference_seams.json"), "w") as f:
        json.dump(rec, f, indent=0, sort_keys=False)
    print("  recorded the integration seams (%d KITTI factory cases, %d NYUv2 model cases)" % (len(factory), len(cases)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--skip-kat", action="store_true", help="skip the two full-size op-count runs (~10 s)")
    args = ap.parse_args()
    assert os.path.isdir(REF), "the reference checkout is only available in the build container"
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_grad_enabled(False)
    torch.set_num_threads(GOLDEN_THREADS)

    def save(name, arrays, meta):
        arrays = dict(arrays)
        arrays["__meta__"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **arrays)

    print("pinning oracle against the unmodified reference (%s)" % REF)
    layers = pin_kitti(save)
    pin_sparse_ops(layers, save)
    pin_nyu(save)
    pin_state_dicts()
    pin_integration_seams()
    if not args.skip_kat:
        pin_known_answers(save)
        pin_full_size()
    print("golden vectors written to", GOLDEN)


if __name__ == "__main__":
    main()
