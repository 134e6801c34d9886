"""CPU: host-side mirror of the reference API - module structure, state-dict contract, loud failure off-GPU."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from wavelet_monodepth_b200 import kitti_decoders as kd
from wavelet_monodepth_b200 import nyu_decoders as nd
from wavelet_monodepth_b200 import synth, wavelets
from wavelet_monodepth_b200._lib import WmdError

from helpers import GOLDEN

CONTRACT = json.load(open(os.path.join(GOLDEN, "state_dict_keys.json")))


@pytest.mark.parametrize("name", ["DepthDecoder", "DepthWaveProgressiveDecoder", "SparseDepthWaveProgressiveDecoder"])
def test_kitti_state_dict_contract(name):
    mod = getattr(kd, name)(np.array(synth.RESNET18_CH))
    got = {k: list(v.shape) for k, v in mod.state_dict().items()}
    assert got == CONTRACT["kitti." + name]
    assert list(got) == list(CONTRACT["kitti." + name])          # same order too


@pytest.mark.parametrize("name", ["DecoderWave", "SparseDecoderWave"])
def test_nyu_state_dict_contract(name):
    mod = getattr(nd, name)(enc_features=list(synth.DENSENET161_CH), decoder_width=0.5)
    got = {k: list(v.shape) for k, v in mod.state_dict().items()}
    assert got == CONTRACT["nyu." + name]


def test_convs_hold_only_conv_parameters():
    """KITTI/trainer.py:74-75 feeds decoder.convs to pyt_utils.group_weight, which asserts exactly this."""
    mod = kd.DepthWaveProgressiveDecoder(np.array(synth.RESNET18_CH))
    assert [k for k in mod.convs][:5] == [("upconv", 4, 0), ("upconv", 4, 1), ("waveconv", 4, 0), ("waveconv", 4, 1),
                                          ("waveconv", 4, -1)]
    for v in mod.convs.values():
        n_conv = sum(len(list(m.parameters(recurse=False))) for m in v.modules() if isinstance(m, nn.Conv2d))
        assert n_conv == len(list(v.parameters()))
    assert len(mod.decoder) == 17


def test_wavelet_modules_keep_dependency_api():
    idwt = wavelets.IDWT(wave="haar", mode="zero")
    dwt = wavelets.DWT(J=4, wave="haar", mode="reflect")
    assert set(idwt.state_dict()) == {"g0_col", "g1_col", "g0_row", "g1_row"}
    assert set(dwt.state_dict()) == {"h0_col", "h1_col", "h0_row", "h1_row"}
    assert idwt.g0_col.shape == (1, 1, 2, 1) and idwt.g1_row.shape == (1, 1, 1, 2)
    with pytest.raises(NotImplementedError):
        wavelets.DWTInverse(wave="db2")


def test_cpu_tensors_fail_loudly():
    """No CPU fallback: the product path refuses host tensors instead of silently computing elsewhere."""
    mod = kd.SparseDepthWaveProgressiveDecoder(np.array((8, 8, 16, 32, 64)))
    feats = [torch.zeros(s) for s in synth.kitti_feature_shapes(1, 64, 96, (8, 8, 16, 32, 64))]
    with pytest.raises(WmdError):
        mod(feats, 0.05)
    with pytest.raises(WmdError):
        wavelets.IDWT(wave="haar")((torch.zeros(1, 1, 4, 4), [torch.zeros(1, 1, 3, 4, 4)]))


def test_product_never_imports_the_oracle():
    import re
    root = os.path.dirname(os.path.abspath(kd.__file__))
    for fn in os.listdir(root):
        if fn.endswith(".py"):
            src = open(os.path.join(root, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn


def test_synthetic_generators_are_deterministic():
    a = synth.blocky_features([(2, 3, 8, 12)], seed=4, cell=4)[0]
    b = synth.blocky_features([(1, 3, 8, 12)], seed=5, cell=4)[0]
    assert torch.equal(a[1:], b)                      # sample n of a batch == stream seed+n
    sd = synth.random_state_dict({"c.weight": (4, 3, 3, 3), "c.bias": (4,)}, seed=1)
    assert abs(float(sd["c.weight"].abs().max())) <= 1 / np.sqrt(27) + 1e-7
    assert float(sd["c.weight"].double().sum()) == pytest.approx(-0.3225997, abs=1e-5)   # frozen MT19937 stream


def test_bench_byte_accounting_matches_the_survey_formulas():
    """bench.account(): the algorithmic bytes / flops behind `roofline.achieved` (SURVEY 8d, DESIGN.md 4)."""
    import bench
    n, h, w = 2, 8, 16
    assert bench.account("idwt_haar", dict(n=n, c=1, h=h, w=w, disp=False))[0] == 32 * n * h * w
    assert bench.account("idwt_haar", dict(n=n, c=1, h=h, w=w, disp=True))[0] == 48 * n * h * w
    assert bench.account("nchw_to_rows", dict(n=n, c=64, hw=h * w))[0] == 8 * n * 64 * h * w
    assert bench.account("nchw_to_rows", dict(n=n, c=64, hw=h * w, marked=10))[0] == 8 * 64 * 10 + n * h * w
    conv = dict(n=n, h=h, w=w, taps=9, c0=32, c1=16, cout=8, shift0=1, count=None, max_rows=n * h * w, m_in0=None, m_in1=None)
    by, fl = bench.account("conv_rows_tc", conv)
    m = n * h * w
    assert fl == 2 * 9 * 48 * 8 * m
    assert by == 4 * (n * (h // 2) * (w // 2) * 32 + m * 16 + m * 8) + 4 * (9 * 48 * 8 + 8)
    by, fl = bench.account("head_mlp", dict(c=32, n1=64, nz=54, count=None, max_rows=100))
    assert (by, fl) == (4 * 100 * (32 + 56) + 4 * (64 * 32 + 54 * 64 + 64), 2 * 100 * (32 * 64 + 64 * 54))
    recs = [("conv_rows_tc", 0.2, dict(conv, kind="tc")), ("idwt_haar", 0.01, dict(n=n, c=1, h=h, w=w, disp=True))] * 2
    table = bench.conv_layer_table(recs, 6500.0, 1600.0, 2)
    assert len(table) == 1 and table[0]["rows"] == m and table[0]["engine"] == "tcgen05_3xtf32"
    main, per_kernel = bench.roofline_from(recs, 6500.0, 1600.0, "test", 2, 1361.0)
    assert main["kernel"] == "conv_rows_tc" and main["bound"] == "tensor" and set(per_kernel) == {"conv_rows_tc", "idwt_haar"}
    assert main["step_view"]["algorithmic_bytes_per_step"] == by_sum(recs, bench) // 2
    assert main["operand_form"] == "tf32x3" and main["peak"] == 800.0            # no tf32 measurement given: bf16 / 2
    # the opt-in fp16-pair operand form is labelled and measured against the fp16 / bf16 tensor peak
    recs16 = [("conv_rows_tc", 0.2, dict(conv, kind="tc", f16=True))] * 2
    assert bench.conv_layer_table(recs16, 6500.0, 1600.0, 2)[0]["engine"] == "tcgen05_f16x3"
    main16, _ = bench.roofline_from(recs16, 6500.0, 1600.0, "test", 2, 1361.0, tf32_peak=760.0)
    assert main16["operand_form"].startswith("f16x3") and main16["peak"] == 1600.0


def test_bench_dump_outputs_fit_the_budget_and_repeat(tmp_path):
    """--dump-outputs: every output as <name>.npy in float32 / float64, small ones whole, large ones sampled at the same
    positions on every run, all within the byte budget."""
    import bench
    g = torch.Generator().manual_seed(0)
    out = {("disp", 0): torch.rand(4, 1, 64, 256, generator=g), ("disp", 3): torch.rand(4, 1, 8, 32, generator=g),
           ("wavelet_mask", 3): torch.rand(4, 1, 8, 32, generator=g) > 0.5, ("wavelets", 2, "LL"): torch.rand(4, 1, 32, 64),
           "total_ops": object()}
    ops = {"total_ops": 123456789012, "total_ops_per_sample": [1, 2, 3, 4]}
    budget = 64 << 10
    for run in ("a", "b"):
        bench.dump_outputs(out, ops, None, str(tmp_path / run), budget_bytes=budget)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(["disp_0.npy", "disp_3.npy", "wavelet_mask_3.npy", "wavelets_2_LL.npy", "total_ops.npy",
                            "total_ops_per_sample.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= budget
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "disp_3.npy"), out[("disp", 3)].numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "wavelet_mask_3.npy"), out[("wavelet_mask", 3)].float().numpy())
    assert np.load(tmp_path / "a" / "total_ops.npy") == 123456789012
    big = np.load(tmp_path / "a" / "disp_0.npy")
    assert big.ndim == 1 and 0 < big.size < out[("disp", 0)].numel()
    assert np.isin(big, out[("disp", 0)].numpy().reshape(-1)).all()


def by_sum(recs, bench):
    return sum(bench.account(name, info)[0] for name, _, info in recs)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the native one): one JSON line with the contract's
    keys, no GPU needed, bounded runtime."""
    import json
    import os
    import subprocess
    import sys
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(repo, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "kitti_r18_640x192_bs16"], capture_output=True, text=True, timeout=600, cwd=repo)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "decoder_frames_per_sec" and d["unit"] == "frames/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "kitti_r18_640x192_bs16"
