"""The gather-GEMM convolution engines against an fp64 restatement of the wmd_conv_desc contract (include/wmd.h).

conv_ref() below is that restatement: explicit int64 index arithmetic (pixel list, border rule, index maps, nearest
upsampling, gate) gathers every tap's source rows, a float64 matmul sums them, and bias + activation follow in fp64.
It runs on CPU and on CUDA (fp64, so TF32 switches do not apply).  The CPU tests pin it to F.conv2d and to the oracle;
the GPU tests hold both engines to it.

Bars, as max|y - ref| / max|ref| (helpers.rel_err): tcgen05 engine 1.5e-5 in the tf32x3 operand form and 1e-5 in the
f16x3 form (WMD_CONV_PRECISION), SIMT engine 1e-5.  The tcgen05 engine is fp32-faithful: 22-bit operand splits, three
MMAs per product, and a round-to-nearest drain of the round-toward-zero TMEM accumulators every 32 chunks (K = 1024).
Its error is the truncation bias of one epoch, so it does not grow with K: on one B200 (148 SMs, 1000 W power limit)
the worst case of every group of this file is 6.3e-6 .. 7.9e-6 in tf32x3 (three truncating MMAs per K = 8 step) and
3.5e-6 .. 4.0e-6 in f16x3 (three per K = 16 step); the SIMT engine stays under 1.2e-6.  Without the drain the long
cases (K = 18000 and 11520) measure 3.0e-5 .. 1.2e-4 in tf32x3 and 1.5e-5 .. 7.2e-5 in f16x3; weights without their
lo part, 1.5e-4 .. 3.2e-4 everywhere.

Every tcgen05 case first asserts the scheduling path it exists to cover (whole-tile rounds, balanced data-parallel
rounds + stream-K remainder, segments per tile, segment starts inside an epoch), from a mirror of the kernel's host
grid rule and of bal_plan driven by the device's SM count, so a GPU with another SM count cannot make a case silently
stop covering its path.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from wavelet_monodepth_b200._lib import (ACT_ELU, ACT_LRELU, ACT_NONE, ACT_SIGMOID, PAD_REFLECT, PAD_REPLICATE,
                                         PAD_ZERO)

from helpers import rel_err

BARS = {"tf32x3": 1.5e-5, "f16x3": 1e-5, "simt": 1e-5}
ACTS = {"none": ACT_NONE, "elu": ACT_ELU, "lrelu": ACT_LRELU, "sigmoid": ACT_SIGMOID}
PADS = {"zero": PAD_ZERO, "reflect": PAD_REFLECT, "replicate": PAD_REPLICATE}


# ------------------------------------------------------------------------------------------ fp64 reference
def _pad_coord(q, n, pad):
    """(q mapped into [0, n), inside) - pad_coord of the kernels, i.e. padding the index map (KITTI/layers.py:444)."""
    if pad == PAD_REFLECT:
        q = torch.where(q < 0, -q, q)
        return torch.where(q >= n, 2 * (n - 1) - q, q), torch.ones_like(q, dtype=torch.bool)
    if pad == PAD_REPLICATE:
        return q.clamp(0, n - 1), torch.ones_like(q, dtype=torch.bool)
    return q.clamp(0, n - 1), (q >= 0) & (q < n)


def _take(x, rows, valid, c):
    """fp64 x[rows, :c] where valid, 0 elsewhere.  Rows behind an invalid index, and columns past c, are never used:
    torch.where selects, so NaN there does not propagate."""
    g = x[rows.clamp(0, x.shape[0] - 1), :c].double()
    return torch.where(valid[:, None], g, torch.zeros((), dtype=torch.float64, device=x.device))


def activation_ref(v, act, p):
    if act == ACT_ELU:
        return torch.where(v > 0, v, torch.expm1(v))
    if act == ACT_LRELU:
        return torch.where(v > 0, v, v * p)
    if act == ACT_SIGMOID:
        return 1.0 / (1.0 + torch.exp(-v))
    return v


def conv_ref(x0, c0, weight, bias, n, h, w, taps=9, pad=PAD_REFLECT, act=ACT_NONE, act_param=0.0, map0=None, shift0=0,
             x1=None, c1=0, gate=None, map1=None, pixels=None, count=None):
    """fp64 rows (rows, cout) of wmd_conv_desc: for output row m (pixel p = pixels[m], or m), over the taps q of p,
      source 0: x0[row0(q), :c0], row0 = map0[n, qy >> shift0, qx >> shift0] (map0 None: that linear index;
                taps == 1 and map0 None: row m itself), zero if row0 < 0;
      source 1: x1[row1(q), :c1], row1 = map1[q] (map1 None: q), zero if row1 < 0;
      everything zero if gate[q] == 0 or q leaves the image under PAD_ZERO;
    y = act(bias + sum in(q) . w).  weight is the plain (cout, c0 + c1, k, k) tensor; count is an int."""
    dev = x0.device
    hw = h * w
    if pixels is None:
        p = torch.arange(n * hw, device=dev)
    else:
        p = pixels[:int(count)].long().to(dev)
    rows = p.numel()
    cout = weight.shape[0]
    pn, rem = p // hw, p % hw
    py, px = rem // w, rem % w
    hs, ws = h >> shift0, w >> shift0
    wt = weight.double().reshape(cout, c0 + c1, taps).to(dev)
    out = torch.zeros(rows, cout, dtype=torch.float64, device=dev)
    for tap in range(taps):
        qy, qx = (py + tap // 3 - 1, px + tap % 3 - 1) if taps == 9 else (py, px)
        qy, oky = _pad_coord(qy, h, pad)
        qx, okx = _pad_coord(qx, w, pad)
        ok = oky & okx
        q = (pn * h + qy) * w + qx
        if gate is not None:
            ok = ok & (gate.reshape(-1).to(dev)[q] != 0)
        if taps == 1 and map0 is None:
            r0 = torch.arange(rows, device=dev)
        else:
            qs = (pn * hs + (qy >> shift0)) * ws + (qx >> shift0)
            r0 = map0.reshape(-1).to(dev)[qs].long() if map0 is not None else qs
        a = _take(x0, r0, ok & (r0 >= 0), c0)
        if c1:
            r1 = map1.reshape(-1).to(dev)[q].long() if map1 is not None else q
            a = torch.cat([a, _take(x1, r1, ok & (r1 >= 0), c1)], 1)
        out += a @ wt[:, :, tap].t()
    if bias is not None:
        out += bias.double().to(dev)
    return activation_ref(out, act, act_param)


def compact(mask):
    """(idxmap int32 (N,H,W): running row over the batch or -1, pixels int32 of the active pixels, count) - what
    wmd_compact_mask produces, restated in torch."""
    flat = mask.reshape(-1) != 0
    run = torch.cumsum(flat.long(), 0) - 1
    idx = torch.where(flat, run, torch.full_like(run, -1)).to(torch.int32).reshape(mask.shape[0], *mask.shape[-2:])
    return idx, torch.nonzero(flat).reshape(-1).to(torch.int32), int(flat.sum())


def rnd(*shape, seed=0, lo=-1.0, hi=1.0):
    rs = np.random.RandomState(seed)
    return torch.from_numpy(rs.uniform(lo, hi, size=shape).astype(np.float32))


def blob_mask(n, h, w, p, seed, grow):
    """uint8 (n,h,w): random seeds dilated `grow` times by a 3x3 window - clustered like the decoder's dilated sets."""
    rs = np.random.RandomState(seed)
    m = torch.from_numpy((rs.uniform(size=(n, 1, h, w)) < p).astype(np.float32))
    for _ in range(grow):
        m = F.max_pool2d(m, 3, 1, 1)
    return m[:, 0].to(torch.uint8)


def nchw_rows(x):
    n, c, h, w = x.shape
    return x.permute(0, 2, 3, 1).reshape(n * h * w, c).contiguous()


# ------------------------------------------------------------------------------------------ CPU: pin the reference
@pytest.mark.parametrize("pad_name", ["reflect", "zero", "replicate"])
@pytest.mark.parametrize("act_name", ["none", "elu", "lrelu", "sigmoid"])
def test_reference_matches_conv2d_fp64(pad_name, act_name):
    pad, act = PADS[pad_name], ACTS[act_name]
    n, cin, cout, h, w = 2, 7, 5, 6, 9
    x = rnd(n, cin, h, w, seed=1).double()
    wt, b = rnd(cout, cin, 3, 3, seed=2).double(), rnd(cout, seed=3).double()
    mode = {"reflect": "reflect", "zero": "constant", "replicate": "replicate"}[pad_name]
    want = activation_ref(F.conv2d(F.pad(x, (1, 1, 1, 1), mode=mode), wt, b), act, 0.2)
    got = conv_ref(nchw_rows(x), cin, wt, b, n, h, w, pad=pad, act=act, act_param=0.2)
    assert rel_err(got, nchw_rows(want)) <= 1e-12
    # 1x1 form: row m reads row m; with a map it reads through the map
    w1 = rnd(cout, cin, 1, 1, seed=4).double()
    want1 = activation_ref(F.conv2d(x, w1, b), act, 0.2)
    assert rel_err(conv_ref(nchw_rows(x), cin, w1, b, n, h, w, taps=1, act=act, act_param=0.2), nchw_rows(want1)) <= 1e-12
    ident = torch.arange(n * h * w, dtype=torch.int32).reshape(n, h, w)
    assert rel_err(conv_ref(nchw_rows(x), cin, w1, b, n, h, w, taps=1, act=act, act_param=0.2, map0=ident),
                   nchw_rows(want1)) <= 1e-12


@pytest.mark.parametrize("pad_name", ["reflect", "zero", "replicate"])
def test_reference_two_sources_upsample_gate_list_matches_conv2d_fp64(pad_name):
    """shift0 = 1 (nearest upsampling of source 0), a dense skip source, a gate and an output list, against the same
    thing built densely: conv2d(pad(cat(up(x0), x1) * gate))."""
    pad = PADS[pad_name]
    n, c0, c1, cout, h, w = 2, 5, 3, 4, 8, 10
    lo, skip = rnd(n, c0, h // 2, w // 2, seed=5).double(), rnd(n, c1, h, w, seed=6).double()
    gate = blob_mask(n, h, w, 0.2, 7, 1)
    wt, b = rnd(cout, c0 + c1, 3, 3, seed=8).double(), rnd(cout, seed=9).double()
    xin = torch.cat([F.interpolate(lo, scale_factor=2, mode="nearest"), skip], 1) * gate[:, None].double()
    mode = {"reflect": "reflect", "zero": "constant", "replicate": "replicate"}[pad_name]
    want = nchw_rows(F.elu(F.conv2d(F.pad(xin, (1, 1, 1, 1), mode=mode), wt, b)))
    _, pixels, count = compact(blob_mask(n, h, w, 0.3, 10, 0))
    got = conv_ref(nchw_rows(lo), c0, wt, b, n, h, w, pad=pad, act=ACT_ELU, shift0=1, x1=nchw_rows(skip), c1=c1,
                   gate=gate, pixels=pixels, count=count)
    assert count > 0 and rel_err(got, want[pixels.long()]) <= 1e-12


@pytest.mark.parametrize("pad_name", ["reflect", "constant", "replicate"])
@pytest.mark.parametrize("p_in,p_out", [(0.6, 0.5), (0.1, 0.9), (1.0, 1.0), (0.0, 0.5)])
def test_reference_matches_oracle_sparse_conv(pad_name, p_in, p_out):
    """Sparse 3x3 on compact rows through an index map, at an output list (oracle.sparse_ops.conv3x3, fp32)."""
    from oracle import sparse_ops as osp
    cin, cout, h, w = 24, 40, 13, 17
    rs = np.random.RandomState(31)
    in_mask = torch.from_numpy((rs.uniform(size=(1, 1, h, w)) < p_in).astype(np.float32))
    out_mask = torch.from_numpy((rs.uniform(size=(1, 1, h, w)) < p_out).astype(np.float32))
    wt, b = rnd(cout, cin, 3, 3, seed=29, lo=-0.2, hi=0.2), rnd(cout, seed=30)
    xv = rnd(cin * int(in_mask.sum()), seed=40)
    idx, _ = osp.index_map(in_mask)
    want, _ = osp.conv3x3(wt, b, xv, idx, out_mask, nonlin=F.elu, padding=pad_name, make_result=True)
    map0, _, _ = compact(in_mask[:, 0])
    _, pixels, count = compact(out_mask[:, 0])
    rows = torch.cat([xv.reshape(cin, -1).t(), torch.zeros(1, cin)]).contiguous()
    got = conv_ref(rows, cin, wt, b, 1, h, w, pad=PADS["zero" if pad_name == "constant" else pad_name], act=ACT_ELU,
                   map0=map0, pixels=pixels, count=count)
    assert rel_err(got, nchw_rows(want)[pixels.long()]) <= 1e-6


def test_reference_matches_oracle_upsample_concat_gate_chain():
    """sparse_upsample + sparse_conv3x3 of one decoder level (depth_decoder.py:355-357) as one reference call."""
    from oracle import sparse_ops as osp
    c0, cs, cout, h, w = 16, 8, 32, 9, 11
    rs = np.random.RandomState(50)
    s0 = torch.from_numpy((rs.uniform(size=(1, 1, h, w)) < 0.25).astype(np.float32))
    u = F.interpolate(s0, scale_factor=2, mode="nearest")
    s2, s3, s4 = F.max_pool2d(s0, 5, 1, 2), F.max_pool2d(u, 5, 1, 2), F.max_pool2d(u, 3, 1, 1)
    xv = rnd(c0 * int(s2.sum()), seed=51)
    skip = rnd(1, cs, 2 * h, 2 * w, seed=52)
    wt, b = rnd(cout, c0 + cs, 3, 3, seed=53, lo=-0.2, hi=0.2), rnd(cout, seed=54)
    map2, _ = osp.index_map(s2)
    map3, _ = osp.index_map(s3)
    up, _ = osp.upsample_concat(xv, c0, map2, skip, s3, make_result=False)
    want, _ = osp.conv3x3(wt, b, up, map3, s4, nonlin=F.elu, padding="reflect", make_result=True)
    idx2, _, _ = compact(s2[:, 0])
    _, pix4, cnt4 = compact(s4[:, 0])
    got = conv_ref(xv.reshape(c0, -1).t().contiguous(), c0, wt, b, 1, 2 * h, 2 * w, act=ACT_ELU, map0=idx2, shift0=1,
                   x1=nchw_rows(skip), c1=cs, gate=s3[:, 0].to(torch.uint8), pixels=pix4, count=cnt4)
    assert rel_err(got, nchw_rows(want)[pix4.long()]) <= 1e-6
    # map1: the skip source as compact rows of the gate's pixels (skip[mask], KITTI/layers.py:500)
    map3i, pix3, _ = compact(s3[:, 0])
    got1 = conv_ref(xv.reshape(c0, -1).t().contiguous(), c0, wt, b, 1, 2 * h, 2 * w, act=ACT_ELU, map0=idx2, shift0=1,
                    x1=nchw_rows(skip)[pix3.long()], c1=cs, gate=s3[:, 0].to(torch.uint8), map1=map3i, pixels=pix4,
                    count=cnt4)
    assert rel_err(got1, got) <= 1e-15


# ------------------------------------------------------------------------------------------ scheduling mirror
TC_BM, FLUSH = 256, 32                 # tile rows; chunks per accumulation epoch (kFlushChunks)


def tile_n(cout):
    return 128 if cout >= 96 else (64 if cout >= 48 else 32)


def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def bal_plan(tiles, grid, nchunks):
    rounds = tiles // grid
    dp_rounds = rounds if tiles % grid == 0 else max(rounds - 1, 0)
    rem_tile0 = dp_rounds * grid
    rem_tiles = tiles - rem_tile0
    even = (rem_tiles * nchunks + grid - 1) // grid
    return rem_tile0, max(even, (nchunks + 5) // 6), (3 if rem_tiles >= grid else 8)


def schedule(rows, max_rows, cout, nchunks, splits, reserved=0):
    """What conv_rows_tc_kernel does with `rows` device rows: grid (launch_tc's rule), whole-tile rounds, and in balanced
    mode the data-parallel tiles and every stream-K segment (cta, tile, first chunk, end chunk)."""
    cap = sm_count() - reserved if sm_count() - reserved > 1 else 1
    nt = -(-cout // tile_n(cout))
    host_tiles = -(-max_rows // TC_BM) * nt
    grid = cap if splits == 0 else min(max(host_tiles, 1), cap)
    tiles = -(-rows // TC_BM) * nt
    s = dict(grid=grid, tiles=tiles, n_tiles=nt, nchunks=nchunks, rounds=-(-tiles // grid), segments=[])
    if splits == 0:
        rem_tile0, U, slabs = bal_plan(tiles, grid, nchunks)
        s.update(dp_tiles=rem_tile0, rem_tiles=tiles - rem_tile0, U=U, slabs=slabs)
        rem_units = (tiles - rem_tile0) * nchunks
        for cta in range(grid):
            u, u_end = cta * U, min(rem_units, (cta + 1) * U)
            while u < u_end:
                t = u // nchunks
                cb = u - t * nchunks
                ce = min(nchunks, cb + (u_end - u))
                s["segments"].append((cta, rem_tile0 + t, cb, ce))
                u += ce - cb
        per_tile = {}
        for _, t, cb, ce in s["segments"]:
            per_tile.setdefault(t, []).append((cb, ce))
        s["cut"] = {t: len(v) for t, v in per_tile.items() if len(v) > 1}
        assert all(v <= slabs for v in s["cut"].values())
    return s


def assert_epoch_crossing(s):
    """some stream-K segment starts inside an accumulation epoch and runs past the next epoch boundary"""
    assert s["U"] % FLUSH != 0, s["U"]
    assert any(cb % FLUSH != 0 and ce - cb > FLUSH for _, _, cb, ce in s["segments"]), s["segments"][:8]


# ------------------------------------------------------------------------------------------ GPU helpers
DEV = "cuda"


def _prec():
    from wavelet_monodepth_b200 import ops
    return ops.default_conv_precision()


def _amax(x, c):
    a = torch.nan_to_num(x[:, :c].float(), nan=0.0).abs().max() if x.shape[0] else torch.zeros(())
    return a.reshape(1).to(DEV)


def run_conv(kind, x0, c0, weight, bias, n, h, w, splits=None, precision=None, amax_out=None, **kw):
    """One launch through ops.conv_rows (engine `kind`, scheduling `splits`, operand form `precision`, default
    WMD_CONV_PRECISION); the f16x3 form gets the sources' max |x| as it would from their producers."""
    from wavelet_monodepth_b200 import ops
    precision = precision or _prec()
    c1 = kw.get("c1", 0)
    wp = ops.pack_weight(weight.to(DEV), c1, kind=kind, precision=precision)
    extra = {}
    if kind == "tc" and precision == "f16x3":
        extra["amax0"] = _amax(x0, c0)
        if c1:
            extra["amax1"] = _amax(kw["x1"], c1)
    return ops.conv_rows(x0, c0, wp, bias, weight.shape[0], n, h, w, splits=splits, amax_out=amax_out, **kw, **extra)


def check(got, want, what, bar=None):
    """rel_err within the bar of the engine / operand form (default: the tcgen05 engine in WMD_CONV_PRECISION)"""
    bar = bar or BARS[_prec()]
    e = rel_err(got, want)
    assert torch.isfinite(got).all(), what
    print("rel_err %.3e %s" % (e, what))
    assert e <= bar, (what, "rel err %.3e > %.1e" % (e, bar))
    return e


def dense_case(n, h, w, c0, cout, seed, c1=0):
    x0 = rnd(n * h * w, c0, seed=seed).to(DEV)
    x1 = rnd(n * h * w, c1, seed=seed + 1).to(DEV) if c1 else None
    wt = rnd(cout, c0 + c1, 3, 3, seed=seed + 2, lo=-0.1, hi=0.1)
    b = rnd(cout, seed=seed + 3).to(DEV)
    return x0, x1, wt, b


def list_case(rows, n, h, w, seed):
    """a sorted random list of `rows` pixels of an (n, h, w) grid, int32 on the device, and its device count"""
    g = torch.Generator().manual_seed(seed)
    pix = torch.randperm(n * h * w, generator=g)[:rows].sort()[0].to(torch.int32).to(DEV)
    return pix, torch.tensor([rows], dtype=torch.int32, device=DEV)


# ------------------------------------------------------------------------------------------ GPU: long reductions
@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 0])
def test_tc_long_reduction_single_source(splits):
    """c0 = 2000 (62.5 chunks: a channel tail), cout 256, 3x3: 567 chunks = 18 epochs (K = 18000), like upconv(4,0)."""
    n, h, w, c0, cout = 2, 48, 64, 2000, 256
    x0, _, wt, b = dense_case(n, h, w, c0, cout, seed=100)
    nch = 9 * -(-c0 // 32)
    s = schedule(n * h * w, n * h * w, cout, nch, splits)
    assert nch >= 560
    if splits == 0:
        assert s["dp_tiles"] == 0 and s["cut"] and any(t % 2 for t in s["cut"])   # fix-up on both N-tiles
        assert_epoch_crossing(s)
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, pad=PAD_REFLECT, act=ACT_ELU)
    want = conv_ref(x0, c0, wt, b, n, h, w, pad=PAD_REFLECT, act=ACT_ELU)
    check(y[:, :cout], want, ("long single source", splits))


@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 0])
def test_tc_long_reduction_two_sources_upsampled_and_gated(splits):
    """upconv(4,1) form: c0 = 1000 through map0 with shift0 = 1 plus a gated skip source c1 = 280 (K = 11520, both
    sources with a channel tail), at a sparse output list."""
    n, h, w, c0, c1, cout = 2, 64, 96, 1000, 280, 256
    lo_mask = blob_mask(n, h // 2, w // 2, 0.08, 110, 2)
    map0, _, m0 = compact(lo_mask)
    gate = F.interpolate(lo_mask[:, None].float(), scale_factor=2, mode="nearest")[:, 0].to(torch.uint8)
    out_mask = blob_mask(n, h, w, 0.05, 111, 2) * gate
    _, pixels, count = compact(out_mask)
    x0 = rnd(m0, c0, seed=112).to(DEV)
    x1 = rnd(n * h * w, c1, seed=113).to(DEV)
    wt, b = rnd(cout, c0 + c1, 3, 3, seed=114, lo=-0.1, hi=0.1), rnd(cout, seed=115).to(DEV)
    nch = 9 * (-(-c0 // 32) + -(-c1 // 32))
    s = schedule(count, n * h * w, cout, nch, splits)
    assert nch * 32 >= 11520 and s["tiles"] >= 16
    if splits == 0:
        assert s["cut"]
        assert_epoch_crossing(s)
    kw = dict(pad=PAD_REFLECT, act=ACT_LRELU, act_param=0.1, map0=map0.to(DEV), shift0=1, x1=x1, c1=c1,
              gate=gate.to(DEV), pixels=pixels.to(DEV), count=torch.tensor([count], dtype=torch.int32, device=DEV))
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)
    kw.pop("count")
    want = conv_ref(x0, c0, wt, b, n, h, w, count=count, **kw)
    check(y[:count, :cout], want, ("long two sources", splits))


# ------------------------------------------------------------------------------------------ GPU: scheduling shapes
def _sched_rows(shape, grid, n_tiles):
    """row count (never a multiple of 256) that gives the tile count `shape` asks for"""
    row_tiles = {"below_grid": 2,
                 "multiple_of_grid": grid,                          # with 2 N-tiles: tiles == 2 x grid
                 "between_grid_and_2grid": -(-3 * grid // (2 * n_tiles)),
                 "two_rounds_plus_remainder": -(-16 * grid // (5 * n_tiles)),
                 "whole_three_rounds": -(-13 * grid // (5 * n_tiles))}[shape]
    return row_tiles * TC_BM - 37


@pytest.mark.gpu
@pytest.mark.parametrize("shape,splits,cout", [("below_grid", 0, 256), ("multiple_of_grid", 0, 256),
                                               ("between_grid_and_2grid", 0, 138), ("two_rounds_plus_remainder", 0, 256),
                                               ("two_rounds_plus_remainder", 0, 138), ("whole_three_rounds", 1, 138)])
def test_tc_scheduling_shapes(shape, splits, cout):
    n, h, w, c0 = 4, 64, 256, 96
    nch = 9 * 3
    grid = sm_count()
    rows = _sched_rows(shape, grid, -(-cout // tile_n(cout)))
    assert rows % TC_BM and rows <= n * h * w
    s = schedule(rows, n * h * w, cout, nch, splits)
    g, t = s["grid"], s["tiles"]
    if shape == "below_grid":
        assert t < g and max(s["cut"].values()) >= 6
    elif shape == "multiple_of_grid":
        assert t == 2 * g and s["dp_tiles"] == t and not s["segments"]
    elif shape == "between_grid_and_2grid":
        assert g < t < 2 * g and s["dp_tiles"] == 0 and s["slabs"] == 3 and s["cut"]
    elif shape == "two_rounds_plus_remainder":
        assert s["dp_tiles"] >= 2 * g and s["rem_tiles"] >= g and s["cut"]
    else:
        assert s["rounds"] > 2
    if s.get("cut"):
        assert any(k % 2 for k in s["cut"]) and any(k % 2 == 0 for k in s["cut"])     # fix-ups on both N-tiles
    pix, cnt = list_case(rows, n, h, w, seed=120)
    x0 = rnd(n * h * w, c0, seed=121).to(DEV)
    wt, b = rnd(cout, c0, 3, 3, seed=122, lo=-0.1, hi=0.1), rnd(cout, seed=123).to(DEV)
    kw = dict(pad=PAD_ZERO, act=ACT_ELU, pixels=pix, count=cnt)
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)
    y2 = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)
    assert torch.equal(y[:rows, :cout], y2[:rows, :cout])
    want = conv_ref(x0, c0, wt, b, n, h, w, pad=PAD_ZERO, act=ACT_ELU, pixels=pix, count=rows)
    check(y[:rows, :cout], want, (shape, splits, cout))


# ------------------------------------------------------------------------------------------ GPU: device-side counts
@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 0])
@pytest.mark.parametrize("which", ["few", "zero", "all"])
def test_tc_device_count_leaves_the_rest_of_out_untouched(which, splits):
    """The tile count comes from *count on the device: rows >= count (and columns >= cout) of `out` keep the sentinel."""
    n, h, w, c0, cout = 2, 60, 100, 160, 138
    total = n * h * w
    rows = {"few": 700, "zero": 0, "all": total}[which]
    pix, _ = list_case(max(rows, 1), n, h, w, seed=130)
    cnt = torch.tensor([rows], dtype=torch.int32, device=DEV)
    x0, _, wt, b = dense_case(n, h, w, c0, cout, seed=131)
    if which != "zero":
        s = schedule(rows, total, cout, 9 * 5, splits)
        assert s["tiles"] < s["grid"] if which == "few" else s["tiles"] > s["grid"] // 2
    out = torch.full((total, 140), -12345.0, device=DEV)
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, pad=PAD_REPLICATE, act=ACT_SIGMOID, pixels=pix, count=cnt,
                 out=out)
    assert y.data_ptr() == out.data_ptr()
    torch.cuda.synchronize()
    assert bool((out[rows:] == -12345.0).all()) and bool((out[:, cout:] == -12345.0).all())
    if rows:
        want = conv_ref(x0, c0, wt, b, n, h, w, pad=PAD_REPLICATE, act=ACT_SIGMOID, pixels=pix, count=rows)
        check(out[:rows, :cout], want, (which, splits))


# ------------------------------------------------------------------------------------------ GPU: reserved SMs
@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 0])
def test_tc_reserved_sms(splits):
    """wmd_conv_tc_set_reserved_sms(k) shrinks the persistent grid.  Whole tiles: the bits do not depend on the grid.
    Balanced: the plan does (segments move), so the result is held to the bar, and is deterministic per grid."""
    from wavelet_monodepth_b200 import _lib
    lib = _lib.load()
    n, h, w, c0, cout = 4, 64, 80, 200, 256
    sms = sm_count()
    rows = (sms // 3 + 4) * TC_BM - 11                     # 2 x (sms/3 + 4) tiles: > 1 round on sms - sms/3 CTAs
    pix, cnt = list_case(rows, n, h, w, seed=140)
    x0, _, wt, b = dense_case(n, h, w, c0, cout, seed=141)
    kw = dict(pad=PAD_REFLECT, act=ACT_LRELU, act_param=0.2, pixels=pix, count=cnt)
    want = conv_ref(x0, c0, wt, b, n, h, w, pad=PAD_REFLECT, act=ACT_LRELU, act_param=0.2, pixels=pix, count=rows)
    nch = 9 * 7
    was = lib.wmd_conv_tc_set_reserved_sms(-1)
    try:
        lib.wmd_conv_tc_set_reserved_sms(0)
        base = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)[:rows, :cout].clone()
        check(base, want, ("reserved", 0, splits))
        assert schedule(rows, n * h * w, cout, nch, splits)["rounds"] == 1
        for k in (1, sms // 3, sms - 1):
            assert lib.wmd_conv_tc_set_reserved_sms(k) in (0, 1, sms // 3)
            s = schedule(rows, n * h * w, cout, nch, splits, reserved=k)
            assert s["grid"] <= max(sms - k, 1)
            if k > 1:
                assert s["rounds"] > 1 if splits == 1 else s["tiles"] > s["grid"]
            y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)[:rows, :cout].clone()
            if splits == 1:
                assert torch.equal(y, base), k
            else:
                check(y, want, ("reserved", k, splits))
                assert torch.equal(run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)[:rows, :cout], y), k
    finally:
        lib.wmd_conv_tc_set_reserved_sms(was)
    assert lib.wmd_conv_tc_set_reserved_sms(-1) == was


# ------------------------------------------------------------------------------------------ GPU: epilogues
@pytest.mark.gpu
@pytest.mark.parametrize("act_name", ["none", "elu", "lrelu", "sigmoid"])
@pytest.mark.parametrize("splits", [1, 0])
def test_tc_epilogue_activations_and_unaligned_bias_and_rows(act_name, splits):
    """Every activation in the per-tile epilogue (splits = 1, and the whole tiles of balanced mode) and in the stream-K
    fix-up (balanced mode, activate()).  A bias that is a 4-byte-offset view, and (whole tiles) an `out` with
    ldy = cout + 1, take the scalar path, which must give the vector path's bits; balanced mode refuses the odd ldy."""
    from wavelet_monodepth_b200 import _lib
    act = ACTS[act_name]
    n, h, w, c0, cout = 4, 64, 256, 160, 138
    x0, _, wt, b = dense_case(n, h, w, c0, cout, seed=150)
    rows = -(-5 * sm_count() // 4) * TC_BM - 37                       # 2.5 x grid tiles (2 N-tiles)
    pix, cnt = list_case(rows, n, h, w, seed=151)
    s = schedule(rows, n * h * w, cout, 9 * 5, splits)
    if splits == 0:
        assert s["dp_tiles"] > 0 and s["cut"]                           # whole tiles and stream-K fix-ups
    kw = dict(pad=PAD_REFLECT, act=act, act_param=0.15, pixels=pix, count=cnt)
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, **kw)[:rows]
    want = conv_ref(x0, c0, wt, b, n, h, w, **dict(kw, count=rows))
    check(y[:, :cout], want, (act_name, splits))
    bbuf = torch.empty(cout + 1, device=DEV)
    bbuf[1:] = b
    b_off = bbuf[1:]
    assert b_off.data_ptr() % 16 == 4
    y_b = run_conv("tc", x0, c0, wt, b_off, n, h, w, splits=splits, **kw)[:rows]
    assert torch.equal(y_b[:, :cout], y[:, :cout])
    odd = torch.full((rows, cout + 1), 7.0, device=DEV)
    if splits == 1:
        run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, out=odd, max_rows=rows, **kw)
        assert torch.equal(odd[:, :cout], y[:, :cout]) and bool((odd[:, cout] == 7.0).all())
    else:
        with pytest.raises(_lib.WmdError, match=r"status -2\b"):
            run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, out=odd, max_rows=rows, **kw)
        torch.cuda.synchronize()
        assert bool((odd == 7.0).all())


# ------------------------------------------------------------------------------------------ GPU: sources, tails, never-read data
def _sources_case(case):
    """(kwargs for conv_rows / conv_ref without the engine, x0, c0, weight, bias, n, h, w)"""
    rs_seed = {"c0_tail_two_sources": 160, "c1_tail": 161, "map1": 162, "tiled_1x1": 163, "tiled_1x1_list": 164,
               "tiled_1x1_gated": 165, "gathered_1x1_list": 166}[case]
    n, h, w = 2, 24, 34
    c0, c1, cout, taps = {"c0_tail_two_sources": (40, 64, 96), "c1_tail": (64, 24, 256), "map1": (72, 40, 64),
                          "tiled_1x1": (136, 0, 128), "tiled_1x1_list": (96, 20, 54), "tiled_1x1_gated": (128, 36, 64),
                          "gathered_1x1_list": (100, 0, 256)}[case] + ((1,) if "1x1" in case else (9,))
    wt = rnd(cout, c0 + c1, 3 if taps == 9 else 1, 3 if taps == 9 else 1, seed=rs_seed, lo=-0.1, hi=0.1)
    b = rnd(cout, seed=rs_seed + 1).to(DEV)
    x0 = rnd(n * h * w, c0, seed=rs_seed + 2).to(DEV)
    kw = dict(taps=taps, pad=PAD_REFLECT, act=ACT_ELU)
    if c1:
        kw.update(x1=rnd(n * h * w, c1, seed=rs_seed + 3).to(DEV), c1=c1)
    if case == "map1":
        skip_mask = blob_mask(n, h, w, 0.1, rs_seed + 4, 2)
        map1, spix, _ = compact(skip_mask)
        kw.update(x1=kw["x1"][spix.long().to(DEV)].contiguous(), map1=map1.to(DEV), gate=skip_mask.to(DEV))
    if case in ("tiled_1x1_list", "gathered_1x1_list", "map1"):
        _, pixels, count = compact(blob_mask(n, h, w, 0.1, rs_seed + 5, 1))
        kw.update(pixels=pixels.to(DEV), count=count)
    if case == "tiled_1x1_gated":
        kw.update(gate=blob_mask(n, h, w, 0.2, rs_seed + 6, 1).to(DEV))
    if case == "gathered_1x1_list":
        ident = torch.arange(n * h * w, dtype=torch.int32).reshape(n, h, w)
        kw.update(map0=ident.flip(-1).contiguous().to(DEV))      # through a map: per-row gathers, not the tiled load
    return kw, x0, c0, wt, b, n, h, w


def _launch_and_ref(kind, splits, kw, x0, c0, wt, b, n, h, w):
    kw = dict(kw)
    count = kw.pop("count", None)
    ckw = dict(kw, count=torch.tensor([count], dtype=torch.int32, device=DEV)) if count is not None else kw
    y = run_conv(kind, x0, c0, wt, b, n, h, w, splits=splits, **ckw)
    want = conv_ref(x0, c0, wt, b, n, h, w, count=count, **kw)
    return y[:want.shape[0], :wt.shape[0]], want


SOURCE_CASES = ["c0_tail_two_sources", "c1_tail", "map1", "tiled_1x1", "tiled_1x1_list", "tiled_1x1_gated",
                "gathered_1x1_list"]


@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 0])
@pytest.mark.parametrize("case", SOURCE_CASES)
def test_tc_sources_and_channel_tails(case, splits):
    kw, x0, c0, wt, b, n, h, w = _sources_case(case)
    if case.startswith("tiled"):
        assert x0.shape[0] % TC_BM and "map0" not in kw          # rows0 not a multiple of 256: zero-filled tail box
    y, want = _launch_and_ref("tc", splits, kw, x0, c0, wt, b, n, h, w)
    check(y, want, (case, splits))


def _poison(kw, x0, c0, extra_cols=8):
    """NaN in everything the contract says is never read: columns c0..ld0 of x0 (ld0 > pad4(c0)) and of x1, x0 rows
    no map entry references, x1 rows under gate == 0."""
    nan = float("nan")
    ld0 = (c0 + 3) // 4 * 4 + extra_cols
    p0 = torch.full((x0.shape[0] + 300, ld0), nan, device=DEV)
    p0[:x0.shape[0], :c0] = x0
    if kw.get("map0") is not None:
        used = torch.zeros(x0.shape[0] + 300, dtype=torch.bool, device=DEV)
        m = kw["map0"].reshape(-1).long()
        used[m[m >= 0]] = True
        p0[~used] = nan
    kw = dict(kw)
    if kw.get("c1"):
        c1, x1 = kw["c1"], kw["x1"]
        p1 = torch.full((x1.shape[0], (c1 + 3) // 4 * 4 + 4), nan, device=DEV)
        p1[:, :c1] = x1
        if kw.get("gate") is not None and kw.get("map1") is None:
            p1[kw["gate"].reshape(-1) == 0] = nan
        kw["x1"] = p1
    return kw, p0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,splits", [("tc", 1), ("tc", 0), ("simt", None)])
@pytest.mark.parametrize("case", ["upsample_skip_gate", "sparse_map0", "map1", "c0_tail_two_sources"])
def test_never_read_rows_and_columns_hold_nan(case, kind, splits):
    """Padding columns, unreferenced rows and gated-off skip rows are NaN: the output stays finite and on the bar."""
    if case in ("map1", "c0_tail_two_sources"):
        kw, x0, c0, wt, b, n, h, w = _sources_case(case)
    else:
        n, h, w, c0, c1, cout = 2, 32, 48, 70, 36, 64 if kind == "tc" else 24
        lo_mask = blob_mask(n, h // 2, w // 2, 0.15, 170, 1)
        map0, _, m0 = compact(lo_mask)
        x0 = rnd(m0, c0, seed=171).to(DEV)
        b = rnd(cout, seed=172).to(DEV)
        _, pixels, count = compact(blob_mask(n, h, w, 0.1, 173, 1))
        kw = dict(pad=PAD_ZERO, act=ACT_LRELU, act_param=0.1, pixels=pixels.to(DEV), count=count)
        if case == "upsample_skip_gate":
            gate = F.interpolate(lo_mask[:, None].float(), scale_factor=2, mode="nearest")[:, 0].to(torch.uint8)
            kw.update(map0=map0.to(DEV), shift0=1, x1=rnd(n * h * w, c1, seed=174).to(DEV), c1=c1, gate=gate.to(DEV))
        else:
            h, w = h // 2, w // 2
            c1 = 0
            _, pixels, count = compact(blob_mask(n, h, w, 0.2, 175, 1))
            kw.update(map0=map0.to(DEV), pixels=pixels.to(DEV), count=count)
        wt = rnd(cout, c0 + c1, 3, 3, seed=176, lo=-0.1, hi=0.1)
    if kind == "simt":
        wt, b = wt[:24], b[:24]
    kw, x0p = _poison(kw, x0, c0)
    assert torch.isnan(x0p).any()
    y, want = _launch_and_ref(kind, splits, kw, x0p, c0, wt, b, n, h, w)
    check(y, want, (case, kind, splits), BARS["simt"] if kind == "simt" else None)


# ------------------------------------------------------------------------------------------ GPU: f16x3 operand form
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["long_whole", "long_balanced", "two_rounds_plus_remainder"])
def test_tc_f16x3_and_amax_out(case):
    """precision = f16x3 on the long and the multi-round balanced cases; amax_out is exactly max |y| over the rows
    written, in the per-tile epilogue and in the stream-K fix-up."""
    if case.startswith("long"):
        n, h, w, c0, cout = 2, 48, 64, 2000, 256
        rows, splits = n * h * w, (1 if case == "long_whole" else 0)
        pix = cnt = None
    else:
        n, h, w, c0, cout = 4, 64, 256, 96, 256
        rows, splits = _sched_rows(case, sm_count(), 2), 0
        pix, cnt = list_case(rows, n, h, w, seed=180)
    x0, _, wt, b = dense_case(n, h, w, c0, cout, seed=181)
    x0 = x0 * 37.0
    s = schedule(rows, n * h * w, cout, 9 * -(-c0 // 32), splits)
    if splits == 0:
        assert s["cut"] and (case == "long_balanced" or s["dp_tiles"] >= 2 * s["grid"])
    am = torch.zeros(1, device=DEV)
    kw = dict(pad=PAD_REFLECT, act=ACT_ELU, pixels=pix, count=cnt)
    y = run_conv("tc", x0, c0, wt, b, n, h, w, splits=splits, precision="f16x3", amax_out=am, **kw)
    kw["count"] = rows if cnt is not None else None
    want = conv_ref(x0, c0, wt, b, n, h, w, **kw)
    check(y[:rows, :cout], want, ("f16x3", case), BARS["f16x3"])
    assert float(am[0]) == float(y[:rows, :cout].abs().max())


# ------------------------------------------------------------------------------------------ GPU: SIMT engine
@pytest.mark.gpu
@pytest.mark.parametrize("cout,c0,c1,taps,form", [(1, 32, 0, 9, "dense"), (3, 64, 0, 9, "sparse"), (5, 6, 0, 9, "dense"),
                                                  (16, 24, 8, 9, "upsample_gate"), (31, 40, 0, 9, "sparse"),
                                                  (16, 96, 0, 1, "dense"), (54, 12, 0, 9, "dense")])
def test_simt_matches_fp64_reference(cout, c0, c1, taps, form):
    """The FMA tiles take the layers the tcgen05 engine does not (cout < 32 or K < 128): heads, thin stages."""
    n, h, w = 2, 18, 26
    k = 3 if taps == 9 else 1
    wt, b = rnd(cout, c0 + c1, k, k, seed=190 + cout, lo=-0.2, hi=0.2), rnd(cout, seed=191).to(DEV)
    kw = dict(taps=taps, pad={1: PAD_REFLECT, 3: PAD_ZERO, 5: PAD_REPLICATE}.get(cout, PAD_REFLECT), act=ACT_SIGMOID)
    if form == "dense":
        x0 = rnd(n * h * w, c0, seed=192).to(DEV)
    elif form == "sparse":
        map0, _, m0 = compact(blob_mask(n, h, w, 0.2, 193, 1))
        _, pixels, count = compact(blob_mask(n, h, w, 0.15, 194, 1))
        x0 = rnd(m0, c0, seed=195).to(DEV)
        kw.update(map0=map0.to(DEV), pixels=pixels.to(DEV), count=count)
    else:
        lo_mask = blob_mask(n, h // 2, w // 2, 0.2, 196, 1)
        map0, _, m0 = compact(lo_mask)
        gate = F.interpolate(lo_mask[:, None].float(), scale_factor=2, mode="nearest")[:, 0].to(torch.uint8)
        _, pixels, count = compact(blob_mask(n, h, w, 0.1, 197, 1) * gate)
        x0 = rnd(m0, c0, seed=198).to(DEV)
        kw.update(map0=map0.to(DEV), shift0=1, x1=rnd(n * h * w, c1, seed=199).to(DEV), c1=c1, gate=gate.to(DEV),
                  pixels=pixels.to(DEV), count=count)
    x0 = F.pad(x0, (0, -c0 % 4))                                  # row pitch: a multiple of 4 floats
    y, want = _launch_and_ref("simt", None, kw, x0, c0, wt, b, n, h, w)
    check(y, want, ("simt", cout, form), BARS["simt"])
