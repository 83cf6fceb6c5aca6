"""Dense / residual split of the Cout-256 convolutions (lb2_tile_split + masked lb2_pair_list + lb2_spconv_scatter into `pre_add`
+ the CTA-pair kernel on the dense masks) against the fp64 oracle, and the split's pair bookkeeping against the kernel map."""
import math

import numpy as np
import pytest
import torch

from oracle import me_cpu as ome

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def rel_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).abs() / (b.abs() + b.pow(2).mean().sqrt() + 1e-30)).max().item()


@pytest.fixture(scope="module")
def geo():
    from lidiff_b200 import _lib
    from lidiff_b200.engine import Geometry
    h = _lib.get_handle(DEV)
    g = torch.Generator().manual_seed(77)
    n = 60_000
    pts = torch.randn(n, 3, generator=g) * torch.tensor([3.0, 3.0, 0.6])         # a slab: 10-20 neighbours per voxel on levels 2-4
    coords = torch.cat([torch.zeros(n, 1), torch.round(pts / 0.05)], 1)
    G = Geometry(h, n)
    G.build(coords.to(DEV).contiguous(), n)
    og = ome.TensorField(pts, coords).sparse().geom
    return dict(h=h, G=G, og=og, n=n, sizes=G.sizes())


def _split(geo, lvl, tau):
    h, G, N = geo["h"], geo["G"], geo["n"]
    i32 = dict(dtype=torch.int32, device=DEV)
    nbr, perm = G.nbr3[lvl], G.perm3[lvl]
    mask = G.mask_of[nbr.data_ptr()]
    dense, res = torch.full((N,), -1, **i32), torch.full((N,), -1, **i32)
    h.tile_split(mask, perm, G.d_n[lvl], N, 27, math.ceil(tau * 256), dense, res)
    to = (torch.zeros((N + 127) // 128, **i32), torch.zeros((N + 255) // 256, **i32))
    h.tile_order(dense, perm, G.d_n[lvl], N, to[0], to[1], torch.zeros((N + 127) // 128, **i32))
    p_in, p_out, koff, toff = torch.zeros(27 * N, **i32), torch.zeros(27 * N, **i32), torch.zeros(28, **i32), torch.zeros(28, **i32)
    h.pair_list(nbr, N, G.d_n[lvl], N, 27, -1, p_in, p_out, koff, toff, torch.zeros(64, **i32), row_mask=res)
    torch.cuda.synchronize()
    return mask, dense, res, to, p_in, p_out, koff, toff


@pytest.mark.parametrize("lvl", [3, 4])
@pytest.mark.parametrize("tau", [0.0, 0.25, 0.5, 1.0])
def test_split_partitions_the_pair_set(geo, lvl, tau):
    G, M = geo["G"], geo["sizes"][lvl]
    mask, dense, res, _, p_in, p_out, koff, _ = _split(geo, lvl, tau)
    m, d, r = (x[:M].cpu().numpy().astype(np.uint32) for x in (mask, dense, res))
    assert np.all(d | r == m) and np.all(d & r == 0)
    perm = G.perm3[lvl][:M].cpu().numpy()
    bits = (m[perm][:, None] >> np.arange(27)) & 1                                   # rows in execution order x offsets
    for t in range(0, M, 256):                                                      # dense offsets of each 256-row super-tile
        keep = bits[t:t + 256].sum(0) >= math.ceil(tau * 256)
        rows = perm[t:t + 256]
        want = np.bitwise_or.reduce(np.where(keep, 1 << np.arange(27), 0).astype(np.uint32))
        assert np.all(d[rows] == (m[rows] & want))
    if tau == 0.0:
        assert np.all(d == m) and koff[27].item() == 0
    nbr = G.nbr3[lvl][:, :M].cpu().numpy()
    ko = koff.cpu().numpy()
    pin, pout = p_in.cpu().numpy(), p_out.cpu().numpy()
    got = []
    for k in range(27):
        o = pout[ko[k]:ko[k + 1]]
        assert np.all(pin[ko[k]:ko[k + 1]] == nbr[k, o]), "pair_in is the map's neighbour"
        got.append(k * M + o.astype(np.int64))
    got = np.concatenate(got)
    ks, os_ = np.nonzero((d[None, :] >> np.arange(27)[:, None]) & 1)
    every = np.sort(np.concatenate([got, ks * M + os_]))
    ks, os_ = np.nonzero(nbr >= 0)
    assert np.array_equal(every, np.sort(ks * M + os_)), "dense slots + compacted pairs = the 3^3 pair set, no pair lost or repeated"


CASES = [(256, 0, 256, 3), (256, 128, 256, 3), (128, 0, 256, 4), (256, 0, 256, 4)]   # c1, c2, cout, level


def _run_split_conv(geo, tau, c1, c2, cout, lvl, algo="pair"):
    """scatter of the residual pairs into pre_add + the convolution of the dense masks; algo: 'pair' (CTA-pair kernel), 'tile'
    (LB2_ALGO_TC_TILE), 'ffma' (CUDA cores, fp32 inputs).  tau None: the map's own masks; tau None or 0: no pre-pass, no pre_add
    (what the engine runs without the split)."""
    from lidiff_b200 import _lib
    from lidiff_b200._lib import ConvDesc, ConvIO, ScatterDesc
    h, G, og, N = geo["h"], geo["G"], geo["og"], geo["n"]
    assert h.scatter_supported(c1, c2, cout, 27)
    _, dense, _, to, p_in, p_out, koff, toff = _split(geo, lvl, tau or 0.0)
    if tau is None:
        dense = G.mask_of[G.nbr3[lvl].data_ptr()]
        to = G.tile_order_of[G.nbr3[lvl].data_ptr()]
    gen = torch.Generator().manual_seed(c1 * 7 + c2 + cout + lvl)
    W = torch.randn(27, c1 + c2, cout, generator=gen) / np.sqrt((c1 + c2) * 27)
    A = torch.randn(2, N, c1, generator=gen)
    B = torch.randn(2, N, c2, generator=gen) if c2 else None
    R = torch.randn(2, N, cout, generator=gen)
    sc_, sh_ = torch.rand(cout, generator=gen) + 0.5, torch.randn(cout, generator=gen)
    tab = torch.randn(40, cout, generator=gen)
    gi = torch.randint(0, 40, (N,), generator=gen, dtype=torch.int32)
    d_ = lambda t: None if t is None else t.to(DEV).contiguous()
    dW, dA, dB, dR, dS, dT, dTab, dGi = map(d_, (W, A, B, R, sc_, sh_, tab, gi))
    Wp = h.pack_weights(dW)

    def split_of(x):                                   # fp16 hi/lo companion through the library's own split (gate_mul by 1)
        if x is None:
            return None
        c = x.shape[-1]
        one = torch.ones(1, c, device=DEV)
        xh = torch.zeros(2, N, 2 * c, dtype=torch.float16, device=DEV)
        for p_ in range(2):
            h.gate_mul(x[p_], one, None, None, N, c, torch.empty_like(x[p_]), xh[p_])
        return xh
    A_h, B_h = split_of(dA), split_of(dB)
    pre = torch.full((2, N, cout), float("nan"), device=DEV)             # rows up to the live count are cleared by the scatter launch
    sd = ScatterDesc()
    sd.c1, sd.c2, sd.cout, sd.kvol = c1, c2, cout, 27
    sd.weight_packed = Wp.data_ptr()
    sd.pair_in, sd.pair_out, sd.koff, sd.tile_off = p_in.data_ptr(), p_out.data_ptr(), koff.data_ptr(), toff.data_ptr()
    sd.npass = 2
    for p_ in range(2):                                 # companions only (lean activations)
        sd.in1[p_], sd.in2[p_], sd.out[p_] = None, None, pre[p_].data_ptr()
        sd.in1_h[p_], sd.in2_h[p_] = A_h[p_].data_ptr(), B_h[p_].data_ptr() if B_h is not None else None
    sd.d_zero_rows, sd.zero_rows_cap = G.d_n[lvl].data_ptr(), N
    out, outg = torch.zeros(2, N, cout, device=DEV), torch.zeros(2, N, cout, device=DEV)
    out_h = torch.zeros(2, N, 2 * cout, dtype=torch.float16, device=DEV)
    d = ConvDesc()
    d.c1, d.c2, d.cout, d.kvol = c1, c2, cout, 27
    d.weight, d.weight_packed = dW.data_ptr(), Wp.data_ptr()
    d.scale, d.shift, d.relu = dS.data_ptr(), dT.data_ptr(), 1
    nbr = G.nbr3[lvl]
    d.nbr, d.nbr_stride, d.d_mout, d.mout_cap, d.npass = nbr.data_ptr(), N, G.d_n[lvl].data_ptr(), N, 2
    d.row_perm, d.row_mask = G.perm3[lvl].data_ptr(), dense.data_ptr()
    d.tile_order128, d.tile_order256 = to[0].data_ptr(), to[1].data_ptr()
    for p_ in range(2):
        d.io[p_] = ConvIO(None, None, dR[p_].data_ptr(), out[p_].data_ptr(), dTab.data_ptr(), dGi.data_ptr() if p_ == 0 else None,
                          outg[p_].data_ptr(), pre[p_].data_ptr(), A_h[p_].data_ptr(), B_h[p_].data_ptr() if B_h is not None else None,
                          out_h[p_].data_ptr(), None)
    if not tau:
        for p_ in range(2):
            d.io[p_].pre_add = None
    if algo == "ffma":                                  # the CUDA-core kernel reads fp32 inputs
        for p_ in range(2):
            d.io[p_].in1, d.io[p_].in2 = dA[p_].data_ptr(), dB[p_].data_ptr() if dB is not None else None
    old = h.get_option(_lib.OPT_TC_PAIR)
    h.set_option(_lib.OPT_TC_PAIR, 2)
    try:
        if tau:
            h.spconv_scatter(sd)
        h.spconv(d, {"pair": _lib.ALGO_TC, "tile": _lib.ALGO_TC_TILE, "ffma": _lib.ALGO_FFMA}[algo])
        torch.cuda.synchronize()
    finally:
        h.set_option(_lib.OPT_TC_PAIR, old)
    return out, outg, out_h, koff, (A, B, W, R, sc_, sh_, tab, gi)


def _check_oracle(geo, res, c1, c2, cout, lvl, what):
    og, M = geo["og"], geo["sizes"][lvl]
    out, outg, out_h, koff, (A, B, W, R, sc_, sh_, tab, gi) = res
    for p_ in range(2):
        Fin = A[p_][:M] if B is None else torch.cat([A[p_][:M], B[p_][:M]], 1)
        y = ome.conv(ome.SparseTensor(Fin.double(), og, 1 << lvl), W.double(), 3, 1, False).F
        y = torch.relu(y * sc_.double() + sh_.double() + R[p_][:M].double())
        e = rel_err(out[p_][:M], y)
        gate = tab[gi[:M].long()] if p_ == 0 else tab[0:1]
        eg = rel_err(outg[p_][:M], y * gate.double())
        oh = out_h[p_][:M].float().cpu()
        es = rel_err(oh[:, :cout] + oh[:, cout:], y)
        print(f"{what} {c1}+{c2}->{cout} L{lvl} pass {p_}: {koff[27].item()} compacted pairs; rel err {e:.2e} gated {eg:.2e} split {es:.2e}")
        assert e < 5e-5 and eg < 5e-5 and es < 5e-5, "split convolution vs fp64 oracle"
    assert out[:, M:].abs().sum() == 0, "rows beyond the live count must stay untouched"


@pytest.mark.parametrize("tau", [0.25, 0.5, 1.0])
@pytest.mark.parametrize("c1,c2,cout,lvl", CASES)
def test_split_conv_matches_fp64_oracle(geo, tau, c1, c2, cout, lvl):
    _check_oracle(geo, _run_split_conv(geo, tau, c1, c2, cout, lvl), c1, c2, cout, lvl, f"pair tau={tau}")


@pytest.mark.parametrize("algo", ["tile", "ffma"])
def test_split_conv_on_every_kernel(geo, algo):
    """the dense masks are the exact offset set for every kernel that lb2_spconv_forward can reach, not only the CTA-pair kernel"""
    res = _run_split_conv(geo, 0.5, 256, 128, 256, 3, algo)
    assert res[3][27].item() > 0
    _check_oracle(geo, res, 256, 128, 256, 3, f"{algo} tau=0.5")


def test_split_tau0_is_bit_identical(geo):
    """tau = 0 keeps every offset: the dense masks equal the map's masks and the convolution gives the unsplit bits"""
    a = _run_split_conv(geo, None, 256, 0, 256, 3)
    b = _run_split_conv(geo, 0.0, 256, 0, 256, 3)
    assert b[3][27].item() == 0
    for x, y in zip(a[:3], b[:3]):
        assert torch.equal(x, y)


def test_engine_split_step_matches_unsplit(monkeypatch):
    """one engine step with the split on levels 3-4 against the same step without it (fp32 reassociation only)"""
    import sys
    import os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from conftest import make_scan
    from oracle.pipeline import calibrated_state_dicts
    from lidiff_b200.engine import DenoiseEngine
    scan = make_scan(2000, 0)
    sds = calibrated_state_dicts(scan, seed=0)
    g = torch.Generator().manual_seed(5)
    start = torch.randn(scan.shape, generator=g)
    noise = torch.randn(scan.shape[1:], generator=g).to(DEV)
    eps = {}
    for tau in ("3:0,4:0", "3:0.5,4:0.5"):
        monkeypatch.setenv("LB2_SPLIT_TAU", tau)
        eng = DenoiseEngine(sds["enc"], sds["diff"], device=DEV, n_points=scan.shape[1], denoising_steps=50)
        on = tau != "3:0,4:0"
        assert bool(eng.geom.split_min_rows) == on
        st = eng.start(scan, scan + start)
        e = torch.empty((scan.shape[1], 3), device=DEV)
        eng.layer_log = []
        eng.step(0, st["xa"], st["xb"], st["ca"], st["cb"], st["x_init"], noise, st["x0s"], eps_out=e)
        torch.cuda.synchronize()
        geom = eng.geom
        assert sorted(geom.split_of) == sorted(geom.nbr3[l].data_ptr() for l in ((3, 4) if on else ()))
        # the level-3/4 Cout-256 3^3 layers (stage4 and up1 blocks) ran the scatter pre-pass, nothing else did
        split_layers = [x["name"] for x in eng.layer_log if x["scatter"]]
        want = [x["name"] for x in eng.layer_log if x["cout"] == 256 and x["kvol"] == 27 and x["map"] in geom.split_of]
        assert split_layers == want and (len(want) == 8 if on else not want), (split_layers, want)
        if on:
            assert all(geom.split_bufs[l][5][27].item() > 0 for l in (3, 4)), "compacted residual pairs exist"
        eps[tau] = e.double().cpu()
    a, b = eps["3:0.5,4:0.5"], eps["3:0,4:0"]
    r = ((a - b).abs() / (b.abs() + b.pow(2).mean().sqrt())).max().item()
    print(f"engine step, split on L3-4 vs off: max rel diff {r:.2e}")
    assert r < 1e-4
