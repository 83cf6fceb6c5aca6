"""Per-convolution timing of the fused engine at chosen steps of the T=50 trajectory (development aid).
Usage: python scripts/profile_layers.py [steps to report, e.g. 0 10 49]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.argv = sys.argv[:1] + sys.argv[1:]
import bench  # noqa: E402


def waste_report(geom, sizes):
    """issued (tile, offset) slots x 128 rows over real (in, out) pairs of the 3^3 maps, for the current row order and for a
    full sort of the rows by their 27-bit neighbour mask (what a better lb2_row_order could reach)"""
    import numpy as np
    pc = np.array([bin(i).count("1") for i in range(1 << 16)])

    def popc(m):
        return pc[m & 0xffff] + pc[m >> 16]

    def issued(mm):
        n = len(mm)
        mm = np.concatenate([mm, np.zeros((-n) % 128, np.uint32)]).reshape(-1, 128)
        return int(popc(np.bitwise_or.reduce(mm, axis=1)).sum()) * 128
    for l, n in enumerate(sizes):
        nbr = geom.nbr3[l]
        m = geom.mask_of[nbr.data_ptr()][:n].cpu().numpy().astype(np.uint32)
        perm = geom.perm3[l][:n].cpu().numpy()
        pairs = int(popc(m).sum())
        cur, lex, ident = issued(m[perm]), issued(np.sort(m)), issued(m)
        print(f"  waste L{l}: rows {n} pairs/row {pairs / n:.2f}; issued/pairs natural {ident / pairs:.2f} current {cur / pairs:.2f} mask-sorted {lex / pairs:.2f}")
        if l < 2:
            continue
        # dense / residual split of the CTA-pair kernel's 256-row super-tiles (lb2_tile_split) for a few tau: issued dense slots x 256
        # rows over pairs, and the compacted residual pairs over pairs (LB2_PROFILE_TAUS="0.25,0.5,0.75")
        mp = m[perm]
        mp = np.concatenate([mp, np.zeros((-n) % 256, np.uint32)]).reshape(-1, 256)
        cnt = ((mp[:, :, None] >> np.arange(27, dtype=np.uint32)) & 1).sum(1)             # super-tiles x offsets: rows that have it
        full = int(popc(np.bitwise_or.reduce(mp, axis=1)).sum()) * 256
        row = [f"union {full / pairs:.2f}"]
        for tau in [float(t) for t in os.environ.get("LB2_PROFILE_TAUS", "0.25,0.5,0.75").split(",")]:
            keep = cnt >= int(np.ceil(tau * 256))
            dense = int(keep.sum()) * 256
            res = int((cnt * ~keep).sum())
            row.append(f"tau {tau}: {dense / pairs:.2f} + {res / pairs:.2f}")
        print(f"  split L{l} (issued dense slots / pairs + compacted pairs / pairs): " + "; ".join(row))


def main():
    report = [int(a) for a in sys.argv[1:]] or [0, 10, 25, 49]
    dev = torch.device("cuda", 0)
    scan, start, g = bench.build_inputs(dev, 0)
    pipe = bench.build_pipeline(dev, scan)
    eng = pipe.engine()
    K = 50
    noise = torch.randn((K, bench.N_POINTS, 3), device=dev, generator=g)
    x_feats = (scan + start).float()
    st = eng.start(scan, x_feats)
    for i in range(3):
        eng.advance(st, noise[i])
    st = eng.start(scan, x_feats)
    torch.cuda.synchronize()
    for i in range(K):
        rec = i in report
        if rec:
            eng.conv_events, eng.layer_log = [], []
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        eng.advance(st, noise[i])
        if rec:
            e1.record()
            torch.cuda.synchronize()
            ev, log = eng.conv_events, eng.layer_log
            eng.conv_events = eng.layer_log = None
            sizes = eng.geom.sizes()
            pairs = eng.geom.pairs.cpu().tolist()
            print(f"\n=== step {i}: {e0.elapsed_time(e1):.2f} ms total; rows {sizes}; 3^3 pairs {pairs[:5]}")
            tot = 0.0
            by_level = {}
            for (a, b, j), ent in zip(ev, log):
                ms = a.elapsed_time(b)
                tot += ms
                lvl = [d.data_ptr() for d in eng.geom.d_n].index(ent["d_m"]) if ent["d_m"] in [d.data_ptr() for d in eng.geom.d_n] else -1
                by_level[lvl] = by_level.get(lvl, 0.0) + ms
                print(f"  {ent['name']:24s} L{lvl} k{ent['kvol']:2d} {ent['cin']:3d}->{ent['cout']:3d} p{ent['npass']} {'scatter' if ent['scatter'] else '       '} {ms:7.3f} ms")
            print(f"  conv total {tot:.2f} ms; by level {dict(sorted(by_level.items()))}")
            if os.environ.get("LB2_PROFILE_WASTE"):
                waste_report(eng.geom, sizes)


if __name__ == "__main__":
    main()
