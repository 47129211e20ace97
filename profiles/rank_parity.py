#!/usr/bin/env python
"""Bit-identity of the tail / relation / pair ranking outputs between two checkouts, and their construction times.

    python profiles/rank_parity.py --other DIR --out OUTDIR

DIR is another checkout of the repository, built (e.g. the parent commit).  Each checkout is imported in a
subprocess of its own (`--dump ROOT FILE`), which computes on the same seeded inputs: `LinkRanker`,
`RelationRanker` and `PairRanker` ranks and metrics, `topk` over the (s, r) of every test edge, `topk_relations`
over the (s, t) of every test edge and `topk_pairs` of every relation, each with and without an `EdgeFilter`.
Inputs: the pose-0 and pose-2 splits of `rank_bench.py` and one integer fixture of each ranking test file.  Floats
are compared bit for bit (NaN payloads and signed zeros included), integers exactly.  The dump also times the
construction of `EdgeFilter` and `LinkRanker` at the pose shapes (host clock around the constructor, after a device
synchronise; median of 5 after one warm-up).  Writes OUTDIR/rank_parity.txt and OUTDIR/rank_build_ms.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
K = 10


def _fixtures(np, torch, dev):
    """(name, z, w, test, filter lists) on the device."""
    sys.path.insert(1, os.path.join(ROOT, "tests"))
    sys.path.insert(1, HERE)
    import rank_bench
    import synthdata
    import test_gpu_pair_ranking as tpr
    import test_gpu_ranking as tr
    import test_gpu_relation_ranking as trr

    def lst(a):
        return (torch.as_tensor(np.asarray(a[0]), dtype=torch.int64, device=dev),
                torch.as_tensor(np.asarray(a[1]), dtype=torch.int64, device=dev))

    def f32(a):
        return torch.as_tensor(a, dtype=torch.float32, device=dev)

    out = []
    for name, g in (("pose0", synthdata.pose_graph()), ("pose2", synthdata.pose2_graph())):
        train, test, z, w = rank_bench._inputs(g, dev)
        out.append((name, z, w, test, [train, test]))
    z, w, test, lists = tr._integer_fixture(0)
    out.append(("int_ranking", f32(z), f32(w), lst(test), [lst(l) for l in lists]))
    z, w, test, lists = trr._integer_fixture(1, 30, 6, 200, 600)
    out.append(("int_relation_ranking", f32(z), f32(w), lst(test), [lst(l) for l in lists]))
    for name, (seed, n, d, r) in (("int_pair_ranking", (2, 50, 7, 3)), ("int_pair_ranker", (3, 70, 80, 4))):
        z, w, lists = tpr._integer_fixture(seed, n, d, r)
        out.append((name, f32(z), f32(w), lst(lists[0]), [lst(l) for l in lists]))
    return out


def dump(root, path):
    import numpy as np
    import torch
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    # imported before _fixtures: rank_bench puts this checkout first on sys.path
    assert os.path.dirname(os.path.dirname(os.path.abspath(gb.__file__))) == root, gb.__file__
    dev = torch.device("cuda:0")
    res, build_ms = {}, {}
    for name, z, w, test, lists in _fixtures(np, torch, dev):
        n, r = z.size(0), w.size(0)
        ei, et = test
        filt = gb.EdgeFilter(lists, n, r)
        hits = (1, 3, 10)
        for tag, f in (("raw", None), ("filtered", filt)):
            key = f"{name}/{tag}"
            for cls in (gb.LinkRanker, gb.RelationRanker, gb.PairRanker):
                ranker = cls(ei, et, n, r, filter=f)
                res[f"{key}/{cls.__name__}.ranks"] = ranker.ranks(z, w)
                res[f"{key}/{cls.__name__}.metrics"] = ranker.metrics(z, w, hits=hits)
                res[f"{key}/{cls.__name__}.n_groups"] = torch.tensor(ranker.n_groups)
            sig = name.startswith("int")
            res[f"{key}/topk"] = ranking.topk(z, w, ei[0], et, K, filter=f, sigmoid=sig)
            res[f"{key}/topk_relations"] = ranking.topk_relations(z, w, ei[0], ei[1], 2 * r if sig else K, filter=f,
                                                                  sigmoid=sig)
            res[f"{key}/topk_pairs"] = ranking.topk_pairs(z, w, torch.arange(r, device=dev), K, filter=f, sigmoid=sig)
        if name.startswith("pose"):
            def timed(fn):
                fn()
                ts = []
                for _ in range(5):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    ts.append((time.perf_counter() - t0) * 1e3)
                return round(float(np.median(ts)), 3)
            build_ms[name] = {"EdgeFilter_ms": timed(lambda: gb.EdgeFilter(lists, n, r)),
                              "LinkRanker_ms": timed(lambda: gb.LinkRanker(ei, et, n, r, filter=filt))}
    torch.cuda.synchronize()
    flat = {}
    for k, v in res.items():
        for i, t in enumerate(v if isinstance(v, tuple) else (v,)):
            flat[f"{k}[{i}]" if isinstance(v, tuple) else k] = t.cpu()
    torch.save({"outputs": flat, "build_ms": build_ms}, path)


def _bits(t):
    import torch
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int64) if t.dtype == torch.float64 else t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other")
    ap.add_argument("--out")
    ap.add_argument("--dump", nargs=2, metavar=("ROOT", "FILE"))
    args = ap.parse_args()
    if args.dump:
        root = os.path.abspath(args.dump[0])
        sys.path.insert(0, root)
        return dump(root, args.dump[1])
    import torch
    os.makedirs(args.out, exist_ok=True)
    files = {}
    for label, root in (("other", os.path.abspath(args.other)), ("this", ROOT)):
        files[label] = os.path.join(args.out, f"rank_parity_{label}.pt")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--dump", root, files[label]], check=True)
    a, b = (torch.load(files[k]) for k in ("other", "this"))
    lines, bad = [], 0
    assert sorted(a["outputs"]) == sorted(b["outputs"]), "the two checkouts computed different output sets"
    for k in sorted(a["outputs"]):
        x, y = a["outputs"][k], b["outputs"][k]
        same = x.dtype == y.dtype and x.shape == y.shape and torch.equal(_bits(x), _bits(y))
        nan = int(torch.isnan(x).sum()) if x.is_floating_point() else 0
        bad += not same
        lines.append(f"{'identical' if same else 'DIFFERENT'}  {k}  {tuple(x.shape)} {str(x.dtype)[6:]}"
                     + (f"  ({nan} NaN)" if nan else ""))
    lines.append(f"{len(a['outputs']) - bad} of {len(a['outputs'])} outputs bit-identical")
    with open(os.path.join(args.out, "rank_parity.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    with open(os.path.join(args.out, "rank_build_ms.json"), "w") as f:
        json.dump({"other": a["build_ms"], "this": b["build_ms"]}, f, indent=1)
    for p in files.values():
        os.remove(p)
    print(lines[-1])
    print(json.dumps({"build_ms_other": a["build_ms"], "build_ms_this": b["build_ms"]}))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
