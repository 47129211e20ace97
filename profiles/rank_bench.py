#!/usr/bin/env python
"""Filtered ranking (LinkRanker.metrics) and top-k (k = 10) over every (s, r) query group of a 90/10 test split,
filtered relation ranking (RelationRanker.metrics) and top-k relations (k = 10) over every directed (s, t) pair of
the same split, and top-k new pairs (topk_pairs, k = 10 and 100) of every relation with train + test filtered, at the
pose-0 and pose-2 shapes, against torch-on-GPU restatements of the same computations timed in the same run.

    python profiles/rank_bench.py --out DIR [--calls 20] [--workloads pose0,pose2] [--queries tail,relation,pair]

Warm-up, then the median of `--calls` calls, each bracketed by CUDA events (warm L2: the score chunks are meant to
stay there).  Writes DIR/rank_bench.json with the device name and power limit beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

D = 80
K = 10
HITS = (1, 3, 10)


def _median_ms(fn, calls, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def _split(g, seed=7):
    ei, et = g["dd_edge_index"], g["dd_edge_type"]
    perm = torch.from_numpy(np.random.RandomState(seed).permutation(ei.size(1)))
    cut = int(0.9 * perm.numel())
    tr, te = perm[:cut].sort().values, perm[cut:].sort().values
    return (ei[:, tr], et[tr]), (ei[:, te], et[te])


class TorchRestatement:
    """The same computation in eager torch: dense filter mask per query group, S = (z[s] * w[r]) z^T in fp32,
    per-edge OGB counts, per-relation means, masked torch.topk."""

    def __init__(self, group_row, test, lists, n, r):
        dev = group_row.device
        self.n, self.r = n, r
        self.s, self.rel = group_row // r, group_row % r
        lut = torch.full((n * r,), -1, dtype=torch.int64, device=dev)
        lut[group_row] = torch.arange(group_row.numel(), device=dev)
        self.mask = torch.zeros((group_row.numel(), n), dtype=torch.bool, device=dev)
        for ei, et in lists:
            g = lut[ei[0] * r + et]
            keep = g >= 0
            self.mask[g[keep], ei[1][keep]] = True
        ei, et = test
        self.eg = lut[ei[0] * r + et]
        self.et, self.tt = et, ei[1]
        self.cnt = torch.bincount(et, minlength=r).double()

    def scores(self, z, w):
        return (z[self.s] * w[self.rel]) @ z.t()

    def ranks(self, z, w, chunk=1 << 17):
        S = self.scores(z, w)
        out = torch.empty(self.eg.numel(), dtype=torch.float32, device=z.device)
        cols = torch.arange(self.n, device=z.device)
        for a in range(0, self.eg.numel(), chunk):
            g, t = self.eg[a:a + chunk], self.tt[a:a + chunk]
            row = S[g]
            st = row.gather(1, t[:, None])
            neg = ~self.mask[g] & (cols[None, :] != t[:, None])
            opt = ((row > st) & neg).sum(1)
            pess = ((row >= st) & neg).sum(1)
            out[a:a + chunk] = 1.0 + (opt + pess).float() * 0.5
        return out

    def metrics(self, z, w):
        rk = self.ranks(z, w).double()
        rows = [torch.zeros(self.r, dtype=torch.float64, device=z.device).index_add_(0, self.et, 1.0 / rk)]
        for k in HITS:
            rows.append(torch.zeros(self.r, dtype=torch.float64, device=z.device).index_add_(0, self.et,
                                                                                          (rk <= k).double()))
        return torch.stack(rows) / self.cnt

    def topk(self, z, w):
        S = self.scores(z, w).masked_fill_(self.mask, float("-inf"))
        return torch.topk(S, K, dim=1)


class TorchRelationRestatement:
    """Relation queries in eager torch: dense filter mask per pair, S = (z[s] * z[t]) W^T in fp32, per-triple OGB
    counts, per-relation means, masked torch.topk."""

    def __init__(self, pair_src, pair_dst, test, lists, n, r):
        dev = pair_src.device
        self.n, self.r = n, r
        self.s, self.t = pair_src, pair_dst
        keys = pair_src * n + pair_dst                                 # ascending: pairs are in (src, dst) order

        def group(ei):
            k = ei[0] * n + ei[1]
            g = torch.searchsorted(keys, k).clamp_max(keys.numel() - 1)
            return g, keys[g] == k

        self.mask = torch.zeros((keys.numel(), r), dtype=torch.bool, device=dev)
        for ei, et in lists:
            g, keep = group(ei)
            self.mask[g[keep], et[keep]] = True
        ei, et = test
        self.eg, _ = group(ei)
        self.et = et
        self.cnt = torch.bincount(et, minlength=r).double()

    def scores(self, z, w):
        return (z[self.s] * z[self.t]) @ w.t()

    def ranks(self, z, w, chunk=1 << 16):
        S = self.scores(z, w)
        out = torch.empty(self.eg.numel(), dtype=torch.float32, device=z.device)
        cols = torch.arange(self.r, device=z.device)
        for a in range(0, self.eg.numel(), chunk):
            g, r = self.eg[a:a + chunk], self.et[a:a + chunk]
            row = S[g]
            sr = row.gather(1, r[:, None])
            neg = ~self.mask[g] & (cols[None, :] != r[:, None])
            opt = ((row > sr) & neg).sum(1)
            pess = ((row >= sr) & neg).sum(1)
            out[a:a + chunk] = 1.0 + (opt + pess).float() * 0.5
        return out

    def metrics(self, z, w):
        rk = self.ranks(z, w).double()
        rows = [torch.zeros(self.r, dtype=torch.float64, device=z.device).index_add_(0, self.et, 1.0 / rk)]
        for k in HITS:
            rows.append(torch.zeros(self.r, dtype=torch.float64, device=z.device).index_add_(0, self.et,
                                                                                          (rk <= k).double()))
        return torch.stack(rows) / self.cnt

    def topk(self, z, w):
        S = self.scores(z, w).masked_fill_(self.mask, float("-inf"))
        return torch.topk(S, K, dim=1)


class TorchPairRestatement:
    """Pair queries in eager torch: relation chunks of batched S_r = (z * w_r) z^T in fp32, a dense upper-triangle and
    symmetric filter mask, a flatten and torch.topk (ties in torch.topk's own order)."""

    def __init__(self, lists, n, r, dev, chunk_bytes=256 << 20):
        self.n, self.r = n, r
        self.chunk = max(1, chunk_bytes // (4 * n * n))
        self.adm = torch.ones((r, n, n), dtype=torch.bool, device=dev).triu_(1)
        for ei, et in lists:
            self.adm[et, ei[0], ei[1]] = False
            self.adm[et, ei[1], ei[0]] = False

    def topk(self, z, w, k):
        n = self.n
        out_s = torch.empty((self.r, k), dtype=torch.float32, device=z.device)
        out_i = torch.empty((self.r, k), dtype=torch.int64, device=z.device)
        for a in range(0, self.r, self.chunk):
            b = min(self.r, a + self.chunk)
            S = torch.matmul(z[None] * w[a:b, None, :], z.t())
            S.masked_fill_(~self.adm[a:b], float("-inf"))
            out_s[a:b], out_i[a:b] = torch.topk(S.view(b - a, n * n), k, dim=1)
        return out_s, out_i // n, out_i % n


def _inputs(g, dev):
    train, test = _split(g)
    train = (train[0].to(dev), train[1].to(dev))
    test = (test[0].to(dev), test[1].to(dev))
    gen = torch.Generator(device="cpu").manual_seed(3)
    z = (torch.randn(g["n_d"], D, generator=gen) / D ** 0.5).to(dev)
    w = torch.randn(g["n_rel"], D, generator=gen).to(dev)
    return train, test, z, w


def run_relations(name, g, calls, dev):
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    train, test, z, w = _inputs(g, dev)
    n, r = g["n_d"], g["n_rel"]
    filt = gb.EdgeFilter([train, test], n, r)
    ranker = gb.RelationRanker(test[0], test[1], n, r, filter=filt)
    G, E = ranker.n_groups, test[0].size(1)
    ps, pd = ranker._q.src[:G].long(), ranker._q.dst[:G].long()
    ref = TorchRelationRestatement(ps, pd, test, [train, test], n, r)
    rec = torch.empty((1 + len(HITS), r), dtype=torch.float64, device=dev)

    t_metrics = _median_ms(lambda: ranker.metrics(z, w, hits=HITS, out=rec), calls)
    t_topk = _median_ms(lambda: ranking.topk_relations(z, w, ps, pd, K, filter=filt, sigmoid=False), calls)
    t_ref_metrics = _median_ms(lambda: ref.metrics(z, w), calls)
    t_ref_topk = _median_ms(lambda: ref.topk(z, w), calls)

    rk, rk_ref = ranker.ranks(z, w), ref.ranks(z, w)
    m, m_ref = ranker.metrics(z, w, hits=HITS), ref.metrics(z, w)
    s, ids = ranking.topk_relations(z, w, ps, pd, K, filter=filt, sigmoid=False)
    s_ref, _ = ref.topk(z, w)
    scale = ref.scores(z, w).abs().amax(1, keepdim=True)
    ok_ids = ids >= 0
    agree = {
        "ranks_equal_fraction": float((rk == rk_ref).double().mean()),
        "metrics_max_abs_diff": float((m - m_ref).abs().nan_to_num(0.0).max()),
        "topk_score_max_rel_diff": float(((s - s_ref).abs() / scale)[ok_ids].max()),
        "topk_padding_matches": bool(torch.equal(~ok_ids, torch.isinf(s_ref))),
        "topk_filtered_ids_returned": int((ref.mask.gather(1, ids.clamp_min(0)) & ok_ids).sum()),
    }
    ok = agree["ranks_equal_fraction"] > 0.999 and agree["metrics_max_abs_diff"] < 1e-3 and \
        agree["topk_score_max_rel_diff"] < 1e-5 and agree["topk_padding_matches"] and \
        agree["topk_filtered_ids_returned"] == 0
    lds = (r + 3) // 4 * 4
    flops = 2.0 * G * r * D
    s_bytes = 2.0 * G * lds * 4                                   # the score rows, written once and read once
    in_bytes = 4.0 * (n * D + r * D) + 4.0 * 2 * E + 4.0 * 4 * G + 4.0 * 2 * (train[0].size(1) + E)
    return {
        "workload": name, "query": "relation", "n": n, "R": r, "D": D, "test_edges": E, "pairs": G, "k": K,
        "metrics_ms": round(t_metrics, 4), "topk_ms": round(t_topk, 4),
        "torch_metrics_ms": round(t_ref_metrics, 4), "torch_topk_ms": round(t_ref_topk, 4),
        "product_flop": flops, "score_bytes": s_bytes, "input_bytes": in_bytes,
        "metrics_product_tflops": round(flops / (t_metrics * 1e-3) / 1e12, 3),
        "agreement": agree, "agree": ok,
    }


def run_pairs(name, g, calls, dev):
    from gripnet_b200 import ranking
    train, test, z, w = _inputs(g, dev)
    n, r = g["n_d"], g["n_rel"]
    import gripnet_b200 as gb
    filt = gb.EdgeFilter([train, test], n, r)
    rel = torch.arange(r, device=dev)
    ref = TorchPairRestatement([train, test], n, r, dev)
    flops = 2.0 * D * r * n * (n - 1) / 2
    res = []
    for k in (10, 100):
        t_fused = _median_ms(lambda: ranking.topk_pairs(z, w, rel, k, filter=filt, sigmoid=False), calls)
        t_ref = _median_ms(lambda: ref.topk(z, w, k), calls)
        s, a, b = ranking.topk_pairs(z, w, rel, k, filter=filt, sigmoid=False)
        s_ref, a_ref, b_ref = ref.topk(z, w, k)
        scale = torch.stack([(z * w[i]) @ z.t() for i in range(r)]).abs().amax((1, 2))[:, None]
        agree = {
            "pair_ids_equal_fraction": float(((a == a_ref) & (b == b_ref)).double().mean()),
            "score_max_rel_diff": float(((s - s_ref).abs() / scale).max()),
            "filtered_or_ordered_pairs_returned": int((~ref.adm[rel[:, None], a, b]).sum()),
        }
        ok = agree["score_max_rel_diff"] < 1e-5 and agree["filtered_or_ordered_pairs_returned"] == 0 and \
            agree["pair_ids_equal_fraction"] > 0.95
        res.append({
            "workload": name, "query": "pair", "n": n, "R": r, "D": D, "k": k, "queries": r,
            "topk_pairs_ms": round(t_fused, 4), "torch_topk_pairs_ms": round(t_ref, 4),
            "pair_flop": flops, "topk_pairs_tflops": round(flops / (t_fused * 1e-3) / 1e12, 3),
            "torch_tflops": round(flops / (t_ref * 1e-3) / 1e12, 3),
            "agreement": agree, "agree": ok,
        })
    return res


def run(name, g, calls, dev):
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    train, test, z, w = _inputs(g, dev)
    n, r = g["n_d"], g["n_rel"]
    filt = gb.EdgeFilter([train, test], n, r)
    ranker = gb.LinkRanker(test[0], test[1], n, r, filter=filt)
    grp = ranker._q.group_row[: ranker.n_groups].long()
    qn, qr = grp // r, grp % r
    ref = TorchRestatement(grp, test, [train, test], n, r)
    G, E = ranker.n_groups, test[0].size(1)
    rec = torch.empty((1 + len(HITS), r), dtype=torch.float64, device=dev)

    t_metrics = _median_ms(lambda: ranker.metrics(z, w, hits=HITS, out=rec), calls)
    t_topk = _median_ms(lambda: ranking.topk(z, w, qn, qr, K, filter=filt, sigmoid=False), calls)
    t_ref_metrics = _median_ms(lambda: ref.metrics(z, w), calls)
    t_ref_topk = _median_ms(lambda: ref.topk(z, w), calls)

    # agreement (fp32 scores in both: rank differences only where candidates tie the target within rounding)
    rk, rk_ref = ranker.ranks(z, w), ref.ranks(z, w)
    m, m_ref = ranker.metrics(z, w, hits=HITS), ref.metrics(z, w)
    s, ids = ranking.topk(z, w, qn, qr, K, filter=filt, sigmoid=False)
    s_ref, _ = ref.topk(z, w)
    scale = ref.scores(z, w).abs().amax(1, keepdim=True)
    agree = {
        "ranks_equal_fraction": float((rk == rk_ref).double().mean()),
        "metrics_max_abs_diff": float((m - m_ref).abs().max()),
        "topk_score_max_rel_diff": float(((s - s_ref).abs() / scale).max()),
        "topk_filtered_ids_returned": int(ref.mask.gather(1, ids.clamp_min(0)).sum()),
    }
    ok = agree["ranks_equal_fraction"] > 0.999 and agree["metrics_max_abs_diff"] < 1e-3 and \
        agree["topk_score_max_rel_diff"] < 1e-5 and agree["topk_filtered_ids_returned"] == 0
    lds = (n + 3) // 4 * 4
    flops = 2.0 * G * n * D
    s_bytes = 2.0 * G * lds * 4                                   # the score rows, written once and read once
    in_bytes = 4.0 * (n * D + r * D) + 4.0 * 3 * E + 4.0 * 2 * (train[0].size(1) + E)
    res = {
        "workload": name, "query": "tail", "n": n, "R": r, "D": D, "test_edges": E, "groups": G, "k": K,
        "metrics_ms": round(t_metrics, 4), "topk_ms": round(t_topk, 4),
        "torch_metrics_ms": round(t_ref_metrics, 4), "torch_topk_ms": round(t_ref_topk, 4),
        "product_flop": flops, "score_bytes": s_bytes, "input_bytes": in_bytes,
        "metrics_product_tflops": round(flops / (t_metrics * 1e-3) / 1e12, 3),
        "agreement": agree, "agree": ok,
    }
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--workloads", default="pose0,pose2")
    ap.add_argument("--queries", default="tail,relation")
    args = ap.parse_args()
    import synthdata
    assert torch.cuda.is_available(), "rank_bench needs a CUDA device"
    dev = torch.device("cuda:0")
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover
        smi = f"unavailable ({e})"
    out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": smi, "results": []}
    graphs = {"pose0": synthdata.pose_graph, "pose2": synthdata.pose2_graph}
    runs = {"tail": run, "relation": run_relations, "pair": run_pairs}
    for name in args.workloads.split(","):
        g = graphs[name]()
        for query in args.queries.split(","):
            res = runs[query](name, g, args.calls, dev)
            for one in res if isinstance(res, list) else [res]:
                print(json.dumps(one), flush=True)
                out["results"].append(one)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rank_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"device": out["device"], "smi": smi}))
    if not all(r["agree"] for r in out["results"]):
        sys.exit("kernels and torch restatement disagree")


if __name__ == "__main__":
    main()
