#!/usr/bin/env python
"""Link-prediction experiment of the reference (``GripNet-pose.py``) on gripnet_b200.

    python examples/gripnet_pose.py EPOCHS datasets/pose/pose-0.pt [--out out/pose-0]
    python examples/gripnet_pose.py EPOCHS --synthetic            # pose-0-shaped synthetic supergraph
    python examples/gripnet_pose.py EPOCHS --synthetic --rank     # + filtered test MRR / Hits@k every epoch
    python examples/gripnet_pose.py EPOCHS --synthetic --novel 100   # + the 100 best new drug pairs per side effect

Same model (``GripNet-pose.py:86-99``), optimiser (Adam, lr 0.01, ``:104``), per-epoch negative sampling
(``:131``), loss (``:140-142``) and per-relation AUPRC / AUROC / AP@all records (``:148-164``, ``:174-199``) —
but an epoch is ONE CUDA-graph replay (``training.PoseTrainer``) and the evaluation never leaves the device.
Writes ``<out>-model.pt`` (``state_dict``, the reference's key names) and ``<out>-record.pt``; with ``--novel K``
also ``<out>-novel.pt``.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("epochs", type=int)
    ap.add_argument("dataset", nargs="?")
    ap.add_argument("--synthetic", action="store_true")
    ap.add_argument("--out", default="out/pose")
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--seed", type=int, default=1111)
    ap.add_argument("--rank", action="store_true",
                    help="also print the filtered test MRR and Hits@10 (all drugs as candidate tails, train + test "
                         "positives filtered), the filtered test relation MRR and Hits@10 (all side effects as "
                         "candidates of each drug pair) and the filtered test pair MRR and Hits@100 (all drug pairs "
                         "as candidates of each side effect), macro-averaged over relations")
    ap.add_argument("--novel", type=int, metavar="K", default=0,
                    help="after training, write <out>-novel.pt: the K (<= 256) most likely drug pairs {s, t} of every "
                         "side effect that are not train or test positives in either direction (scores after the "
                         "sigmoid, src < dst, each [R, K])")
    args = ap.parse_args()

    from gripnet_b200 import data as gd, metrics, ranking, utils
    from gripnet_b200.pipelines import PoseModel, to_device
    from gripnet_b200.training import PoseTrainer
    dev = torch.device("cuda:0")
    torch.manual_seed(args.seed)
    if args.synthetic or args.dataset is None:
        from gripnet_b200.synthetic import pose_graph
        train = pose_graph(seed=args.seed)
        test = dict(train)                                  # synthetic: evaluate on the training relations
    else:
        ds = gd.load(args.dataset)
        train, test = gd.pose_inputs(ds, "train"), gd.pose_inputs(ds, "test")
    train, test = to_device(train, dev), to_device(test, dev)
    model = PoseModel(train["n_g"], train["n_d"], train["n_rel"]).to(dev)
    print(model)

    trainer = PoseTrainer(model, train, lr=args.lr, seed=args.seed, with_metrics=True)
    # fixed typed negatives for the test relations (GripNet-pose.py:169-171)
    test_neg = utils.typed_negative_sampling(test["dd_edge_index"], test["n_d"], test["dd_range_list"])
    n_rel = train["n_rel"]
    train_rec = torch.empty(args.epochs, 3, n_rel, dtype=torch.float64, device=dev)
    test_rec = torch.empty(args.epochs, 3, n_rel, dtype=torch.float64, device=dev)
    losses = torch.empty(args.epochs, device=dev)
    ranker = None
    if args.rank:                                           # built once; one filtered ranking pass per epoch
        pos = [(train["dd_edge_index"], train["dd_edge_type"]), (test["dd_edge_index"], test["dd_edge_type"])]
        filt = ranking.EdgeFilter(pos, test["n_d"], n_rel)
        ranker = ranking.LinkRanker(test["dd_edge_index"], test["dd_edge_type"], test["n_d"], n_rel, filter=filt)
        rel_ranker = ranking.RelationRanker(test["dd_edge_index"], test["dd_edge_type"], test["n_d"], n_rel,
                                            filter=filt)
        rank_rec = torch.empty(args.epochs, 2, n_rel, dtype=torch.float64, device=dev)
        rel_rank_rec = torch.empty(args.epochs, 2, n_rel, dtype=torch.float64, device=dev)
        # about 2 * 10^5 candidate pairs per side effect at pose shapes: Hits@100
        pair_ranker = ranking.PairRanker(test["dd_edge_index"], test["dd_edge_type"], test["n_d"], n_rel, filter=filt)
        pair_rank_rec = torch.empty(args.epochs, 2, n_rel, dtype=torch.float64, device=dev)
    for epoch in range(args.epochs):
        t0 = time.time()
        losses[epoch] = trainer.train_epoch().detach()
        train_rec[epoch] = trainer.record
        with torch.no_grad():                               # test(z), GripNet-pose.py:174-199
            z = trainer.z.detach()
            pos = model.dmt(z, test["dd_edge_index"], test["dd_edge_type"])
            neg = model.dmt(z, test_neg, test["dd_edge_type"])
            metrics.lp_metrics(pos, neg, test["dd_range_list"], out=test_rec[epoch])
            if ranker is not None:
                ranker.metrics(z, model.dmt.weight, hits=(10,), out=rank_rec[epoch])
                rel_ranker.metrics(z, model.dmt.weight, hits=(10,), out=rel_rank_rec[epoch])
                pair_ranker.metrics(z, model.dmt.weight, hits=(100,), out=pair_rank_rec[epoch])
        tr, te = train_rec[epoch].nanmean(dim=1).tolist(), test_rec[epoch].nanmean(dim=1).tolist()   # one sync per epoch
        line = "{:3d}   loss:{:0.4f}   train auprc:{:0.4f} auroc:{:0.4f} ap:{:0.4f}   test auprc:{:0.4f} auroc:{:0.4f} " \
               "ap:{:0.4f}".format(epoch, float(losses[epoch].detach()), *tr, *te)
        if ranker is not None:
            line += "   test mrr:{:0.4f} hits@10:{:0.4f}".format(*rank_rec[epoch].nanmean(dim=1).tolist())
            line += "   test relation mrr:{:0.4f} hits@10:{:0.4f}".format(*rel_rank_rec[epoch].nanmean(dim=1).tolist())
            line += "   test pair mrr:{:0.4f} hits@100:{:0.4f}".format(*pair_rank_rec[epoch].nanmean(dim=1).tolist())
        print(line + "   time:{:0.3f}".format(time.time() - t0))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    torch.save({k: v.cpu() for k, v in model.state_dict().items()}, args.out + "-model.pt")
    rec = {"train_record": train_rec.cpu(), "test_record": test_rec.cpu(), "loss": losses.cpu()}
    if ranker is not None:
        rec["test_rank_record"] = rank_rec.cpu()             # [epochs, 2 (mrr, hits@10), R]
        rec["test_relation_rank_record"] = rel_rank_rec.cpu()   # [epochs, 2 (mrr, hits@10), R]
        rec["test_pair_rank_record"] = pair_rank_rec.cpu()   # [epochs, 2 (mrr, hits@100), R]
    torch.save(rec, args.out + "-record.pt")
    if args.novel:
        pos = [(train["dd_edge_index"], train["dd_edge_type"]), (test["dd_edge_index"], test["dd_edge_type"])]
        filt = ranking.EdgeFilter(pos, test["n_d"], n_rel)
        with torch.no_grad():
            scores, src, dst = model.dmt.topk_pairs(trainer.z.detach(), torch.arange(n_rel, device=dev), args.novel,
                                                    filter=filt)
        torch.save({"scores": scores.cpu(), "src": src.cpu(), "dst": dst.cpu()}, args.out + "-novel.pt")
        print("side effect 0, best new pairs: " + ", ".join(
            "({}, {}) {:0.4f}".format(a, b, v) for a, b, v in zip(src[0, :5].tolist(), dst[0, :5].tolist(),
                                                                  scores[0, :5].tolist())))


if __name__ == "__main__":
    main()
