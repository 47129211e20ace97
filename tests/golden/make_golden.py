"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container only (needs the read-only checkout at
``/root/reference``):

    python tests/golden/make_golden.py

The reference's ``gripnet/layers.py`` / ``decoder.py`` are executed from where
they lie through ``oracle/ref_loader.py`` (PyG-1.x symbols supplied by
``oracle/pyg_shim.py``); inputs come from ``oracle/synth.py``.  Each fixture is
a flat ``.npz``: ``in.*`` inputs, ``p.*`` parameters (reference ``state_dict``
names with a model prefix), ``out.*`` forward results, ``grad.*`` parameter
gradients of the scalar loss.  Tests never need the reference at run time.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_loader, synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
L, D, U = ref_loader.load()


def _load(module, p, prefix):
    sd = {k[len(prefix):]: v.clone() for k, v in p.items() if k.startswith(prefix)}
    missing = set(module.state_dict().keys()) ^ set(sd.keys())
    assert not missing, (prefix, missing)
    module.load_state_dict(sd)
    return module


def _save(name, inputs, params, outs, grads):
    flat = {}
    for k, v in inputs.items():
        if v is not None:
            flat["in." + k] = np.asarray(v.numpy() if torch.is_tensor(v) else v)
    for k, v in params.items():
        flat["p." + k] = v.detach().numpy()
    for k, v in outs.items():
        flat["out." + k] = v.detach().numpy()
    for k, v in grads.items():
        flat["grad." + k] = v.detach().numpy()
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **flat)
    print(f"{name}: {len(flat)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")


def _grads(named_modules):
    g = {}
    for prefix, m in named_modules:
        if isinstance(m, torch.nn.Parameter):
            g[prefix.rstrip(".")] = m.grad
            continue
        for k, v in m.named_parameters():
            if v.grad is not None:
                g[prefix + k] = v.grad
    return g


# ---------------------------------------------------------------- a1: norm KATs
def norm_cases():
    rs = np.random.RandomState(5)
    cases = {"kat6": (np.array([[0, 1, 1, 2, 2, 0], [1, 1, 2, 0, 0, 3]]), 4, None, False)}
    ei = rs.randint(0, 50, size=(2, 400))
    ei[:, ::37] = ei[0, ::37]                      # a few self loops, some repeated on one node
    ei[:, 5] = ei[:, 42] = 7
    cases["loops_w"] = (ei, 50, rs.uniform(0.5, 1.5, 400).astype(np.float32), False)
    cases["loops_improved"] = (ei, 50, None, True)
    cases["isolated"] = (rs.randint(0, 20, size=(2, 60)), 64, None, False)   # nodes 20..63 isolated
    cases["empty"] = (np.zeros((2, 0), dtype=np.int64), 5, None, False)
    flat = {}
    for name, (ei, n, w, imp) in cases.items():
        ei_t = torch.from_numpy(np.asarray(ei, dtype=np.int64))
        w_t = None if w is None else torch.from_numpy(w)
        ei2, nrm = L.myGCN.norm(ei_t, n, w_t, imp, torch.float32)
        flat[f"{name}.edge_index"] = ei_t.numpy()
        flat[f"{name}.num_nodes"] = np.int64(n)
        flat[f"{name}.improved"] = np.bool_(imp)
        if w is not None:
            flat[f"{name}.edge_weight"] = w
        flat[f"{name}.out_edge_index"] = ei2.numpy()
        flat[f"{name}.out_norm"] = nrm.numpy()
    np.savez_compressed(os.path.join(HERE, "gcn_norm.npz"), **flat)
    print("gcn_norm:", len(cases), "cases")


# ---------------------------------------------------------------- full models
def pose_case(name, g, p, gg=(32, 16, 16), gd=(16, 32), dd_out=32):
    m_gg = _load(L.homoGraph(list(gg), start_graph=True, in_dim=g["n_g"]), p, "gg.")
    m_gd = _load(L.interGraph(sum(gg), gd[0], g["n_d"], target_feat_dim=gd[1]), p, "gd.")
    m_dd = _load(L.homoGraph([sum(gd), dd_out], multi_relational=True, n_rela=g["n_rel"]), p, "dd.")
    m_dmt = _load(D.multiRelaInnerProductDecoder(sum(gd) + dd_out, g["n_rel"]), p, "dmt.")
    ew = g.get("gg_edge_weight")
    if ew is None:
        ew = torch.ones(g["gg_edge_index"].shape[1])          # GripNet-pose.py:52
    z_gg = m_gg(None, g["gg_edge_index"], edge_weight=ew, if_catout=True)
    z_gd = m_gd(z_gg, g["gd_edge_index"], mod="cat", if_relu=True)
    z = m_dd(z_gd, g["dd_edge_index"], edge_type=g["dd_edge_type"], range_list=g["dd_range_list"], if_catout=True)
    pos = m_dmt(z, g["dd_edge_index"], g["dd_edge_type"])
    neg = m_dmt(z, g["neg_edge_index"], g["dd_edge_type"])
    loss = -torch.log(pos + U.EPS).mean() - torch.log(1 - neg + U.EPS).mean()   # GripNet-pose.py:140-142
    loss.backward()
    grads = _grads([("gg.", m_gg), ("gd.", m_gd), ("dd.", m_dd), ("dmt.", m_dmt)])
    _save(name, {k: v for k, v in g.items()}, p,
          {"z_gg": z_gg, "z_gd": z_gd, "z": z, "pos": pos, "neg": neg, "loss": loss}, grads)


def aminer_case(name, g, p, pp=(128, 64, 64), pa=(64, 64), aa_hid=(128, 32)):
    aa = [sum(pa)] + list(aa_hid)
    m_pp = _load(L.homoGraph(list(pp), start_graph=True, in_dim=g["n_p"]), p, "pp.")
    m_pa = _load(L.interGraph(sum(pp), pa[0], g["n_a"], target_feat_dim=pa[1]), p, "pa.")
    m_aa = _load(L.homoGraph(aa), p, "aa.")
    m_dec = _load(D.multiClassInnerProductDecoder(sum(aa), g["n_class"]), p, "mcip.")
    z_pp = m_pp(None, g["pp_edge_index"], if_catout=True)
    z_pa = m_pa(z_pp, g["pa_edge_index"], if_relu=True, mod="cat")
    z = m_aa(z_pa, g["aa_edge_index"], if_catout=True)
    score = m_dec(z, g["train_node_idx"])
    loss = -torch.log(score[range(score.shape[0]), g["train_node_class"]] + U.EPS).mean()  # aminer.py:133
    loss.backward()
    grads = _grads([("pp.", m_pp), ("pa.", m_pa), ("aa.", m_aa), ("mcip.", m_dec)])
    _save(name, g, p, {"z_pp": z_pp, "z_pa": z_pa, "z": z, "score": score, "loss": loss}, grads)


def freebase_d_case(name, g, p, pp=(256, 128, 128), pa=(128, 128), aa_out=32):
    m_pp = _load(L.homoGraph(list(pp), start_graph=True, in_dim=g["n_p"]), p, "pp.")
    m_pa = _load(L.interGraph(sum(pp), pa[0], g["n_a"], target_feat_dim=pa[1], if_one_external=False), p, "pa.")
    m_qq = _load(L.homoGraph(list(pp), start_graph=True, in_dim=g["n_q"]), p, "qq.")
    m_qa = _load(L.interGraph(sum(pp), pa[0], g["n_a"], target_feat_dim=pa[1], if_one_external=False), p, "qa.")
    emb = torch.nn.Parameter(p["aa_embeddings"].clone())
    m_aa = _load(L.homoGraph([pa[1], aa_out]), p, "aa.")
    m_dec = _load(D.multiClassInnerProductDecoder(aa_out, g["n_class"]), p, "mcip.")
    z = m_pa(m_pp(None, g["pp_edge_index"], if_catout=True), g["pa_edge_index"], mod="add", if_relu=True)
    z1 = m_qa(m_qq(None, g["qq_edge_index"], if_catout=True), g["qa_edge_index"], mod="add", if_relu=True)
    zz = m_aa((z + z1 + emb) / 3, g["aa_edge_index"])          # freebase-d.py:160-164
    score = m_dec(zz, g["train_node_idx"])
    loss = -torch.log(score[range(score.shape[0]), g["train_node_class"]] + U.EPS).mean()
    loss.backward()
    grads = _grads([("pp.", m_pp), ("pa.", m_pa), ("qq.", m_qq), ("qa.", m_qa), ("aa_embeddings", emb),
                    ("aa.", m_aa), ("mcip.", m_dec)])
    _save(name, g, p, {"z_pa": z, "z_qa": z1, "z": zz, "score": score, "loss": loss}, grads)


# ---------------------------------------------------------------- module variants
def variants():
    gen = torch.Generator().manual_seed(3)
    rs = np.random.RandomState(3)
    flat = {}

    def put(prefix, **kw):
        for k, v in kw.items():
            if v is not None:
                flat[f"{prefix}.{k}"] = v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)

    # interGraph tails: mod="add" with equal widths, with target_feat_down, and no relu
    n_s, n_t = 60, 25
    x = torch.randn(n_s, 24, generator=gen)
    ei = torch.from_numpy(np.stack([rs.randint(0, n_s, 150), rs.randint(0, n_t, 150)]).astype(np.int64))
    ew = torch.from_numpy(rs.uniform(0.5, 1.5, 150).astype(np.float32))
    for tag, tdim, tfd, mod, relu, w in [("add_eq", 16, 16, "add", True, None), ("add_down", 16, 12, "add", True, ew),
                                         ("cat_norelu", 16, 8, "cat", False, None)]:
        p = {}
        synth.inter_params(gen, 24, tdim, n_t, tfd, "", p)
        p["conv.bias"] = torch.randn(tdim, generator=gen) * 0.1
        m = _load(L.interGraph(24, tdim, n_t, target_feat_dim=tfd), p, "")
        xin = x.clone().requires_grad_(True)
        out = m(xin, ei, edge_weight=w, if_relu=relu, mod=mod)
        (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
        put("inter_" + tag, x=x, edge_index=ei, edge_weight=w, out=out, grad_x=xin.grad,
            **{"p." + k: v for k, v in p.items()}, **{"grad." + k: v.grad for k, v in m.named_parameters()})

    # homoGraph GCN without catout / not start_graph, weighted
    n = 80
    ei = torch.from_numpy(rs.randint(0, n, (2, 500)).astype(np.int64))
    ew = torch.from_numpy(rs.uniform(0.5, 1.5, 500).astype(np.float32))
    p = {}
    synth.homo_params(gen, [20, 16, 8], "", p)
    for k in list(p):
        if k.endswith("bias"):
            p[k] = torch.randn(p[k].shape, generator=gen) * 0.1
    m = _load(L.homoGraph([20, 16, 8]), p, "")
    x = torch.randn(n, 20, generator=gen)
    xin = x.clone().requires_grad_(True)
    out = m(xin, ei, edge_weight=ew, if_catout=False)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("homo_nocat", x=x, edge_index=ei, edge_weight=ew, out=out, grad_x=xin.grad,
        **{"p." + k: v for k, v in p.items()}, **{"grad." + k: v.grad for k, v in m.named_parameters()})

    # two-layer RGCN stack (after_relu init on layer 1), odd widths, one empty relation
    n, n_rel = 50, 4
    sizes = [70, 0, 45, 90]
    chunks, ranges, s = [], [], 0
    for k in sizes:
        chunks.append(rs.randint(0, n, (2, k)))
        ranges.append((s, s + k))
        s += k
    ei = torch.from_numpy(np.concatenate(chunks, axis=1).astype(np.int64))
    et = torch.from_numpy(np.concatenate([np.full(k, r) for r, k in enumerate(sizes)]).astype(np.int64))
    rl = torch.tensor(ranges, dtype=torch.int64)
    p = {}
    synth.homo_params(gen, [12, 20, 8], "", p, n_rel=n_rel, n_base=6)
    m = _load(L.homoGraph([12, 20, 8], multi_relational=True, n_rela=n_rel, n_base=6), p, "")
    x = torch.randn(n, 12, generator=gen)
    xin = x.clone().requires_grad_(True)
    out = m(xin, ei, edge_type=et, range_list=rl, if_catout=True)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("rgcn2", x=x, edge_index=ei, edge_type=et, range_list=rl, out=out, grad_x=xin.grad,
        **{"p." + k: v for k, v in p.items()}, **{"grad." + k: v.grad for k, v in m.named_parameters()})

    # standalone myRGCN with bias
    conv = L.myRGCN(12, 10, n_rel, 6, after_relu=False, bias=True)
    conv.bias.data.normal_(generator=gen)
    xin = x.clone().requires_grad_(True)
    out = conv(xin, ei, et, rl)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("rgcn_bias", x=x, edge_index=ei, edge_type=et, range_list=rl, out=out, grad_x=xin.grad,
        **{"p." + k: v for k, v in conv.state_dict().items()},
        **{"grad." + k: v.grad for k, v in conv.named_parameters()})

    # standalone myGCN improved, not cached, no bias
    n = 40
    ei = torch.from_numpy(rs.randint(0, n, (2, 200)).astype(np.int64))
    conv = L.myGCN(10, 6, improved=True, cached=False, bias=False)
    x = torch.randn(n, 10, generator=gen)
    xin = x.clone().requires_grad_(True)
    out = conv(xin, ei)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("gcn_improved", x=x, edge_index=ei, out=out, grad_x=xin.grad,
        **{"p." + k: v for k, v in conv.state_dict().items()},
        **{"grad." + k: v.grad for k, v in conv.named_parameters()})

    # decoders without the final non-linearity
    z = torch.randn(30, 20, generator=gen)
    ei = torch.from_numpy(rs.randint(0, 30, (2, 100)).astype(np.int64))
    et = torch.from_numpy(rs.randint(0, 3, 100).astype(np.int64))
    dec = D.multiRelaInnerProductDecoder(20, 3)
    zin = z.clone().requires_grad_(True)
    out = dec(zin, ei, et, sigmoid=False)
    (out * torch.linspace(-1, 1, out.numel())).sum().backward()
    put("dmt_raw", z=z, edge_index=ei, edge_type=et, out=out, grad_z=zin.grad,
        **{"p.weight": dec.weight, "grad.weight": dec.weight.grad})
    dec = D.multiClassInnerProductDecoder(20, 7)
    nodes = torch.tensor([3, 3, 9, 0, 29, 9, 17], dtype=torch.int64)      # duplicates on purpose
    zin = z.clone().requires_grad_(True)
    out = dec(zin, nodes, softmax=False)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("mcip_raw", z=z, node_list=nodes, out=out, grad_z=zin.grad,
        **{"p.weight": dec.weight, "grad.weight": dec.weight.grad})
    zin = z.clone().requires_grad_(True)
    dec.weight.grad = None
    out = dec(zin, nodes, softmax=True)
    (out * torch.linspace(-1, 1, out.numel()).view_as(out)).sum().backward()
    put("mcip_softmax", z=z, node_list=nodes, out=out, grad_z=zin.grad,
        **{"p.weight": dec.weight, "grad.weight": dec.weight.grad})

    np.savez_compressed(os.path.join(HERE, "variants.npz"), **flat)
    print("variants:", len(flat), "arrays")


if __name__ == "__main__":
    torch.set_num_threads(1)          # sequential index_add order -> reproducible fixtures
    torch.manual_seed(20261017)       # default initialisers of the reference modules draw from the global RNG
    # tests/test_init_distributions.py replays every module construction below, in this order, with this seed
    norm_cases()
    g = synth.pose_small()
    pose_case("pose_small", g, synth.pose_params(g))
    g = synth.pose_small(seed=2, weighted=True)
    pose_case("pose_small_weighted", g, synth.pose_params(g, seed=8))
    g = synth.aminer_small()
    aminer_case("aminer_small", g, synth.aminer_params(g, pp=(32, 16, 16), pa=(16, 16), aa_hid=(32, 8)),
                pp=(32, 16, 16), pa=(16, 16), aa_hid=(32, 8))
    g = synth.freebase_d_small()
    freebase_d_case("freebase_d_small", g, synth.freebase_d_params(g, pp=(32, 16, 16), pa=(16, 16), aa_out=8),
                    pp=(32, 16, 16), pa=(16, 16), aa_out=8)
    variants()
