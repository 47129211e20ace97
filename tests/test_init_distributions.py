"""SURVEY.md §8 row a10: every parameter of the drop-in modules is drawn from the reference's initial
distribution — checked statistically (moments / support against the formula the cited reference line implies) and
bit for bit against parameters drawn by the unmodified reference's own initialisers, stored in
``tests/golden/variants.npz``.  CPU only: constructors do not touch the device."""
import math
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _moments(t):
    t = t.detach().double().flatten()
    return float(t.mean()), float(t.std()), float(t.min()), float(t.max())


def _check_normal(t, std, what):
    m, s, _, _ = _moments(t)
    n = t.numel()
    assert abs(m) < 5 * std / math.sqrt(n), (what, "mean", m)
    assert abs(s / std - 1) < 5 / math.sqrt(2 * n) + 1e-3, (what, "std", s, std)
    # a normal sample this large exceeds 3 sigma somewhere: rules out a uniform of the same variance
    if n >= 20000:
        assert float(t.detach().abs().max()) > 3 * std, what


def _check_uniform(t, bound, what):
    m, s, lo, hi = _moments(t)
    n = t.numel()
    assert lo >= -bound and hi <= bound, (what, lo, hi, bound)
    assert abs(s / (bound / math.sqrt(3)) - 1) < 5 / math.sqrt(n) + 2e-3, (what, "std", s)
    assert abs(m) < 5 * bound / math.sqrt(3 * n), (what, "mean", m)
    assert hi > 0.98 * bound and lo < -0.98 * bound, (what, "support not reached")


def test_initial_distributions_follow_the_reference_formulas():
    import gripnet_b200 as gb
    torch.manual_seed(3)
    gcn = gb.myGCN(300, 200)
    _check_uniform(gcn.weight, math.sqrt(6.0 / 500), "myGCN.weight glorot (layers.py:42-44)")
    assert float(gcn.bias.abs().sum()) == 0.0                                   # layers.py:46-47
    for after_relu in (False, True):
        r = gb.myRGCN(120, 90, 40, 32, after_relu=after_relu)
        _check_normal(r.att, 1.0 / math.sqrt(32), "myRGCN.att (layers.py:152)")
        std = 2.0 / 120 if after_relu else 1.0 / math.sqrt(120)                 # layers.py:154-160
        _check_normal(r.basis, std, f"myRGCN.basis after_relu={after_relu}")
        _check_normal(r.root, std, f"myRGCN.root after_relu={after_relu}")
        assert r.bias is None                                                   # bias=False by default, :128
    h = gb.homoGraph([64, 32, 16], start_graph=True, in_dim=2000)
    _check_normal(h.embedding, 1.0, "homoGraph.embedding (layers.py:249-250)")
    hr = gb.homoGraph([48, 32, 32], multi_relational=True, n_rela=16, n_base=8)
    assert [c.after_relu for c in hr.conv_list] == [False, True]                # layers.py:232
    ig = gb.interGraph(64, 16, 3000, target_feat_dim=32)
    _check_normal(ig.target_feat, 1.0, "interGraph.target_feat (layers.py:359-360)")
    _check_normal(ig.target_feat_down, 1.0, "interGraph.target_feat_down (layers.py:348-353)")
    _check_uniform(ig.conv.weight, math.sqrt(6.0 / 80), "interGraph.conv.weight")
    dm = gb.multiRelaInnerProductDecoder(80, 400)
    _check_normal(dm.weight, 1.0 / math.sqrt(80), "DistMult weight (decoder.py:25-26)")
    mc = gb.multiClassInnerProductDecoder(288, 100)
    _check_uniform(mc.weight, math.sqrt(6.0 / 388), "multiclass weight glorot (decoder.py:47-49)")
    enc = gb.encoder.RGCN(500, 64, 32, 16, 8, 4)
    _check_normal(enc.embedding, 1.0, "encoder.RGCN.embedding (encoder.py:11-12)")
    assert (enc.rgcn1.after_relu, enc.rgcn2.after_relu) == (False, True)        # encoder.py:14-18


def _make_golden_constructions(gb):
    """Every module constructor ``tests/golden/make_golden.py`` calls, with the same arguments and in the same
    order, our classes in place of the reference's.  Returns the four modules whose fresh parameters the script
    stored (``variants.npz``: ``rgcn_bias``, ``gcn_improved``, ``dmt_raw``, ``mcip_raw``)."""
    from oracle import synth
    for g in (synth.pose_small(), synth.pose_small(seed=2, weighted=True)):                        # pose_case
        gb.homoGraph([32, 16, 16], start_graph=True, in_dim=g["n_g"])
        gb.interGraph(64, 16, g["n_d"], target_feat_dim=32)
        gb.homoGraph([48, 32], multi_relational=True, n_rela=g["n_rel"])
        gb.multiRelaInnerProductDecoder(80, g["n_rel"])
    g = synth.aminer_small()                                                                         # aminer_case
    gb.homoGraph([32, 16, 16], start_graph=True, in_dim=g["n_p"])
    gb.interGraph(64, 16, g["n_a"], target_feat_dim=16)
    gb.homoGraph([32, 32, 8])
    gb.multiClassInnerProductDecoder(72, g["n_class"])
    g = synth.freebase_d_small()                                                                     # freebase_d_case
    for n in (g["n_p"], g["n_q"]):
        gb.homoGraph([32, 16, 16], start_graph=True, in_dim=n)
        gb.interGraph(64, 16, g["n_a"], target_feat_dim=16, if_one_external=False)
    gb.homoGraph([16, 8])
    gb.multiClassInnerProductDecoder(8, g["n_class"])
    for tdim, tfd in ((16, 16), (16, 12), (16, 8)):                                                  # variants
        gb.interGraph(24, tdim, 25, target_feat_dim=tfd)
    gb.homoGraph([20, 16, 8])
    gb.homoGraph([12, 20, 8], multi_relational=True, n_rela=4, n_base=6)      # layer 2: after_relu=True
    return {"rgcn_bias": gb.myRGCN(12, 10, 4, 6, after_relu=False, bias=True),
            "gcn_improved": gb.myGCN(10, 6, improved=True, cached=False, bias=False),
            "dmt_raw": gb.multiRelaInnerProductDecoder(20, 3),
            "mcip_raw": gb.multiClassInnerProductDecoder(20, 7)}


def test_initial_distributions_match_the_reference_modules():
    """``tests/golden/make_golden.py`` seeded the global RNG, constructed the reference's modules one after the
    other and stored the fresh parameters of four of them.  Replaying its constructions with our modules under
    the same seed reproduces those parameters bit for bit: the glorot and normal initialisers of myGCN, myRGCN
    and both decoders draw the reference's values, and every module constructed before them — homoGraph with
    an embedding, multi-relational homoGraph (with an after_relu RGCN layer), interGraph with and without
    target_feat_down, both decoders — takes exactly as many numbers from the RNG as the reference's.  The script
    overwrote the RGCN bias from its own generator before storing it; the reference's took nothing from the RNG
    (the draws after it match), and ours is zero."""
    import gripnet_b200 as gb
    golden = np.load(os.path.join(GOLDEN, "variants.npz"))
    with torch.random.fork_rng():
        torch.manual_seed(20261017)                   # make_golden.py's seed
        mods = _make_golden_constructions(gb)
    for tag, m in mods.items():
        prefix = tag + ".p."
        ref = {k[len(prefix):]: golden[k] for k in golden.files if k.startswith(prefix)}
        ours = {k: v.detach().numpy() for k, v in m.named_parameters()}
        assert sorted(ours) == sorted(ref), tag
        for k in ours:
            if (tag, k) == ("rgcn_bias", "bias"):
                assert ours[k].shape == ref[k].shape and not ours[k].any(), (tag, k)
                continue
            assert ours[k].dtype == ref[k].dtype and np.array_equal(ours[k], ref[k]), (tag, k)
