"""CPU: the nn.Module surface mirrors the reference layer
(utils/graphUtils/graphML.py:2369-2488) — names, shapes, init law, asserts, repr,
state_dict compatibility — and the product refuses to run without CUDA."""
import math
import os

import numpy as np
import pytest
import torch

import gnnfc
from oracle import refimport

from util import rel_err

NO_REFERENCE = "runs the original project's code: set GFC_REFERENCE_ROOT to a checkout of it"


def test_constructor_and_parameters():
    torch.manual_seed(0)
    m = gnnfc.GraphFilterBatch(128, 64, 3)
    assert (m.G, m.F, m.K, m.E) == (128, 64, 3, 1) and m.S is None
    assert tuple(m.weight.shape) == (64, 1, 3, 128) and tuple(m.bias.shape) == (64, 1)
    assert list(m.state_dict().keys()) == ["weight", "bias"]
    s = 1.0 / math.sqrt(128 * 3)
    assert float(m.weight.abs().max()) <= s and float(m.bias.abs().max()) <= s
    assert float(m.weight.abs().max()) > 0.9 * s        # uniform, not tiny
    m2 = gnnfc.GraphFilterBatch(4, 8, 2, E=2, bias=False)
    assert m2.bias is None and list(m2.state_dict().keys()) == ["weight"]
    assert tuple(m2.weight.shape) == (8, 2, 2, 4)


def test_extra_repr_matches_reference_format():
    m = gnnfc.GraphFilterBatch(4, 8, 3)
    assert repr(m) == ("GraphFilterBatch(in_features=4, out_features=8, filter_taps=3, "
                       "edge_features=1, bias=True, no GSO stored)")
    m.addGSO(torch.zeros(2, 1, 5, 5))
    assert repr(m).endswith("GSO stored)") and "no GSO" not in repr(m)


def test_addgso_asserts_like_reference():
    m = gnnfc.GraphFilterBatch(4, 8, 3, E=1)
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(2, 5, 5))            # rank != 4   (graphML.py:2451)
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(2, 2, 5, 5))         # E mismatch  (graphML.py:2453)
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(2, 1, 5, 4))         # non-square  (graphML.py:2455)
    S = torch.zeros(2, 1, 5, 5)
    m.addGSO(S)
    assert m.N == 5 and m.S is S                  # stored by reference (graphML.py:2456)


def test_no_cpu_fallback():
    m = gnnfc.GraphFilterBatch(8, 8, 2)
    m.addGSO(torch.zeros(2, 1, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU"):
        m(torch.zeros(2, 8, 4))
    with pytest.raises(RuntimeError, match="no CPU|CUDA"):
        gnnfc.build_gso(torch.zeros(2, 4, 2), 2.0)


# (golden, torch seed): the taps stored in these goldens are the reference layer's own draw right after
# torch.manual_seed(seed) (oracle/make_golden.py)
REF_INIT_GOLDENS = {
    "GraphFilterBatch": (("filter_cfg1.npz", 0), ("filter_general_e2.npz", 1), ("filter_k1_nobias.npz", 2),
                         ("filter_nin_lt_n.npz", 3), ("filter_cfg2_symnorm.npz", 4), ("filter_cyclic.npz", 5),
                         ("filter_cfg4_n12.npz", 6), ("filter_relu.npz", 12)),
    "GraphFilter": (("samegso_e2_nin.npz", 10), ("samegso_cfg2_f32.npz", 11)),
    "GraphFilterBatchGSO": (("batchgso_cfg2_3d.npz", 20), ("batchgso_e2_4d.npz", 21)),
}


def _check_reference_init(golden_dir, name):
    """the reference layer's parameters load into ours (same keys / shapes) and our init law draws exactly them"""
    layers = []
    for fname, seed in REF_INIT_GOLDENS[name]:
        g = np.load(os.path.join(golden_dir, fname))
        F, E, K, G = g["h"].shape
        ref_sd = {"weight": torch.from_numpy(g["h"])}
        if "b" in g:
            ref_sd["bias"] = torch.from_numpy(g["b"])
        torch.manual_seed(seed)
        ours = getattr(gnnfc, name)(G, F, K, E, bias="b" in g)
        assert list(ours.state_dict().keys()) == list(ref_sd.keys())
        for k, v in ref_sd.items():
            assert torch.equal(ours.state_dict()[k], v), (fname, k)
        ours.load_state_dict(ref_sd)
        layers.append((ours, g))
    return layers


def test_state_dict_roundtrip_with_reference_layer(golden_dir):
    _check_reference_init(golden_dir, "GraphFilterBatch")


def test_shard_range_partitions_batch():
    for total in (0, 1, 7, 64, 4096, 65537):
        for world in (1, 2, 3, 8):
            spans = [gnnfc.shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_grad_bucket_pack_unpack_single_process():
    p1 = torch.nn.Parameter(torch.randn(3, 4)); p2 = torch.nn.Parameter(torch.randn(5))
    p1.grad = torch.randn(3, 4); p2.grad = None
    b = gnnfc.GradBucket([p1, p2])
    flat = b.pack()
    assert flat.numel() == 17 and torch.equal(flat[:12].view(3, 4), p1.grad) and float(flat[12:].abs().sum()) == 0
    flat.mul_(2)
    g1 = p1.grad.clone()
    b.allreduce(); b.unpack()
    assert torch.allclose(p1.grad, 2 * g1) and p2.grad is not None and float(p2.grad.abs().sum()) == 0


# --------------------------------------------------------------------------- #
# recorded-data re-layout (SURVEY §8 f-4)
# --------------------------------------------------------------------------- #
def test_recording_relayout_matches_the_reference_loops():
    """gnnfc.data.* == the Python loops of RobotDataset.__init__ (custom_dataset.py:15-63) and the agent's
    robot-0 view (suhaas_agent.py:117)"""
    import numpy as np
    import torch
    import gnnfc
    rng = np.random.default_rng(5)
    nA, T = 4, 7
    graph_rows = (rng.random((nA * T, nA * nA)) < 0.5).astype(np.float32)     # data.py:43 layout, robots concatenated
    gt_rows = rng.standard_normal((nA * T, 2)).astype(np.float32)
    # the reference's loops, restated
    c3 = np.zeros((T, nA, nA, nA))
    c2 = np.zeros((T, nA, 2))
    for i in range(T):
        for j in range(nA):
            c3[i, j] = graph_rows[j * T + i].reshape((nA, nA))                  # custom_dataset.py:40-42
            c2[i, j] = gt_rows[j * T + i]                                        # custom_dataset.py:32-34
    assert np.array_equal(gnnfc.graphs_from_recording(graph_rows, nA).numpy(), c3.astype(np.float32))
    assert np.array_equal(gnnfc.robot_major_to_batch(gt_rows, nA).numpy(), c2.astype(np.float32))
    S = gnnfc.gso_batch_from_recording(graph_rows, nA)
    assert S.shape == (T, 1, nA, nA) and S.is_contiguous() and S.dtype == torch.float32
    assert np.array_equal(S[:, 0].numpy(), c3[:, 0].astype(np.float32))          # suhaas_agent.py:117
    # the live reference class, when a checkout of the original project is given (GFC_REFERENCE_ROOT)
    from oracle import refimport
    if refimport.available():
        import sys
        sys.path.insert(0, refimport.REF_ROOT)
        try:
            from custom_dataset import RobotDataset
        finally:
            sys.path.pop(0)
        obs = rng.standard_normal((nA * T, 4)).astype(np.float32)
        ds = RobotDataset(obs, gt_rows, graph_rows, np.zeros(nA * T), np.zeros(nA * T), nA, inW=2, inH=2)
        assert np.array_equal(ds.graphs, c3) and np.array_equal(ds.gt, c2)
        assert np.array_equal(gnnfc.graphs_from_recording(graph_rows, nA).numpy(), ds.graphs.astype(np.float32))
    # positionList fixtures: [E, steps*nA, 2] with index t*nA + r
    pl = rng.standard_normal((2, 5 * 3, 2))
    p = gnnfc.positions_from_recording(pl, 3)
    assert p.shape == (10, 3, 2) and np.allclose(p[6, 2].numpy(), pl[1, 1 * 3 + 2].astype(np.float32))


# --------------------------------------------------------------------------- #
# the other two drop-in layers: GraphFilter (graphML.py:1111) and GraphFilterBatchGSO (graphML.py:2174)
# --------------------------------------------------------------------------- #
def test_same_gso_and_batch_gso_layers_surface():
    m = gnnfc.GraphFilter(4, 8, 3, E=2)
    assert tuple(m.weight.shape) == (8, 2, 3, 4) and tuple(m.bias.shape) == (8, 1) and m.S is None
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(1, 2, 5, 5))           # rank != 3   (graphML.py:1192)
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(1, 5, 5))              # E mismatch  (graphML.py:1194)
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(2, 5, 4))              # non-square  (graphML.py:1196)
    m.addGSO(torch.zeros(2, 5, 5))
    assert m.N == 5 and repr(m).endswith("GSO stored)")
    with pytest.raises(RuntimeError, match="no CPU"):
        m(torch.zeros(3, 4, 5))

    g = gnnfc.GraphFilterBatchGSO(4, 8, 3)
    assert g.extra_repr().endswith("no GSO stored")
    g.addGSO(torch.zeros(6, 5, 5))                  # 3-d: one edge feature (graphML.py:2231-2233)
    assert tuple(g.S.shape) == (6, 1, 5, 5) and (g.N, g.B) == (5, 6)
    assert g.extra_repr().endswith("GSO stored: number_nodes=5, batch_size=6")
    g.addGSO(torch.zeros(6, 5, 4))                  # any other shape is ignored, the previous GSO stays (:2241-2244)
    assert tuple(g.S.shape) == (6, 1, 5, 5)
    S = torch.rand(2, 1, 3, 3)
    g.addGSO(S)
    SK = g.SK                                       # matrixPowersBatch (graphML.py:2063): I, S, S^2
    assert tuple(SK.shape) == (2, 1, 3, 3, 3)
    assert torch.equal(SK[:, :, 0], torch.eye(3).expand(2, 1, 3, 3)) and torch.equal(SK[:, :, 1], S)
    assert torch.allclose(SK[:, :, 2], S @ S)
    with pytest.raises(AssertionError):
        g(torch.zeros(2, 4, 2))                     # batchLSIGF asserts the node count, no zero-padding (:2154)


def test_new_layers_match_the_live_reference_surface(golden_dir):
    """same keys, init law and draw order as the reference's GraphFilter / GraphFilterBatchGSO, and the
    reference's extra_repr once a GSO is stored (both recorded from the reference by oracle/make_golden.py)"""
    for ours, g in _check_reference_init(golden_dir, "GraphFilter"):
        ours.addGSO(torch.from_numpy(g["S"]))
        assert ours.N == g["S"].shape[-1]
    for ours, g in _check_reference_init(golden_dir, "GraphFilterBatchGSO"):
        ours.addGSO(torch.from_numpy(g["S"]))
        assert ours.extra_repr() == str(g["repr"]) and ours.N == g["S"].shape[-1]
        # the powers attribute: contracted with x and the taps it gives the reference's fp32 output
        z = torch.einsum("bgm,bekmn->bekgn", torch.from_numpy(g["x"]).double(), ours.SK.double())
        y = torch.einsum("fekg,bekgn->bfn", torch.from_numpy(g["h"]).double(), z) + torch.from_numpy(g["b"]).double()
        if int(g["leaky"]):
            y = torch.nn.functional.leaky_relu(y, 0.01)
        assert rel_err(y.numpy(), g["y"]) < 3e-6


@pytest.mark.skipif(not refimport.available(), reason=NO_REFERENCE)
def test_reference_policy_constructs_with_the_dropin_layer():
    """a10: the UNMODIFIED reference model file (graphs/models/suhaas_model.py) executed with its
    ``import utils.graphUtils.graphML as gml`` resolving to gnnfc: the GFL stage is built from the drop-in layer
    (:114), the reference model's own state_dict loads into it, and ``addGSO`` + the per-forward wiring
    ``self.GFL[2*l].addGSO(self.S)`` (:149-159,182) hand the layer the ``[B,1,N,N]`` GSO it expects."""
    RefNet = refimport.decentral_planner_net()
    SwapNet = refimport.decentral_planner_net(gnnfc)
    torch.manual_seed(0)
    ref = RefNet(nA=3)
    swp = SwapNet(nA=3)
    assert type(swp.GFL[0]) is gnnfc.GraphFilterBatch and type(ref.GFL[0]) is not gnnfc.GraphFilterBatch
    assert repr(swp.GFL) == repr(ref.GFL)
    assert [(k, tuple(v.shape)) for k, v in swp.state_dict().items()] == \
           [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    assert sum(p.numel() for p in swp.parameters()) == 2584034          # SURVEY 8c(4)
    missing, unexpected = swp.load_state_dict(ref.state_dict())
    assert not missing and not unexpected
    assert torch.equal(swp.GFL[0].weight, ref.GFL[0].weight) and torch.equal(swp.GFL[0].bias, ref.GFL[0].bias)
    S = torch.zeros(5, 3, 3, dtype=torch.float64)
    swp.addGSO(S)
    assert swp.S.shape == (5, 1, 3, 3)
    for l in range(swp.L):
        swp.GFL[2 * l].addGSO(swp.S)                                     # suhaas_model.py:182
    assert swp.GFL[0].N == 3 and swp.GFL[0].S is swp.S
    with pytest.raises(AssertionError):
        swp.addGSO(torch.zeros(5, 1, 3, 3))                              # :153  E == 1 wants [B,N,N]
    assert swp.double().GFL[0].weight.dtype == torch.float64            # the agent runs the model in double


# --------------------------------------------------------------------------- #
# §8 f-4: recurrent layers (graphML.py:2491-2987) — surface; the arithmetic is checked on the GPU against goldens
# --------------------------------------------------------------------------- #
def test_recurrent_layers_surface():
    m = gnnfc.GraphFilterRNNBatch(4, 8, 6, 3)
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == [
        ("weight_A", (8, 1, 3, 4)), ("weight_B", (8, 1, 3, 8)), ("weight_D", (6, 1, 3, 8)),
        ("bias_A", (8, 1)), ("bias_B", (8, 1)), ("bias_D", (6, 1))]
    assert float(m.weight_A.abs().max()) <= 1 / math.sqrt(4 * 3) and float(m.weight_B.abs().max()) <= 1 / math.sqrt(8 * 3)
    assert repr(m) == ("GraphFilterRNNBatch(in_features=4, out_features=6, hidden_features=8, filter_taps=3, "
                       "edge_features=1, bias=True, no GSO stored)")
    with pytest.raises(AssertionError):
        m.addGSO(torch.zeros(2, 5, 5))                       # graphML.py:2587
    m.addGSO(torch.zeros(2, 1, 5, 5))
    assert m.N == 5 and repr(m).endswith("GSO stored)")
    h = torch.zeros(2, 8, 5)
    m.updateHiddenState(h)
    assert m.hiddenState is h
    with pytest.raises(RuntimeError, match="no CPU"):
        m(torch.zeros(2, 4, 5))
    mo = gnnfc.GraphFilterMoRNNBatch(4, 8, 6, 3)
    assert tuple(mo.weight_B.shape) == (8, 8) and tuple(mo.weight_D.shape) == (6, 8)
    assert float(mo.weight_B.abs().max()) <= 1 / math.sqrt(8)
    nb = gnnfc.GraphFilterRNNBatch(4, 8, 6, 3, bias=False)   # the reference raises here (documented deviation)
    assert nb.bias_A is None and nb.bias_D is None and "bias=False" in repr(nb)
    # torchpermul is the reference's elementwise broadcast product, not a matmul (graphML.py:2656-2679)
    x, w, b = torch.rand(2, 3, 3), torch.rand(3, 3), torch.rand(3, 1)
    assert torch.equal(gnnfc.torchpermul(w, x, b), (x.permute(0, 2, 1) * w.permute(1, 0)).permute(0, 2, 1) + b)


def test_recurrent_layers_match_the_live_reference_surface(golden_dir):
    """the parameters of the reference's recurrent layers right after torch.manual_seed(seed), as recorded in the
    recurrent goldens (p_*, registration order; oracle/make_golden.py): ours draws the same ones in the same order"""
    for tag, name, seed in (("rnn_n8", "GraphFilterRNNBatch", 21), ("rnn_nin", "GraphFilterRNNBatch", 22),
                            ("mornn_n16", "GraphFilterMoRNNBatch", 23), ("l2share_n16", "GraphFilterL2ShareBatch", 24)):
        g = np.load(os.path.join(golden_dir, "recurrent_%s.npz" % tag))
        G, H, F, K, N = (int(v) for v in g["dims"][:5])
        ref_sd = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("p_")}
        torch.manual_seed(seed)
        ours = getattr(gnnfc, name)(G, H, F, K)
        assert list(ours.state_dict().keys()) == list(ref_sd.keys())
        for k, v in ref_sd.items():
            assert torch.equal(ours.state_dict()[k], v), (tag, k)                  # same init law and draw order
        ours.load_state_dict(ref_sd)
        ours.addGSO(torch.from_numpy(g["S"]))
        assert ours.N == N


# --------------------------------------------------------------------------- #
# §8 f-4: device-side recording loader vs RobotDataset + DataLoader (custom_dataset.py, suhaas_agent.py:110-121)
# --------------------------------------------------------------------------- #
def _recording(rng, nA, T, inW, inH):
    per_robot = []
    for r in range(nA):
        per_robot.append(dict(observations=rng.random((T, inW * inH)).astype(np.float32),
                              actions=rng.standard_normal((T, 2)).astype(np.float32),
                              graph=(rng.random((T, nA * nA)) < 0.5).astype(np.float32),
                              obs2=rng.standard_normal((T, 6 + nA)).astype(np.float32)))
    return per_robot


def test_recording_loader_matches_the_reference_dataset_loops():
    rng = np.random.default_rng(8)
    nA, T, inW, inH = 3, 11, 4, 5
    rec = _recording(rng, nA, T, inW, inH)
    ld = gnnfc.RecordingLoader.from_recordings(rec, batch_size=4, shuffle=False, device="cpu", inW=inW, inH=inH)
    assert len(ld) == 2                                                   # drop_last=True like suhaas_agent.py:111
    batches = list(ld)
    assert [tuple(batches[0][k].shape) for k in ("data", "graphs", "actions", "refs", "alphas", "S")] == \
           [(4, nA, inW, inH), (4, nA, nA, nA), (4, nA, 2), (4, nA, 1), (4, nA, 1), (4, nA, nA)]
    assert all(v.dtype == torch.float64 for v in batches[0].values())
    # the reference's loops restated (custom_dataset.py:15-63): c[i, j] = rows[j*T + i]
    for bi, bt in enumerate(batches):
        for q in range(4):
            i = bi * 4 + q
            for j in range(nA):
                assert np.array_equal(bt["data"][q, j].numpy(), rec[j]["observations"][i].reshape(inW, inH).astype(np.float64))
                assert np.array_equal(bt["graphs"][q, j].numpy(), rec[j]["graph"][i].reshape(nA, nA).astype(np.float64))
                assert np.array_equal(bt["actions"][q, j].numpy(), rec[j]["actions"][i].astype(np.float64))
                assert bt["refs"][q, j, 0] == float(rec[j]["obs2"][i, 1]) and bt["alphas"][q, j, 0] == float(rec[j]["obs2"][i, 2])
            assert torch.equal(bt["S"][q], bt["graphs"][q, 0])            # suhaas_agent.py:117
    # shuffling: a permutation of the time steps, every step at most once, remainder dropped
    g = torch.Generator().manual_seed(0)
    ld2 = gnnfc.RecordingLoader.from_recordings(rec, batch_size=4, shuffle=True, device="cpu", inW=inW, inH=inH, generator=g)
    seen = torch.cat([b["actions"][:, 0, 0] for b in ld2])
    ref_col = torch.from_numpy(rec[0]["actions"][:, 0].astype(np.float64))
    assert len(seen) == 8 and len(set(seen.tolist())) == 8 and all(v in ref_col.tolist() for v in seen.tolist())
    ld3 = gnnfc.RecordingLoader.from_recordings(rec, batch_size=4, shuffle=False, drop_last=False, device="cpu", inW=inW, inH=inH)
    assert len(ld3) == 3 and list(ld3)[-1]["data"].shape[0] == 3


@pytest.mark.skipif(not refimport.available(), reason=NO_REFERENCE)
def test_recording_loader_matches_the_live_robot_dataset():
    import sys
    sys.path.insert(0, refimport.REF_ROOT)
    try:
        from custom_dataset import RobotDataset
    finally:
        sys.path.pop(0)
    rng = np.random.default_rng(9)
    nA, T, inW, inH = 4, 6, 3, 3
    rec = _recording(rng, nA, T, inW, inH)
    cat = lambda k: np.concatenate([r[k] for r in rec], axis=0)           # noqa: E731  (Data.append, data.py:153-156)
    ds = RobotDataset(cat("observations"), cat("actions"), cat("graph"), cat("obs2")[:, 1], cat("obs2")[:, 2], nA,
                      inW=inW, inH=inH, transform=True)
    ld = gnnfc.RecordingLoader.from_recordings(rec, batch_size=T, shuffle=False, device="cpu", inW=inW, inH=inH)
    bt = next(iter(ld))
    for i in range(T):
        item = ds[i]
        for k in ("data", "graphs", "actions", "refs", "alphas"):
            assert torch.equal(bt[k][i], item[k]), k
