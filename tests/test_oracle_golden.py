"""CPU: pins the oracle restatement (oracle/) against golden vectors that were
produced by EXECUTING THE REFERENCE (oracle/make_golden.py), and against the
live reference when GFC_REFERENCE_ROOT names a checkout of the original project."""
import glob
import os

import numpy as np
import pytest

from oracle import gso as ogso
from oracle import lsigf
from oracle import refimport

from util import rel_err

GSO_FILES = ["gso_expert3.npz", "gso_expert8.npz", "gso_expert12.npz", "gso_ties.npz", "gso_ties_r5.npz"]
FILTER_FILES = ["filter_cfg1.npz", "filter_general_e2.npz", "filter_k1_nobias.npz", "filter_nin_lt_n.npz",
                "filter_cfg2_symnorm.npz", "filter_cyclic.npz", "filter_cfg4_n12.npz"]
SAME_GSO_FILES = ["samegso_e2_nin.npz", "samegso_cfg2_f32.npz"]
BATCH_GSO_FILES = ["batchgso_cfg2_3d.npz", "batchgso_e2_4d.npz"]
RELU_FILES = ["filter_relu.npz"]
MODEL_FILES = ["model_gfl_n3.npz", "model_gfl_n8.npz"]
RECURRENT_FILES = ["recurrent_rnn_n8.npz", "recurrent_rnn_nin.npz", "recurrent_mornn_n16.npz", "recurrent_l2share_n16.npz"]
ROLLOUT_FILES = ["rollout_n12.npz", "rollout_n8.npz"]


def test_golden_inventory(golden_dir):
    have = sorted(os.path.basename(p) for p in glob.glob(os.path.join(golden_dir, "*.npz")))
    assert have == sorted(GSO_FILES + FILTER_FILES + SAME_GSO_FILES + BATCH_GSO_FILES + RELU_FILES + MODEL_FILES +
                          RECURRENT_FILES + ROLLOUT_FILES)


@pytest.mark.parametrize("name", GSO_FILES)
def test_gso_oracle_matches_reference_golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    pos, R = g["pos"], float(g["radius"])
    a = ogso.adjacency(pos, R, ogso.MODE_BINARY_LE)
    assert a.dtype == np.uint8 and np.array_equal(a, g["adj_le"])          # bit-exact
    if "s_symnorm" in g:
        s, w = ogso.gso(pos, R, ogso.MODE_SYM_NORM_LT)
        assert np.array_equal(s, g["s_symnorm"])                              # fp64-exact
        assert np.array_equal(w, (g["s_symnorm"] != 0).astype(np.uint8))
    # the scalar python-float loop (operation-for-operation scene.py:143-152) agrees too
    for p, ref in list(zip(pos.astype(np.float64), g["adj_le"]))[:40]:
        assert np.array_equal(ogso.adjacency_scalar_le(p, R), ref)


def test_gso_fixture_facts(golden_dir):
    """facts SURVEY §8c records about the cfg1 fixture"""
    g = np.load(os.path.join(golden_dir, "gso_expert3.npz"))
    assert g["pos"].shape == (3000, 3, 2) and g["pos"].dtype == np.float32
    a = g["adj_le"]
    assert np.array_equal(a, a.transpose(0, 2, 1)) and a[:, np.arange(3), np.arange(3)].sum() == 0
    deg = a.sum(2).ravel()
    assert [int((deg == d).sum()) for d in range(3)] == [6127, 2238, 635]


def _run_oracle(g):
    h, S, x = g["h"], g["S"], g["x"]
    b = g["b"] if "b" in g else None
    N, Nin = S.shape[2], x.shape[2]
    dO = g["dOut"]
    if Nin < N:
        x = np.concatenate([x, np.zeros((x.shape[0], x.shape[1], N - Nin), x.dtype)], 2)
        dO = np.concatenate([dO, np.zeros((dO.shape[0], dO.shape[1], N - Nin))], 2)
    act = lsigf.ACT_LEAKY_RELU if int(g["leaky"]) else lsigf.ACT_NONE
    y, dX, dH, db = lsigf.filter_fwd_bwd(h, S, x, b, dO, act)
    return y[:, :, :Nin], dX[:, :, :Nin], dH, db


@pytest.mark.parametrize("name", FILTER_FILES)
def test_filter_oracle_matches_reference_golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    y, dX, dH, db = _run_oracle(g)
    assert rel_err(y, g["y"]) < 1e-13                  # reference forward is fp64
    # the reference returns parameter / input grads in fp32 -> fp32 rounding of an fp64 value
    assert rel_err(dX, g["dX"]) < 2e-7
    assert rel_err(dH, g["dH"]) < 2e-7
    if "db" in g:
        assert rel_err(db, g["db"]) < 2e-7


@pytest.mark.parametrize("name", FILTER_FILES)
def test_torch_port_matches_golden(golden_dir, name):
    """the op-faithful torch port (timed as the CPU baseline) gives the reference's numbers"""
    import torch
    g = np.load(os.path.join(golden_dir, name))
    h = torch.from_numpy(g["h"]).requires_grad_(True)
    b = torch.from_numpy(g["b"]).requires_grad_(True) if "b" in g else None
    x = torch.from_numpy(g["x"]).requires_grad_(True)
    y = lsigf.graph_filter_forward_torch(h, torch.from_numpy(g["S"]), x, b)
    assert y.dtype == torch.float64
    if int(g["leaky"]):
        y = lsigf.activation_torch(y, lsigf.ACT_LEAKY_RELU)
    (y * torch.from_numpy(g["dOut"])).sum().backward()
    assert rel_err(y.detach().numpy(), g["y"]) < 1e-13
    assert rel_err(x.grad.numpy(), g["dX"]) < 2e-7
    assert rel_err(h.grad.numpy(), g["dH"]) < 2e-7
    if b is not None:
        assert rel_err(b.grad.numpy(), g["db"]) < 2e-7


@pytest.mark.parametrize("name", SAME_GSO_FILES)
def test_same_gso_oracle_matches_reference_golden(golden_dir, name):
    """GraphFilter / LSIGF (graphML.py:1111, :48): one GSO for the batch == the batch filter on
    B copies of it; the reference runs this layer in fp32, so its outputs are fp32-rounded."""
    import torch
    g = np.load(os.path.join(golden_dir, name))
    B = g["x"].shape[0]
    gb = {k: g[k] for k in g.files}
    gb["S"] = np.broadcast_to(g["S"], (B,) + g["S"].shape).copy()
    y, dX, dH, db = _run_oracle(gb)
    assert g["y"].dtype == np.float32
    assert rel_err(y, g["y"]) < 2e-6 and rel_err(dX, g["dX"]) < 2e-6
    assert rel_err(dH, g["dH"]) < 2e-6 and rel_err(db, g["db"]) < 2e-6
    # op-faithful fp32 port reproduces the reference's own rounding
    h = torch.from_numpy(g["h"]).requires_grad_(True)
    b = torch.from_numpy(g["b"]).requires_grad_(True)
    x = torch.from_numpy(g["x"]).requires_grad_(True)
    yt = lsigf.lsigf_same_gso_torch(h, torch.from_numpy(g["S"]), x, b)
    assert yt.dtype == torch.float32
    if int(g["leaky"]):
        yt = lsigf.activation_torch(yt, lsigf.ACT_LEAKY_RELU)
    (yt * torch.from_numpy(g["dOut"])).sum().backward()
    assert rel_err(yt.detach().numpy(), g["y"]) < 1e-6
    assert rel_err(x.grad.numpy(), g["dX"]) < 1e-6 and rel_err(h.grad.numpy(), g["dH"]) < 1e-6


@pytest.mark.parametrize("name", BATCH_GSO_FILES)
def test_batch_gso_oracle_matches_reference_golden(golden_dir, name):
    """GraphFilterBatchGSO (graphML.py:2174) contracts x with precomputed powers S^k in fp32: the same filter as
    GraphFilterBatch up to fp32 rounding, so the fp64 oracle reproduces its outputs to ~1e-6"""
    g = np.load(os.path.join(golden_dir, name))
    gb = {k: g[k] for k in g.files}
    if gb["S"].ndim == 3:
        gb["S"] = gb["S"][:, None]
    y, dX, dH, db = _run_oracle(gb)
    assert g["y"].dtype == np.float32
    assert rel_err(y, g["y"]) < 3e-6 and rel_err(dX, g["dX"]) < 3e-6
    assert rel_err(dH, g["dH"]) < 3e-6 and rel_err(db, g["db"]) < 3e-6


def test_relu_pairing_oracle_matches_reference_golden(golden_dir):
    """GraphFilterBatch + nn.ReLU as wired in decentralplanner.py:215-221"""
    g = np.load(os.path.join(golden_dir, "filter_relu.npz"))
    y, dX, dH, db = lsigf.filter_fwd_bwd(g["h"], g["S"], g["x"], g["b"], g["dOut"], lsigf.ACT_RELU)
    assert rel_err(y, g["y"]) < 1e-13
    assert rel_err(dX, g["dX"]) < 2e-7 and rel_err(dH, g["dH"]) < 2e-7 and rel_err(db, g["db"]) < 2e-7


@pytest.mark.parametrize("name", MODEL_FILES)
def test_model_gfl_stage_oracle_matches_reference_golden(golden_dir, name):
    """the graph-filter stage of the reference policy executed end to end (DecentralPlannerNet.addGSO / GFL,
    suhaas_model.py:149-159,182-185; loss of suhaas_agent.py:123-126): S [B,N,N] -> unsqueeze(1), LeakyReLU(0.01)"""
    g = np.load(os.path.join(golden_dir, name))
    S = g["S"][:, None]                                   # addGSO: [B,N,N] -> [B,1,N,N]  (suhaas_model.py:155)
    y, dX, dH, db = lsigf.filter_fwd_bwd(g["h"], S, g["x"], g["b"], g["dOut"], lsigf.ACT_LEAKY_RELU)
    assert rel_err(y, g["y"]) < 1e-13
    assert rel_err(dX, g["dX"]) < 2e-7                    # the stage's input is fp32 (torch.zeros default, :165): its grad is too
    assert rel_err(dH, g["dH"]) < 1e-12 and rel_err(db, g["db"]) < 1e-12


def test_closed_form_gradients_match_autograd():
    """analytic dX/dH/db/dS (SURVEY §8a a9) == torch autograd through the op-faithful port"""
    import torch
    rng = np.random.default_rng(7)
    F, E, K, G, B, N = 5, 2, 4, 3, 4, 6
    h = rng.standard_normal((F, E, K, G)); S = rng.standard_normal((B, E, N, N))
    x = rng.standard_normal((B, G, N)); b = rng.standard_normal((F, 1)); dY = rng.standard_normal((B, F, N))
    ht, St, xt, bt = [torch.from_numpy(a).requires_grad_(True) for a in (h, S, x, b)]
    y = lsigf.batch_lsigf_torch(ht, St, xt, bt)
    (y * torch.from_numpy(dY)).sum().backward()
    assert rel_err(lsigf.lsigf_forward(h, S, x, b), y.detach().numpy()) < 1e-13
    dX, dH, db, dS = lsigf.lsigf_backward(h, S, x, dY, need_dS=True)
    assert rel_err(dX, xt.grad.numpy()) < 1e-12
    assert rel_err(dH, ht.grad.numpy()) < 1e-12
    assert rel_err(db, bt.grad.numpy()) < 1e-12
    assert rel_err(dS, St.grad.numpy()) < 1e-12


def test_algebraic_properties_of_oracle():
    rng = np.random.default_rng(3)
    F, K, G, B, N = 4, 3, 5, 2, 7
    h = rng.standard_normal((F, 1, K, G)); x = rng.standard_normal((B, G, N)); b = rng.standard_normal((F, 1))
    # S = 0  =>  y = h_0 x + b ; S = I => y = (sum_k h_k) x + b
    y0 = lsigf.lsigf_forward(h, np.zeros((B, 1, N, N)), x, b)
    assert rel_err(y0, np.einsum("fg,bgn->bfn", h[:, 0, 0], x) + b.reshape(1, F, 1)) < 1e-13
    yI = lsigf.lsigf_forward(h, np.broadcast_to(np.eye(N), (B, 1, N, N)), x, b)
    assert rel_err(yI, np.einsum("fg,bgn->bfn", h[:, 0].sum(1), x) + b.reshape(1, F, 1)) < 1e-13
    # permutation equivariance
    S = rng.standard_normal((B, 1, N, N)); P = np.eye(N)[rng.permutation(N)]
    y = lsigf.lsigf_forward(h, S, x, b)
    yp = lsigf.lsigf_forward(h, P.T @ S @ P, x @ P, b)
    assert rel_err(yp, y @ P) < 1e-12


@pytest.mark.skipif(not refimport.available(),
                    reason="runs the original project's code: set GFC_REFERENCE_ROOT to a checkout of it")
def test_oracle_matches_live_reference():
    import torch
    gml = refimport.graphml()
    torch.manual_seed(11)
    m = gml.GraphFilterBatch(6, 5, 3, 2, bias=True)
    S = torch.randn(3, 2, 4, 4); x = torch.randn(3, 6, 4)
    m.addGSO(S)
    y = m(x)
    ours = lsigf.lsigf_forward(m.weight.detach().numpy(), S.numpy(), x.numpy(), m.bias.detach().numpy())
    assert y.dtype == torch.float64 and tuple(y.stride()) == (20, 1, 5)
    assert rel_err(ours, y.detach().numpy()) < 1e-13
    rng = np.random.default_rng(5)
    pos = (rng.random((30, 7, 2)) * 5).astype(np.float32)
    for p in pos:
        ref = refimport.scene_read_adj(p.astype(np.float64).tolist(), 2).reshape(7, 7).astype(np.uint8)
        assert np.array_equal(ogso.adjacency(p[None], 2, ogso.MODE_BINARY_LE)[0], ref)
        W, _ = refimport.fixed_radius_gso(p[None].astype(np.float64), 2.0)
        assert np.array_equal(ogso.gso(p[None], 2.0, ogso.MODE_SYM_NORM_LT)[0], W)


@pytest.mark.parametrize("name", RECURRENT_FILES)
def test_recurrent_oracle_matches_reference_golden(golden_dir, name):
    """oracle restatement of graphML.py:2491-2987 (two steps, hidden state carried, backward through time) vs the
    outputs and gradients of the executed reference classes"""
    import torch
    g = np.load(os.path.join(golden_dir, name))
    kind = name.split("_")[1]
    p = {k[2:]: torch.from_numpy(g[k]).requires_grad_(True) for k in g.files if k.startswith("p_")}
    S = torch.from_numpy(g["S"])
    h0 = torch.from_numpy(g["h0"]).double().requires_grad_(True)
    xs = [torch.from_numpy(g["x0"]).requires_grad_(True), torch.from_numpy(g["x1"]).requires_grad_(True)]
    hid, loss, ys = h0, 0, []
    for x, dO in zip(xs, (g["dOut0"], g["dOut1"])):
        y, hid = lsigf.recurrent_step_torch(kind, p, S, x, hid)
        ys.append(y)
        loss = loss + (y * torch.from_numpy(dO).to(y.dtype)).sum()
    loss.backward()
    assert rel_err(ys[0].detach().numpy(), g["y0"]) < 1e-12 and rel_err(ys[1].detach().numpy(), g["y1"]) < 1e-12
    assert rel_err(hid.detach().numpy(), g["hT"]) < 1e-12
    assert rel_err(xs[0].grad.numpy(), g["dx0"]) < 1e-6 and rel_err(h0.grad.numpy(), g["dh0"]) < 1e-12
    for k, v in p.items():
        assert rel_err(v.grad.numpy(), g["g_" + k]) < 1e-6, k          # reference grads are fp32-rounded


@pytest.mark.parametrize("name", ROLLOUT_FILES)
def test_rollout_oracle_matches_reference_golden(golden_dir, name):
    """the reference's per-robot batch-1 pattern gives, for every robot, the same column as ONE batched pass: oracle GSO
    (scene.py:140-154 restatement) + oracle filter stack vs the golden produced by the per-robot loop"""
    g = np.load(os.path.join(golden_dir, name))
    S = ogso.gso(g["pos"], float(g["radius"]), ogso.MODE_BINARY_LE)[0][:, None]
    y = g["x"]
    for l in range(len(g["dims"]) - 1):
        y = lsigf.activation(lsigf.lsigf_forward(g["h%d" % l], S, y, g["b%d" % l]), lsigf.ACT_LEAKY_RELU)
    assert rel_err(y, g["expected"]) < 1e-12
