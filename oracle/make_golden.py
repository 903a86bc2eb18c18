"""TEST INFRASTRUCTURE ONLY — generate ``tests/golden/*.npz`` by EXECUTING THE
REFERENCE ITSELF (only possible with a checkout of the original project).  Re-run
with ``GFC_REFERENCE_ROOT=<checkout> python -m oracle.make_golden`` from the repo root.

Everything stored under "expected" comes out of reference code:
  * ``Scene.readADjMatrix``                             (scene.py:140-154)
  * ``computeAdjacencyMatrix_fixedCommRadius``          (utils/multirobotsim_dcenlocal.py:291-317)
  * ``GraphFilterBatch.addGSO/forward`` + autograd      (utils/graphUtils/graphML.py:2369-2488)
  * ``nn.LeakyReLU`` as wired in the policy             (graphs/models/suhaas_model.py:120)
Inputs are the reference's recorded trajectories (positionList_*.npy; layout
index = t*N + robot, test5_more_robots.py:176-178) or seeded random tensors.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import refimport as ri  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def load_frames(name, n):
    """positionList_* [episodes, T*n, 2] float64 -> [episodes*T, n, 2]."""
    a = np.load(os.path.join(ri.REF_ROOT, name))
    ep, tn, _ = a.shape
    assert tn % n == 0
    return a.reshape(ep * (tn // n), n, 2)


def ref_binary(frames, radius):
    out = np.zeros((len(frames), frames.shape[1], frames.shape[1]), dtype=np.uint8)
    for i, fr in enumerate(frames):
        a = ri.scene_read_adj(fr.tolist(), radius)
        assert a.shape == (1, fr.shape[0] ** 2)
        out[i] = a.reshape(fr.shape[0], fr.shape[0]).astype(np.uint8)
    return out


def ref_symnorm(frames, radius):
    out = np.zeros((len(frames), frames.shape[1], frames.shape[1]), dtype=np.float64)
    for i, fr in enumerate(frames):
        W, _ = ri.fixed_radius_gso(fr[None].astype(np.float64), radius)
        out[i] = W[0]
    return out


def gso_goldens():
    # cfg1: every frame of the 3-robot expert run (3000 graphs)
    f3 = load_frames("positionList_expert_3.npy", 3)
    assert np.array_equal(f3.astype(np.float32).astype(np.float64), f3), "fixture not fp32-exact"
    np.savez_compressed(os.path.join(OUT, "gso_expert3.npz"),
                        pos=f3.astype(np.float32), radius=2.0,
                        adj_le=ref_binary(f3, 2), )
    # 8 robots: every 8th frame; both builders
    f8 = load_frames("positionList_expert_8.npy", 8)[::8]
    np.savez_compressed(os.path.join(OUT, "gso_expert8.npz"),
                        pos=f8.astype(np.float32), radius=2.0,
                        adj_le=ref_binary(f8, 2), s_symnorm=ref_symnorm(f8, 2.0))
    # 12 robots (long run): 250 frames spread over the file
    f12 = load_frames("positionList_expert_12_longer.npy", 12)
    f12 = f12[:: max(1, len(f12) // 250)][:250]
    np.savez_compressed(os.path.join(OUT, "gso_expert12.npz"),
                        pos=f12.astype(np.float32), radius=2.0,
                        adj_le=ref_binary(f12, 2), s_symnorm=ref_symnorm(f12, 2.0))
    # ties d == R and near-threshold pairs; isolated nodes; coincident robots
    ties = np.array([
        [[0, 0], [2, 0], [0, -2], [2, 2], [4, 0], [1, 0]],
        [[0, 0], [1.2, 1.6], [-1.2, 1.6], [0, 2.0000002], [0, 1.9999999], [9, 9]],
        [[0, 0], [0, 0], [2, 0], [2, 0], [50, 50], [-50, 50]],
        [[1, 1], [1 + 2 ** -20, 1], [3, 1], [3 + 2 ** -22, 1], [1, 3], [1, 3 - 2 ** -22]],
    ], dtype=np.float32).astype(np.float64)
    np.savez_compressed(os.path.join(OUT, "gso_ties.npz"),
                        pos=ties.astype(np.float32), radius=2.0,
                        adj_le=ref_binary(ties, 2), s_symnorm=ref_symnorm(ties, 2.0))
    tri = np.array([[[0, 0], [3, 4], [-3, 4], [6, 8], [3, 4.000001], [0, 5]]],
                   dtype=np.float32).astype(np.float64)
    np.savez_compressed(os.path.join(OUT, "gso_ties_r5.npz"),
                        pos=tri.astype(np.float32), radius=5.0,
                        adj_le=ref_binary(tri, 5), s_symnorm=ref_symnorm(tri, 5.0))


def run_ref_filter(gml, h, b, S, x, dOut, leaky, nin=None):
    F, E, K, G = h.shape
    m = gml.GraphFilterBatch(G, F, K, E, bias=b is not None)
    with torch.no_grad():
        m.weight.copy_(torch.from_numpy(h))
        if b is not None:
            m.bias.copy_(torch.from_numpy(b))
    xt = torch.from_numpy(x).clone().requires_grad_(True)
    m.addGSO(torch.from_numpy(S))
    y = m(xt)
    if leaky:
        y = torch.nn.LeakyReLU()(y)
    assert y.dtype == torch.float64
    (y * torch.from_numpy(dOut)).sum().backward()
    out = dict(h=h, S=S, x=x, dOut=dOut, leaky=np.int32(leaky),
               y=y.detach().numpy(), dX=xt.grad.numpy().astype(np.float64),
               dH=m.weight.grad.numpy().astype(np.float64))
    if b is not None:
        out["b"] = b
        out["db"] = m.bias.grad.numpy().astype(np.float64)
    return out


def run_ref_same_gso(gml, h, b, S, x, dOut, leaky):
    """the reference's same-GSO layer (GraphFilter / LSIGF, graphML.py:1111, :48)."""
    F, E, K, G = h.shape
    m = gml.GraphFilter(G, F, K, E, bias=b is not None)
    with torch.no_grad():
        m.weight.copy_(torch.from_numpy(h))
        if b is not None:
            m.bias.copy_(torch.from_numpy(b))
    xt = torch.from_numpy(x).clone().requires_grad_(True)
    m.addGSO(torch.from_numpy(S))
    y = m(xt)
    if leaky:
        y = torch.nn.LeakyReLU()(y)
    (y * torch.from_numpy(dOut).to(y.dtype)).sum().backward()
    out = dict(h=h, S=S, x=x, dOut=dOut, leaky=np.int32(leaky),
               y=y.detach().numpy(), dX=xt.grad.numpy(), dH=m.weight.grad.numpy())
    if b is not None:
        out["b"] = b
        out["db"] = m.bias.grad.numpy()
    return out


def same_gso_goldens():
    gml = ri.graphml()
    rng = np.random.default_rng(4321)

    def taps(G, F, K, E, bias, seed):
        torch.manual_seed(seed)
        m = gml.GraphFilter(G, F, K, E, bias=bias)
        return (m.weight.detach().numpy().copy(),
                m.bias.detach().numpy().copy() if bias else None)

    # E=2, weighted asymmetric GSO, Nin < N, LeakyReLU (float32 throughout: LSIGF has no
    # dtype casts, so the reference's float32 parameters reject a float64 input)
    h, b = taps(6, 5, 3, 2, True, 10)
    S = rng.standard_normal((2, 7, 7)).astype(np.float32)
    x = rng.standard_normal((4, 6, 5)).astype(np.float32)
    dOut = rng.standard_normal((4, 5, 5)).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "samegso_e2_nin.npz"),
                        **run_ref_same_gso(gml, h, b, S, x, dOut, True))

    # float32 in (the dtype the reference's models feed), one 8-robot normalised GSO, 32->32, K=3
    g8 = np.load(os.path.join(OUT, "gso_expert8.npz"))
    S = g8["s_symnorm"][5].astype(np.float32)[None]
    h, b = taps(32, 32, 3, 1, True, 11)
    x = rng.standard_normal((16, 32, 8)).astype(np.float32)
    dOut = rng.standard_normal((16, 32, 8)).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "samegso_cfg2_f32.npz"),
                        **run_ref_same_gso(gml, h, b, S, x, dOut, False))


def batch_gso_goldens():
    """GraphFilterBatchGSO (graphML.py:2174): precomputed powers, fp32, S given as [B,N,N] and as [B,E,N,N]"""
    gml = ri.graphml()
    rng = np.random.default_rng(777)

    def run(h, b, S, x, dOut, leaky):
        F, E, K, G = h.shape
        m = gml.GraphFilterBatchGSO(G, F, K, E, bias=True)
        with torch.no_grad():
            m.weight.copy_(torch.from_numpy(h))
            m.bias.copy_(torch.from_numpy(b))
        xt = torch.from_numpy(x).clone().requires_grad_(True)
        m.addGSO(torch.from_numpy(S))
        y = m(xt)
        if leaky:
            y = torch.nn.LeakyReLU()(y)
        (y * torch.from_numpy(dOut)).sum().backward()
        return dict(h=h, b=b, S=S, x=x, dOut=dOut, leaky=np.int32(leaky), y=y.detach().numpy(), dX=xt.grad.numpy(),
                    dH=m.weight.grad.numpy(), db=m.bias.grad.numpy(), repr=np.array(m.extra_repr()))

    def taps(G, F, K, E, seed):
        torch.manual_seed(seed)
        m = gml.GraphFilterBatchGSO(G, F, K, E, bias=True)
        return m.weight.detach().numpy().copy(), m.bias.detach().numpy().copy()

    # 3-d S: the normalised GSOs of 24 frames of the 8-robot fixture, 32 -> 32, K = 3, LeakyReLU
    g8 = np.load(os.path.join(OUT, "gso_expert8.npz"))
    S = g8["s_symnorm"][40:64].astype(np.float32)
    h, b = taps(32, 32, 3, 1, 20)
    x = rng.standard_normal((24, 32, 8)).astype(np.float32)
    dOut = rng.standard_normal((24, 32, 8)).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "batchgso_cfg2_3d.npz"), **run(h, b, S, x, dOut, True))

    # 4-d S with two edge features, weighted and asymmetric, odd sizes
    h, b = taps(5, 6, 4, 2, 21)
    S = (0.5 * rng.standard_normal((3, 2, 7, 7))).astype(np.float32)
    x = rng.standard_normal((3, 5, 7)).astype(np.float32)
    dOut = rng.standard_normal((3, 6, 7)).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "batchgso_e2_4d.npz"), **run(h, b, S, x, dOut, False))


def relu_golden():
    """GraphFilterBatch followed by nn.ReLU, the pairing of decentralplanner.py:215-221 (suhaas_model.py uses
    LeakyReLU): 5 robots of the expert fixture family shape, 16 -> 24, K = 2"""
    gml = ri.graphml()
    rng = np.random.default_rng(99)
    torch.manual_seed(12)
    m = gml.GraphFilterBatch(16, 24, 2, 1, bias=True)
    h, b = m.weight.detach().numpy().copy(), m.bias.detach().numpy().copy()
    S = (rng.random((9, 1, 5, 5)) < 0.5).astype(np.float32)
    x = rng.standard_normal((9, 16, 5)).astype(np.float32)
    dOut = rng.standard_normal((9, 24, 5))
    xt = torch.from_numpy(x).clone().requires_grad_(True)
    m.addGSO(torch.from_numpy(S))
    y = torch.nn.ReLU()(m(xt))
    (y * torch.from_numpy(dOut)).sum().backward()
    np.savez_compressed(os.path.join(OUT, "filter_relu.npz"), h=h, b=b, S=S, x=x, dOut=dOut, leaky=np.int32(0),
                        relu=np.int32(1), y=y.detach().numpy(), dX=xt.grad.numpy().astype(np.float64),
                        dH=m.weight.grad.numpy().astype(np.float64), db=m.bias.grad.numpy().astype(np.float64))


def filter_goldens():
    gml = ri.graphml()
    rng = np.random.default_rng(1234)

    def taps(G, F, K, E, bias, seed):
        torch.manual_seed(seed)
        m = gml.GraphFilterBatch(G, F, K, E, bias=bias)  # reference reset_parameters()
        return (m.weight.detach().numpy().copy(),
                m.bias.detach().numpy().copy() if bias else None)

    # case cfg1: first 64 graphs of the 3-robot expert fixture, 128->128, K=3, LeakyReLU
    g = np.load(os.path.join(OUT, "gso_expert3.npz"))
    idx = np.arange(0, 3000, 3000 // 64)[:64]
    S = g["adj_le"][idx].astype(np.float32)[:, None]
    h, b = taps(128, 128, 3, 1, True, 0)
    torch.manual_seed(0)
    x = torch.randn(64, 128, 3).numpy()
    dOut = rng.standard_normal((64, 128, 3))
    np.savez_compressed(os.path.join(OUT, "filter_cfg1.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, True))

    # case general: asymmetric weighted S, E=2, odd sizes, no activation
    h, b = taps(5, 7, 4, 2, True, 1)
    S = rng.standard_normal((3, 2, 6, 6)).astype(np.float32)
    x = rng.standard_normal((3, 5, 6)).astype(np.float32)
    dOut = rng.standard_normal((3, 7, 6))
    np.savez_compressed(os.path.join(OUT, "filter_general_e2.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, False))

    # case K=1, no bias
    h, b = taps(8, 4, 1, 1, False, 2)
    S = rng.standard_normal((5, 1, 4, 4)).astype(np.float32)
    x = rng.standard_normal((5, 8, 4)).astype(np.float32)
    dOut = rng.standard_normal((5, 4, 4))
    np.savez_compressed(os.path.join(OUT, "filter_k1_nobias.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, False))

    # case Nin < N zero-pad (graphML.py:2464-2476)
    h, b = taps(6, 6, 3, 1, True, 3)
    S = (rng.random((4, 1, 6, 6)) < 0.4).astype(np.float32)
    x = rng.standard_normal((4, 6, 4)).astype(np.float32)
    dOut = rng.standard_normal((4, 6, 4))
    np.savez_compressed(os.path.join(OUT, "filter_nin_lt_n.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, True))

    # case cfg2-shaped slice with the normalised GSO of the 8-robot fixture
    g8 = np.load(os.path.join(OUT, "gso_expert8.npz"))
    S = g8["s_symnorm"][:32].astype(np.float32)[:, None]
    h, b = taps(32, 32, 3, 1, True, 4)
    x = rng.standard_normal((32, 32, 8)).astype(np.float32)
    dOut = rng.standard_normal((32, 32, 8))
    np.savez_compressed(os.path.join(OUT, "filter_cfg2_symnorm.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, True))

    # case cyclic (asymmetric) GSO from suhaas_test.py:16
    cyc = np.array([[0, 0, 1], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    S = np.broadcast_to(cyc, (2, 1, 3, 3)).copy()
    h, b = taps(16, 16, 3, 1, True, 5)
    x = rng.standard_normal((2, 16, 3)).astype(np.float32)
    dOut = rng.standard_normal((2, 16, 3))
    np.savez_compressed(os.path.join(OUT, "filter_cyclic.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, True))

    # case 12 robots, binary GSO, 128->128 (rollout layer shape, cfg4)
    g12 = np.load(os.path.join(OUT, "gso_expert12.npz"))
    S = g12["adj_le"][:8].astype(np.float32)[:, None]
    h, b = taps(128, 128, 3, 1, True, 6)
    x = rng.standard_normal((8, 128, 12)).astype(np.float32)
    dOut = rng.standard_normal((8, 128, 12))
    np.savez_compressed(os.path.join(OUT, "filter_cfg4_n12.npz"),
                        **run_ref_filter(gml, h, b, S, x, dOut, True))


def model_goldens():
    """The reference policy ``DecentralPlannerNet`` (graphs/models/suhaas_model.py) executed end to end on CPU, as
    ``suhaas_agent.py:115-128`` drives it (``model.addGSO(S)``; ``model(inputs, refs, alphas)``; summed MSE loss;
    ``backward``).  Stored: what goes into and comes out of its graph-filter stage ``self.GFL``
    (suhaas_model.py:112-123,182-185) — the only part the drop-in replaces — plus the gradients autograd hands to and
    takes from that stage.  The CNN / MLP weights (2.5 M parameters) are not stored: the stage's input is."""
    Net = ri.decentral_planner_net()
    for tag, nA, B, seed in (("n3", 3, 16, 11), ("n8", 8, 4, 12)):
        torch.manual_seed(seed)
        rng = np.random.default_rng(seed)
        model = Net(nA=nA).double()      # the agent runs the model in double (suhaas_agent.py / forward :169)
        model.device = "cpu"
        model.train()
        frames = load_frames("positionList_expert_%d.npy" % nA, nA)
        idx = rng.choice(len(frames), B, replace=False)
        S = torch.from_numpy(ref_binary(frames[idx], 2).astype(np.float64))          # [B,N,N] as custom_dataset hands it over
        inputs = torch.rand(B, nA, 100, 100, dtype=torch.float64)
        refs = torch.rand(B, nA, 1, dtype=torch.float64)
        alphas = torch.rand(B, nA, 1, dtype=torch.float64)
        actions = torch.randn(B, nA, 2, dtype=torch.float64)
        cap = {}

        def pre_hook(mod, args):
            x = args[0]
            x.retain_grad()
            cap["x"] = x

        def post_hook(mod, args, out):
            out.retain_grad()
            cap["y"] = out

        h1 = model.GFL.register_forward_pre_hook(pre_hook)
        h2 = model.GFL.register_forward_hook(post_hook)
        model.addGSO(S)
        outs = model(inputs, refs, alphas)
        crit = torch.nn.MSELoss()
        loss = crit(outs[0], actions[:, 0])
        for i in range(1, nA):
            loss = loss + crit(outs[i], actions[:, i])
        loss.backward()
        h1.remove(); h2.remove()
        gf = model.GFL[0]
        np.savez_compressed(os.path.join(OUT, "model_gfl_%s.npz" % tag),
                            S=S.numpy().astype(np.float32), x=cap["x"].detach().numpy(),
                            h=gf.weight.detach().numpy(), b=gf.bias.detach().numpy(),
                            y=cap["y"].detach().numpy(), dOut=cap["y"].grad.numpy(),
                            dX=cap["x"].grad.numpy(), dH=gf.weight.grad.numpy(), db=gf.bias.grad.numpy(),
                            loss=float(loss), slope=0.01)


def recurrent_goldens():
    """The reference's recurrent graph-filter layers (graphML.py:2491-2987) executed on CPU over two time steps with
    the hidden state carried (``updateHiddenState``), loss = sum of both outputs against seeded cotangents, backward
    through time.  Stored: inputs, parameters, outputs, the final hidden state and every gradient."""
    gml = ri.graphml()
    g8 = np.load(os.path.join(OUT, "gso_expert8.npz"))
    for tag, cls, (G, H, F, K, N, B), seed in (
            ("rnn_n8", "GraphFilterRNNBatch", (32, 32, 16, 3, 8, 6), 21),
            ("rnn_nin", "GraphFilterRNNBatch", (8, 16, 16, 2, 8, 3), 22),
            ("mornn_n16", "GraphFilterMoRNNBatch", (8, 16, 16, 2, 16, 4), 23),
            ("l2share_n16", "GraphFilterL2ShareBatch", (8, 16, 16, 2, 16, 4), 24)):
        torch.manual_seed(seed)
        rng = np.random.default_rng(seed)
        m = getattr(gml, cls)(G, H, F, K)
        if N == 8:
            S = g8["adj_le"][5:5 + B].astype(np.float32)[:, None]
        else:
            A = (rng.random((B, N, N)) < 0.25).astype(np.float32)
            A = np.triu(A, 1); S = (A + A.transpose(0, 2, 1))[:, None]
        Nin = N - 2 if tag == "rnn_nin" else N
        xs = [rng.standard_normal((B, G, Nin)).astype(np.float32) for _ in range(2)]
        dOuts = [rng.standard_normal((B, F, Nin)) for _ in range(2)]
        h0 = rng.standard_normal((B, H, N)).astype(np.float32)
        m.addGSO(torch.from_numpy(S))
        h0t = torch.from_numpy(h0).double().requires_grad_(True)
        xts = [torch.from_numpy(x).clone().requires_grad_(True) for x in xs]
        m.updateHiddenState(h0t)
        loss = 0
        ys = []
        for xt, dO in zip(xts, dOuts):
            y = m(xt)
            ys.append(y)
            loss = loss + (y * torch.from_numpy(dO).to(y.dtype)).sum()
        loss.backward()
        out = dict(S=S, h0=h0, x0=xs[0], x1=xs[1], dOut0=dOuts[0], dOut1=dOuts[1],
                   y0=ys[0].detach().numpy(), y1=ys[1].detach().numpy(), hT=m.hiddenState.detach().numpy(),
                   dx0=xts[0].grad.numpy(), dx1=xts[1].grad.numpy(), dh0=h0t.grad.numpy(),
                   dims=np.array([G, H, F, K, N, B, Nin]))
        for n, p in m.named_parameters():
            out["p_" + n] = p.detach().numpy()
            out["g_" + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(OUT, "recurrent_%s.npz" % tag), **out)


def rollout_golden():
    """The reference's per-step inference pattern (scene.py:385-394 -> robot.py:654 -> suhaas_agent.py:30-57): at every
    simulation step EVERY robot rebuilds the adjacency with ``Scene.readADjMatrix`` and runs the policy at batch 1,
    keeping only its own column of the output.  Executed here for the graph-filter stack (two reference
    ``GraphFilterBatch`` + ``LeakyReLU`` layers, the GFL of suhaas_model.py:112-123 with L = 2) on recorded 12- and
    8-robot frames; expected[t, :, i] is robot i's own result at step t."""
    gml = ri.graphml()
    for tag, nA, fname, T, dims, seed in (("n12", 12, "positionList_expert_12_longer.npy", 6, (128, 128, 128), 31),
                                          ("n8", 8, "positionList_expert_8.npy", 10, (32, 64, 32), 32)):
        path = os.path.join(ri.REF_ROOT, fname)
        if not os.path.exists(path):
            cands = [f for f in sorted(os.listdir(ri.REF_ROOT)) if f.startswith("positionList") and ("_%d" % nA) in f]
            fname = cands[0]
        frames = load_frames(fname, nA)
        rng = np.random.default_rng(seed)
        idx = np.sort(rng.choice(len(frames), T, replace=False))
        pos = frames[idx]
        assert np.array_equal(pos.astype(np.float32).astype(np.float64), pos)
        torch.manual_seed(seed)
        layers = []
        for l in range(len(dims) - 1):
            layers += [gml.GraphFilterBatch(dims[l], dims[l + 1], 3, 1, True), torch.nn.LeakyReLU(inplace=True)]
        gfl = torch.nn.Sequential(*layers)
        x = rng.standard_normal((T, dims[0], nA)).astype(np.float32)
        exp = np.zeros((T, dims[-1], nA))
        with torch.no_grad():
            for t_ in range(T):
                for i in range(nA):                       # every robot: its own GSO build + its own batch-1 forward
                    S = ri.scene_read_adj(pos[t_].tolist(), 2).reshape(1, 1, nA, nA)
                    St = torch.from_numpy(np.array(S))
                    for l in range(len(dims) - 1):
                        gfl[2 * l].addGSO(St)
                    out = gfl(torch.from_numpy(x[t_:t_ + 1]).double())
                    exp[t_, :, i] = out[0, :, i].numpy()
        out = dict(pos=pos.astype(np.float32), x=x, expected=exp, radius=2.0, dims=np.array(dims), source=fname)
        for l in range(len(dims) - 1):
            out["h%d" % l] = gfl[2 * l].weight.detach().numpy()
            out["b%d" % l] = gfl[2 * l].bias.detach().numpy()
        np.savez_compressed(os.path.join(OUT, "rollout_%s.npz" % tag), **out)


def model_param_layout():
    """(name, shape) of every parameter of the reference policy (2 584 034 parameters, suhaas_model.py:53-143), in
    registration order: the layout the data-parallel gradient buckets are tested with."""
    import json
    Net = ri.decentral_planner_net()
    model = Net(nA=3)
    lay = [[n, list(p.shape)] for n, p in model.named_parameters()]
    assert sum(int(np.prod(s)) for _, s in lay) == 2584034
    json.dump(lay, open(os.path.join(OUT, "model_param_layout.json"), "w"))


if __name__ == "__main__":
    assert ri.available(), "set GFC_REFERENCE_ROOT to a checkout of the original project"
    os.makedirs(OUT, exist_ok=True)
    gso_goldens()
    filter_goldens()
    same_gso_goldens()
    batch_gso_goldens()
    relu_golden()
    model_goldens()
    recurrent_goldens()
    rollout_golden()
    model_param_layout()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
