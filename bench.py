#!/usr/bin/env python
"""bench.py — agent-graphs/s of the fused GSO-build + K-hop graph filter, forward +
backward, on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --steps K --warmup W     # reference CPU path (oracle port)
    torchrun ... bench.py --gpus N ...                        # one rank per GPU, weak scaling

One "step" = one pass of the hot path over ONE batch of the workload: positions ->
GSO (rebuilt on chip), filter forward (+bias, LeakyReLU), filter backward (dX, dH,
db) from a resident synthetic upstream gradient, deterministic gradient reduction,
and — for N > 1 — the all-reduce of the flat [dH | db] bucket, fused into the gradient-reduction kernel as a one-shot
exchange over NVLink peer memory (`--nccl`: separate reduction kernel + ncclAllReduce).

Timing: CUDA events on the launching stream around exactly K steps, barrier +
synchronize on both sides, max over ranks.  Inputs rotate through a ring of
distinct batches larger than L2 (or a single batch that is itself > L2); the K steps are replayed from CUDA
graphs of several ring passes each, so the host enqueues far ahead of the device.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "agent-graphs/sec fwd+bwd (GSO build+K-hop filter)"
L2_BYTES = 126 * 1024 * 1024

# BASELINE.json configs -> concrete synthetic inputs (SURVEY §8d)
WORKLOADS = {
    "cfg1": dict(desc="cfg1: 3-robot expert fixture shape, GraphFilterBatch K=3 128->128, batch 64",
                 B=64, N=3, G=128, F=128, K=3, box=4.0, seed=0, mode="binary_le", train=True),
    "cfg2": dict(desc="cfg2: 8-robot formation policy, K=3, F=32->32, synthetic random-geometric graphs, "
                      "batch 4096 graphs", B=4096, N=8, G=32, F=32, K=3, box=5.0, seed=1,
                 mode="binary_le", train=True),
    "cfg2_x64": dict(desc="cfg2 shapes, 64 batches of 4096 graphs per launch (steady-state rate of the same kernels)",
                     B=262144, N=8, G=32, F=32, K=3, box=5.0, seed=1, mode="binary_le", train=True),
    "cfg3": dict(desc="cfg3: 64-agent synthetic swarm, K=4, F=128->128, batch 65536 graphs",
                 B=65536, N=64, G=128, F=128, K=4, box=10.0, seed=2, mode="binary_le", train=True),
    # the SAME kernels as cfg3 with one fp16 plane per operand (1 MMA per product instead of 3): NOT the parity mode — opt-in,
    # stated bound 2e-3 (tests/test_gpu_parity.py::test_f16_single_plane_mode_has_the_stated_bound).  Reported beside cfg3
    # (SURVEY 8d: "state this next to the numbers") to show the kernels' rate when the fp32 split is not required.
    "cfg3_f16": dict(desc="cfg3 shapes in the opt-in single-fp16-plane mode (GFC_PREC_F16, bound 2e-3; not the parity mode)",
                     B=65536, N=64, G=128, F=128, K=4, box=10.0, seed=2, mode="binary_le", train=True, prec="f16"),
    "cfg4": dict(desc="cfg4: rollout inference, 16384 parallel 12-robot swarms, per-step GSO rebuild + "
                      "2-layer graph filter 128->128->128, K=3", B=16384, N=12, G=128, F=128, K=3, box=6.0,
                 seed=3, mode="binary_le", train=False, layers=2),
}
# cfg5 goes through the CSR entry points (kernel (d)): radius graph with ~16 neighbours (L = 28.3 at R = 2)
CFG5 = dict(desc="cfg5: 1024-agent sparse swarm (radius graph, ~16 neighbours), K=5, F=32->32, CSR SpMM diffusion, "
                 "batch 256 graphs", B=256, N=1024, G=32, F=32, K=5, box=28.3, seed=4, mode="binary_le", train=True, cpu_sample=8)
RADIUS = 2.0
SLOPE = 0.01


def bytes_per_graph(w):
    """algorithmic HBM bytes per graph (SURVEY §8d): positions + x + y (+ dY, dX, activation mask)."""
    N, G, F = w["N"], w["G"], w["F"]
    fwd = 8 * N + 4 * G * N + 4 * F * N
    if not w["train"]:
        return dict(fwd=fwd, bwd=0, total=fwd)
    bwd = 8 * N + 4 * G * N + 4 * F * N + 4 * G * N + 4 * F * N   # pos, x, dY, dX, y (activation mask)
    return dict(fwd=fwd, bwd=bwd, total=fwd + bwd)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the measured section (profiling guide)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)),
                    samples=len(sm), reasons=sorted(reasons))


# ----------------------------------------------------------------------------- inputs
def make_positions(B, N, box, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((B, N, 2)) * box).astype(np.float32)


def make_taps(G, F, K, seed):
    rng = np.random.default_rng(seed)
    s = 1.0 / np.sqrt(G * K)   # reset_parameters law, graphML.py:2442-2447
    return (rng.uniform(-s, s, (F, 1, K, G)).astype(np.float32), rng.uniform(-s, s, (F,)).astype(np.float32))


# ----------------------------------------------------------------------------- our arm
class HotPath:
    """ring of resident batches + direct C-ABI calls (no autograd) for the device-timed loop"""

    def __init__(self, w, dev, ring):
        import torch
        import gnnfc
        self.torch, self.C, self.w, self.dev = torch, gnnfc._cabi, w, dev
        C = self.C
        B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
        self.ring = ring
        gen = torch.Generator(device=dev).manual_seed(w["seed"])
        self.pos = [torch.from_numpy(make_positions(B, N, w["box"], w["seed"] + 17 * i)).to(dev) for i in range(ring)]
        self.x = [torch.randn(B, G, N, device=dev, generator=gen) for _ in range(ring)]
        self.y = [torch.empty(B, N, F, device=dev) for _ in range(ring)]
        h, b = make_taps(G, F, K, w["seed"])
        self.h, self.b = torch.from_numpy(h).to(dev), torch.from_numpy(b).to(dev)
        self.mode = C.GSO_MODES[w["mode"]]
        self.train = w["train"]
        self.layers = w.get("layers", 1)
        self.prec = C.PRECISIONS[w.get("prec", "fp32")]   # every config runs the fp32-parity mode unless it names another
        nbf = C.lib.gfc_filter_workspace_bytes(B, N, G, F, K, 1, 0)
        self.wsf = torch.empty(max(nbf, 256), dtype=torch.uint8, device=dev); self.nbf = nbf
        # operand statistics handed from each batch's forward call to its backward call (gfc_use_stats)
        self.stats = [torch.zeros(4, device=dev) for _ in range(ring)]
        if self.train:
            self.dY = [torch.randn(B, N, F, device=dev, generator=gen) for _ in range(ring)]
            self.dX = [torch.empty(B, G, N, device=dev) for _ in range(ring)]
            self.grads = torch.zeros(F * K * G + F, device=dev)       # flat bucket [dH | db]
            self.dH, self.db = self.grads[:F * K * G], self.grads[F * K * G:]
            nbb = C.lib.gfc_filter_workspace_bytes(B, N, G, F, K, 1, 1)
            self.wsb = torch.empty(max(nbb, 256), dtype=torch.uint8, device=dev); self.nbb = nbb
        if self.layers == 2:
            self.h2, self.b2 = self.h.clone(), self.b.clone()
            self.y2 = [torch.empty(B, N, F, device=dev) for _ in range(ring)]
            self.xt = torch.empty(B, F, N, device=dev)
        self.launches_per_step = 0
        # activation mask handed from each batch's forward call to its backward call (gfc_use_mask): the tcgen05 backward
        # kernels then read 1 bit per output element instead of y
        nbm = C.lib.gfc_filter_mask_bytes(B, N, G, F, K) if self.train else 0
        self.masks = [torch.empty(nbm // 4, dtype=torch.int32, device=dev) for _ in range(ring)] if nbm else None
        self.mask_ok = [False] * ring
        # the hand-over only exists on the tcgen05 wide path (elsewhere it would just add a 16-byte memset to the step)
        self.use_stats = G in (64, 128) and F in (64, 128) and N <= 128

    def stream(self):
        return self.C.ct.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def fwd(self, i, st):
        C, w = self.C, self.w
        B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
        if self.train and self.use_stats:
            C.lib.gfc_use_stats(C.ptr(self.stats[i]))
        if self.masks is not None:
            C.check(C.lib.gfc_use_mask(C.ptr(self.masks[i]), self.masks[i].numel() * 4), "gfc_use_mask")
        C.check(C.lib.gfc_filter_fwd_pos(C.ptr(self.x[i]), C.ptr(self.pos[i]), RADIUS, self.mode, C.ptr(self.h),
                                         C.ptr(self.b), C.ptr(self.y[i]), B, N, G, F, K, C.ACT_LEAKY_RELU, SLOPE,
                                         self.prec, C.ptr(self.wsf), self.nbf, st), "gfc_filter_fwd_pos")
        n = C.last_launch_count()
        if self.masks is not None:
            self.mask_ok[i] = bool(C.lib.gfc_mask_filled())
        if self.layers == 2:
            # layer 2 consumes layer 1's node-major output in place (the reference hands the next GraphFilterBatch
            # a [B,F,N] view over exactly this memory, graphML.py:2362): no transposing copy between the layers
            C.check(C.lib.gfc_filter_fwd_pos_nm(C.ptr(self.y[i]), C.ptr(self.pos[i]), RADIUS, self.mode,
                                                C.ptr(self.h2), C.ptr(self.b2), C.ptr(self.y2[i]), B, N, G, F, K,
                                                C.ACT_LEAKY_RELU, SLOPE, self.prec, C.ptr(self.wsf),
                                                self.nbf, st), "gfc_filter_fwd_pos_nm")
            n += C.last_launch_count()
        return n

    def offer_mask(self, i):
        if self.masks is not None and self.mask_ok[i]:
            self.C.check(self.C.lib.gfc_use_mask(self.C.ptr(self.masks[i]), self.masks[i].numel() * 4), "gfc_use_mask")

    def bwd(self, i, st):
        C, w = self.C, self.w
        B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
        if self.use_stats:
            C.lib.gfc_use_stats(C.ptr(self.stats[i]))
        self.offer_mask(i)
        C.check(C.lib.gfc_filter_bwd_pos(C.ptr(self.x[i]), C.ptr(self.pos[i]), RADIUS, self.mode, C.ptr(self.h),
                                         C.ptr(self.y[i]), C.ptr(self.dY[i]), C.ptr(self.dX[i]), C.ptr(self.dH),
                                         C.ptr(self.db), B, N, G, F, K, C.ACT_LEAKY_RELU, SLOPE,
                                         self.prec, C.ptr(self.wsb), self.nbb, st), "gfc_filter_bwd_pos")
        return C.last_launch_count()

    def enable_peer_exchange(self, px):
        """data-parallel: the backward's second-stage reduction becomes the fused reduce + one-shot all-reduce
        over NVLink peer memory (gfc_filter_bwd_pos_dp) instead of reduce kernel + NCCL all-reduce"""
        self.px = px

    def bwd_dp(self, i, st):
        C, w, px = self.C, self.w, self.px
        B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
        if self.use_stats:
            C.lib.gfc_use_stats(C.ptr(self.stats[i]))
        self.offer_mask(i)
        C.check(C.lib.gfc_filter_bwd_pos_dp(C.ptr(self.x[i]), C.ptr(self.pos[i]), RADIUS, self.mode, C.ptr(self.h),
                                            C.ptr(self.y[i]), C.ptr(self.dY[i]), C.ptr(self.dX[i]), C.ptr(self.grads),
                                            B, N, G, F, K, C.ACT_LEAKY_RELU, SLOPE, self.prec,
                                            C.ptr(self.wsb), self.nbb, px.buf_ptrs, px.sig_ptrs, px.rank, px.world,
                                            1.0, st), "gfc_filter_bwd_pos_dp")
        return C.last_launch_count()

    def step(self, i):
        st = self.stream()
        n = self.fwd(i, st)
        if self.train:
            n += self.bwd_dp(i, st) if getattr(self, "px", None) is not None else self.bwd(i, st)
        self.launches_per_step = n
        return n


def tensor_flops_per_graph(w):
    """fp16 tensor-core flops ISSUED per graph by the tcgen05 wide path (fp32 accuracy costs 3 fp16 MMAs per tap
    product — hi hi + hi lo + lo hi — and 2 per hop product, the 0/1 hop matrix being exact in one plane; 128-row tiles of
    floor(128/N) graphs, block-diagonal hop matrix) and the algorithmic fp32-equivalent flops of SURVEY §8d, forward
    (+ backward when training)."""
    N, G, F, K = w["N"], w["G"], w["F"], w["K"]
    gpc = max(1, 128 // N)
    single = w.get("prec", "fp32") != "fp32" and G == 128 and F == 128 and K <= 5   # opt-in single fp16 plane (GFC_PREC_F16)
    taps = 2 * 128 * (K * G) * F * (1 if single else 3) / gpc                  # per graph share of a tile
    hops = (K - 1) * 2 * 128 * (((gpc * N + 15) // 16) * 16) * G * (1 if single else 2) / gpc
    issued_fwd = taps + hops
    useful_fwd = 2 * (K - 1) * G * N * N + 2 * N * K * G * F
    layers = w.get("layers", 1)
    if not w["train"]:
        return issued_fwd * layers, useful_fwd * layers
    # backward: dX kernel = forward with the roles swapped; dH kernel = the same MMA volume again
    useful_bwd = useful_fwd + 2 * N * K * G * F + (K - 1) * 2 * G * N * N
    return 3 * issued_fwd, useful_fwd + useful_bwd


def ring_size(w):
    per = w["B"] * bytes_per_graph(w)["total"]
    if per >= 2 * L2_BYTES:
        return 2 if per < 8e9 else 1
    return int(min(64, max(2, -(-2 * L2_BYTES // per))))


def timed_steps(torch, hp, steps, warmup, world, dist, use_graph):
    """W warm-up + exactly K timed steps; returns ms for the K steps (this rank)."""
    ring = hp.ring
    allreduce = world > 1 and hp.train and getattr(hp, "px", None) is None   # NCCL only without the fused exchange

    def one(i):
        hp.step(i % ring)
        if allreduce:
            dist.all_reduce(hp.grads)

    for s in range(max(warmup, 1)):
        one(s)
    torch.cuda.synchronize()
    graphs = None
    if use_graph:
        # capture the whole ring once (ring consecutive steps, incl. the all-reduce for N > 1) plus
        # single-step graphs for the remainder; if NCCL refuses capture fall back to the python loop
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for s in range(ring):
                    one(s)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            # one graph = several passes over the ring (about a millisecond of GPU work per replay, so the host
            # enqueues far ahead of the device even with the clock sampler running); the remainder is ONE graph
            unit = ring * max(1, min(8, 64 // ring))
            while unit > ring and unit > steps:
                unit -= ring
            gring = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gring):
                for s in range(unit):
                    one(s)
            singles = []
            if steps % unit:
                g1 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g1):
                    for s in range(steps % unit):
                        one(s)
                singles.append(g1)
            graphs = (gring, singles, unit)
            gring.replay()
            torch.cuda.synchronize()
        except Exception as ex:
            if not allreduce:
                raise
            sys.stderr.write("bench: CUDA-graph capture with NCCL failed (%s); python loop\n" % str(ex)[:120])
            graphs = None
            torch.cuda.synchronize()
    hp.graph_used = graphs is not None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if graphs is not None:
        gring, singles, unit = graphs
        for _ in range(steps // unit):
            gring.replay()
        for g1 in singles:
            g1.replay()
    else:
        for s in range(steps):
            one(s)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    return e0.elapsed_time(e1)


DUMP_BYTES = 48 << 20   # --dump-outputs: bytes of the per-graph outputs written (dH and db come on top)


def dump_outputs(hp, steps, out_dir):
    """--dump-outputs: what the last timed step handed back to its caller, as float32 DIR/<name>.npy: y [B,N,F] (the
    last layer's, node-major memory) and, when training, dX [B,G,N], dH [F,1,K,G], db [F].  Where y and dX of the whole
    batch exceed DUMP_BYTES, the same graphs (drawn with a fixed seed) are written on every run."""
    torch, w = hp.torch, hp.w
    i = (steps - 1) % hp.ring                        # ring slot of the last timed step
    per_graph = dict(y=hp.y2[i] if hp.layers == 2 else hp.y[i])
    whole = {}
    if hp.train:
        per_graph["dX"] = hp.dX[i]
        whole = dict(dH=hp.dH.view(w["F"], 1, w["K"], w["G"]), db=hp.db)
    B = w["B"]
    n = min(B, DUMP_BYTES // sum(t[0].numel() * t.element_size() for t in per_graph.values()))
    if n < B:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, n, replace=False))).to(hp.dev)
        per_graph = {k: t.index_select(0, idx) for k, t in per_graph.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in list(per_graph.items()) + list(whole.items()):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def kernel_alone_ms(torch, hp, which, reps):
    """average duration of the dominant kernel launched back to back (graph of `ring` launches,
    rotating batches) — second-stage reductions switched off so only that kernel runs."""
    C = hp.C
    ring = hp.ring
    st_fn = hp.stream
    if which == "bwd":
        C.check(C.lib.gfc_set_option(C.OPT_SKIP_GRAD_REDUCE, 1), "gfc_set_option")
    try:
        call = (lambda i: hp.bwd(i, st_fn())) if which == "bwd" else (lambda i: hp.fwd(i, st_fn()))
        for i in range(ring):
            call(i)
        torch.cuda.synchronize()
        n_launch = call(0)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(ring):
                call(i)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (reps * ring), n_launch
    finally:
        if which == "bwd":
            C.check(C.lib.gfc_set_option(C.OPT_SKIP_GRAD_REDUCE, 0), "gfc_set_option")


def e2e_steps(torch, w, dev, steps, warmup, world, dist, use_graph=True):
    """same metric through the public module API with HOST (pinned) inputs.  Every step copies that
    step's positions + x host->device (copy stream, double-buffered so the copy of step s+1 overlaps
    the compute of step s), runs addPositions + forward + loss + backward through the drop-in
    nn.Module, and reads the loss back to pinned host memory (checked one step later)."""
    import gnnfc
    B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
    nbuf = 4
    hpos = [torch.from_numpy(make_positions(B, N, w["box"], 1000 + i)).pin_memory() for i in range(nbuf)]
    hx = [torch.randn(B, G, N).pin_memory() for _ in range(nbuf)]
    m = gnnfc.GraphFilterBatch(G, F, K, activation="leaky_relu").to(dev)
    dpos = [torch.empty(B, N, 2, device=dev) for _ in range(2)]
    dx = [torch.empty(B, G, N, device=dev) for _ in range(2)]
    hloss = [torch.zeros(1).pin_memory() for _ in range(2)]
    bucket = gnnfc.GradBucket(m.parameters(), average=True) if world > 1 else None
    layers2 = w.get("layers", 1) == 2
    m2 = gnnfc.GraphFilterBatch(F, F, K, activation="leaky_relu").to(dev) if layers2 else None
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream()
    for e in free:
        e.record(main)
    seen = []

    def prefetch(s):
        i = s % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(free[i])
            dpos[i].copy_(hpos[s % nbuf], non_blocking=True)
            dx[i].copy_(hx[s % nbuf], non_blocking=True)
            ready[i].record(copy_stream)

    def compute(s):
        i = s % 2
        main.wait_event(ready[i])
        m.addPositions(dpos[i], RADIUS, w["mode"])
        if w["train"]:
            xin = dx[i].detach().requires_grad_(True)
            m.zero_grad(set_to_none=True)
            y = m(xin)
            loss = y.square().mean()
            loss.backward()
            if bucket is not None:
                bucket.sync_grads()
        else:
            with torch.no_grad():
                y = m(dx[i])
                if layers2:
                    m2.addPositions(dpos[i], RADIUS, w["mode"])
                    y = m2(y)
                loss = y.mean()
        free[i].record(main)
        hloss[i].copy_(loss.detach().reshape(1), non_blocking=True)
        done[i].record(main)

    # The training step (addPositions + forward + loss + backward [+ gradient exchange] + loss read-back) is
    # captured once per device buffer set with torch.cuda.graph — PyTorch's whole-step capture, the way a user
    # removes Python launch overhead from a fixed-shape loop — and replayed; the H2D copies of the next step's
    # inputs stay outside the graphs on the copy stream so that they overlap the current step.
    graphs = None
    if use_graph:
        try:
            xin_static = [dx[i].detach().requires_grad_(True) for i in range(2)]

            def body(i):
                m.addPositions(dpos[i], RADIUS, w["mode"])
                if w["train"]:
                    m.zero_grad(set_to_none=True)
                    xin_static[i].grad = None
                    y = m(xin_static[i])
                    loss = y.square().mean()
                    loss.backward()
                    if bucket is not None:
                        bucket.sync_grads()
                else:
                    with torch.no_grad():
                        y = m(dx[i])
                        if layers2:
                            m2.addPositions(dpos[i], RADIUS, w["mode"])
                            y = m2(y)
                        loss = y.mean()
                hloss[i].copy_(loss.detach().reshape(1), non_blocking=True)

            side = torch.cuda.Stream(device=dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for _ in range(3):
                    body(0); body(1)
            main.wait_stream(side)
            torch.cuda.synchronize()
            graphs = []
            for i in range(2):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    body(i)
                graphs.append(g)
            torch.cuda.synchronize()
        except Exception as ex:
            sys.stderr.write("bench: e2e CUDA-graph capture failed (%s); eager module calls\n" % str(ex)[:160])
            graphs = None
            torch.cuda.synchronize()

    def compute_graphed(s):
        i = s % 2
        main.wait_event(ready[i])
        graphs[i].replay()
        free[i].record(main)
        done[i].record(main)

    step_fn = compute_graphed if graphs is not None else compute

    def run(n):
        prefetch(0)
        for s in range(n):
            if s + 1 < n:
                prefetch(s + 1)
            step_fn(s)
            if s > 0:   # result of the previous step: wait for ITS copy only, step s is already enqueued
                done[(s - 1) % 2].synchronize()
                seen.append(float(hloss[(s - 1) % 2][0]))
        torch.cuda.synchronize()
        seen.append(float(hloss[(n - 1) % 2][0]))

    run(max(warmup, 2))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(steps)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    h2d = hpos[0].numel() * 4 + hx[0].numel() * 4
    e2e_steps.graphed = graphs is not None
    return ms, h2d, 4, seen[-1]


def csr_workload(torch, dev, steps=20, cpu_budget=4.0):
    """cfg5 through the public module API: per step CSR build from positions (ONE launch, cell list, sync-free capacity
    mode), SpMM-diffusion forward and backward.  Device-timed with CUDA events; nothing in the step reads the device."""
    import gnnfc
    w = CFG5
    B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
    pos = torch.from_numpy(make_positions(B, N, w["box"], w["seed"])).to(dev)
    gen = torch.Generator(device=dev).manual_seed(w["seed"])
    x = torch.randn(B, G, N, device=dev, generator=gen).requires_grad_(True)
    dY = torch.randn(B, F, N, device=dev, generator=gen)
    m = gnnfc.GraphFilterBatch(G, F, K, activation="leaky_relu").to(dev)

    def step():
        m.addSparseGSO(pos, RADIUS, w["mode"], max_degree=64)
        m.zero_grad(set_to_none=True); x.grad = None
        y = m(x)
        y.backward(dY)
        return m.S

    def timed(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for _ in range(3):
        csr = step()
    # the step has no host round trip (sync-free CSR build), so it can be captured once and replayed like the other configs
    graphed = False
    try:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            csr = step()
        g.replay(); torch.cuda.synchronize()
        ms = timed(g.replay, steps)
        graphed = True
    except Exception as ex:   # capture refused: python loop
        sys.stderr.write("bench: cfg5 CUDA-graph capture failed (%s); python loop\n" % str(ex)[:120])
        torch.cuda.synchronize()
        ms = timed(step, steps)
    csr.check()
    ms_build = timed(lambda: gnnfc.build_csr(pos, RADIUS, w["mode"], max_degree=64), steps)
    with torch.no_grad():
        ms_fwd = timed(lambda: m(x), steps)
    nnz = float(csr.rowptr[:, N].float().mean().item())
    bytes_per_graph = 2 * (4 * (N + 1) + 4 * nnz) + 4 * N * (3 * G + 2 * F)     # SURVEY §8d, CSR read fwd+bwd
    peaks = load_peaks()
    gbps = B * bytes_per_graph / (ms * 1e-3) / 1e9
    rec = dict(workload=w["desc"], value=B / (ms * 1e-3), unit="graphs/s", ms_per_step=ms, steps=steps,
               mean_degree=nnz / N, algorithmic_GBps=gbps,
               roofline=dict(bound="hbm", achieved=gbps, peak=peaks["hbm"], unit="GB/s", frac=gbps / peaks["hbm"],
                             algorithmic_bytes_per_graph=bytes_per_graph, kernel="whole step (build + fwd + bwd)"),
               launch="CUDA graph replay" if graphed else "python loop",
               breakdown_ms=dict(csr_build_python_loop=ms_build, forward_python_loop=ms_fwd),
               note="CSR build (one launch, cell list, no host round trip) + one fused forward kernel + one fused backward "
                    "kernel per step (diffusion state in shared memory)")
    try:
        cb, _, _ = time_cpu(w, 20, 1, budget_s=cpu_budget)
        cb["sample"] += " — DENSE GSO: the reference has no sparse path"
        rec["cpu_baseline"] = cb
    except Exception as ex:
        rec["cpu_baseline"] = dict(error=str(ex)[:160])
    return rec


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_reference_step_fn(w, sample_B):
    """the reference's CPU path for one batch: vectorised GSO builder restatement +
    op-faithful GraphFilterBatch port (fp64 inside, as graphML.py:2350) + LeakyReLU + autograd backward."""
    import torch
    from oracle import gso as ogso
    from oracle import lsigf
    N, G, F, K = w["N"], w["G"], w["F"], w["K"]
    pos = make_positions(sample_B, N, w["box"], w["seed"])
    h, b = make_taps(G, F, K, w["seed"])
    ht = torch.from_numpy(h).requires_grad_(True)
    bt = torch.from_numpy(b.reshape(F, 1)).requires_grad_(True)
    x = torch.randn(sample_B, G, N)
    dY = torch.randn(sample_B, F, N, dtype=torch.float64)
    omode = ogso.MODE_BINARY_LE if w["mode"] == "binary_le" else ogso.MODE_SYM_NORM_LT
    layers = w.get("layers", 1)

    def step():
        S, _ = ogso.gso(pos, RADIUS, omode)
        St = torch.from_numpy(S[:, None])
        if w["train"]:
            xt = x.clone().requires_grad_(True)
            ht.grad = None; bt.grad = None
            y = lsigf.activation_torch(lsigf.batch_lsigf_torch(ht, St, xt, bt), lsigf.ACT_LEAKY_RELU)
            y.backward(dY)
            return float(y.detach()[0, 0, 0])
        with torch.no_grad():
            y = lsigf.activation_torch(lsigf.batch_lsigf_torch(ht, St, x, bt), lsigf.ACT_LEAKY_RELU)
            for _ in range(layers - 1):
                y = lsigf.activation_torch(lsigf.batch_lsigf_torch(ht, St, y, bt), lsigf.ACT_LEAKY_RELU)
            return float(y[0, 0, 0])
    return step


def cpu_sample_batch(w):
    """bounded sample: the reference materialises fp64 z = B*K*G*N*8 bytes; keep it <= ~1 GB"""
    z_bytes = w["K"] * w["G"] * w["N"] * 8
    if "cpu_sample" in w:
        return int(w["cpu_sample"])
    return int(max(1, min(w["B"], (1 << 30) // (8 * z_bytes))))


def time_cpu(w, steps, warmup, budget_s):
    import torch
    sb = cpu_sample_batch(w)
    best = None
    ncores = os.cpu_count() or 1
    for threads in sorted({1, ncores}):
        torch.set_num_threads(threads)
        fn = cpu_reference_step_fn(w, sb)
        for _ in range(max(1, warmup)):
            fn()
        t0 = time.perf_counter()
        done = 0
        while done < steps:
            fn(); done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = (time.perf_counter() - t0) / done
        if best is None or dt < best[0]:
            best = (dt, threads, done)
    dt, threads, done = best
    return dict(value=sb / dt, unit="graphs/s", cores=threads, kind="port",
                sample="%d graphs/step x %d steps (%s), best of 1 and %d threads; oracle port of "
                       "graphML.py:2273-2367 + vectorised scene.py:140-154" % (sb, done, w["desc"].split(":")[0], ncores)), dt, sb


# ----------------------------------------------------------------------------- main
def config_dict(w, **more):
    """the keys BOTH arms print (the driver compares them): workload string + shape per GPU"""
    d = dict(workload=w["desc"], B_per_gpu=w["B"], N=w["N"], G=w["G"], F=w["F"], K=w["K"],
             gso="position -> GSO rebuilt every step, radius 2, " + w["mode"], activation="leaky_relu(0.01)",
             train=bool(w["train"]), layers=w.get("layers", 1))
    d.update(more)
    return d


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p.get("bf16_tflops_burst", p.get("bf16_tflops", 1639.5))),
                    tf_sustained=float(p.get("bf16_tflops_sustained", 1375.0)),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1500.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


def kernel_flops(w):
    """algorithmic fp32-equivalent flops per graph of each kernel (SURVEY §8d): dense hops 2(K-1)GN^2, taps 2NKGF"""
    N, G, F, K = w["N"], w["G"], w["F"], w["K"]
    hops_g, hops_f, taps = 2 * (K - 1) * G * N * N, 2 * (K - 1) * F * N * N, 2 * N * K * G * F
    return dict(fwd=hops_g + taps, bwd_dx=hops_f + taps, bwd_dh=hops_g + taps)   # dH kernel: recompute-equivalent hops


def per_kernel_times(torch, hp, reps):
    """average duration of the forward kernel, the dX kernel and the dH/db kernel of ONE batch, each launched back
    to back over the (rotating) ring through the C ABI with the other outputs switched off (NULL dX / NULL dH, db)."""
    C = hp.C
    w = hp.w
    B, N, G, F, K = w["B"], w["N"], w["G"], w["F"], w["K"]
    out = {}

    def bwd_partial(i, st, want_dx, want_dh):
        if hp.use_stats:
            C.lib.gfc_use_stats(C.ptr(hp.stats[i]))   # filled by the forward call of this ring slot during the step
        hp.offer_mask(i)                               # likewise the activation mask
        C.check(C.lib.gfc_filter_bwd_pos(C.ptr(hp.x[i]), C.ptr(hp.pos[i]), RADIUS, hp.mode, C.ptr(hp.h),
                                         C.ptr(hp.y[i]), C.ptr(hp.dY[i]), C.ptr(hp.dX[i]) if want_dx else None,
                                         C.ptr(hp.dH) if want_dh else None, C.ptr(hp.db) if want_dh else None,
                                         B, N, G, F, K, C.ACT_LEAKY_RELU, SLOPE, hp.prec,
                                         C.ptr(hp.wsb), hp.nbb, st), "gfc_filter_bwd_pos")
        return C.last_launch_count()

    calls = dict(fwd=lambda i: hp.fwd(i, hp.stream()))
    if hp.train:
        calls["bwd_dx"] = lambda i: bwd_partial(i, hp.stream(), True, False)
        # the dH / db kernel as it runs inside the step (fed by the dX kernel's dY o act'(y) and batch maximum) = the whole
        # backward call minus the dX-only call; a dH-only call would add a pass over dY and read dY + y instead of one tensor
        calls["bwd_all"] = lambda i: bwd_partial(i, hp.stream(), True, True)
        C.check(C.lib.gfc_set_option(C.OPT_SKIP_GRAD_REDUCE, 1), "gfc_set_option")
    try:
        for name, call in calls.items():
            for i in range(hp.ring):
                call(i)
            torch.cuda.synchronize()
            nl = call(0)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(hp.ring):
                    call(i)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                g.replay()
            e1.record(); torch.cuda.synchronize()
            out[name] = dict(ms=e0.elapsed_time(e1) / (reps * hp.ring), launches=nl)
        if "bwd_all" in out:
            allb = out.pop("bwd_all")
            out["bwd_dh"] = dict(ms=max(allb["ms"] - out["bwd_dx"]["ms"], 1e-6), launches=allb["launches"] - out["bwd_dx"]["launches"],
                                 how="whole backward call minus the dX-only call")
    finally:
        if hp.train:
            C.check(C.lib.gfc_set_option(C.OPT_SKIP_GRAD_REDUCE, 0), "gfc_set_option")
    return out


def roofline_of(torch, w, hp, cfg_name, step_ms, peaks):
    """roofline of the dominant kernel (+ the whole step beside it).  Narrow features (G, F < 64): HBM-bound, the
    dominant kernel is the backward launch.  Wide features: the binding limit in the fp32-parity mode is the tensor
    pipe (SURVEY §8d table), so `bound` = tensor with USEFUL (algorithmic fp32-equivalent) flops as `achieved`;
    the HBM fraction of the same kernel and the issued low-precision flops are given beside it."""
    bpg = bytes_per_graph(w)
    B = w["B"]
    ring = hp.ring
    reps = int(min(2000, max(3, 50e-3 / max(step_ms * 1e-3, 1e-6) / ring)))
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic_tab = json.load(open(tpath))
    wide = w["G"] >= 64 and w["F"] >= 64
    if not wide:
        which = "bwd" if w["train"] else "fwd"
        k_ms, k_launch = kernel_alone_ms(torch, hp, which, reps)
        alg = B * bpg[which]
        ach = alg / (k_ms * 1e-3) / 1e9
        return dict(bound="hbm", achieved=ach, peak=peaks["hbm"], unit="GB/s", frac=ach / peaks["hbm"],
                    traffic=traffic_tab.get("%s:%s" % (cfg_name, which)),
                    kernel=("tc5_n8_bwd_kernel (tcgen05)" if cfg_name.startswith("cfg2") else "%s kernel of %s" % (which, cfg_name)),
                    kernel_ms=k_ms, algorithmic_bytes_per_launch=alg, launches_in_timed_call=k_launch,
                    peak_source=peaks["src"] + " hbm_gbs, burst copy",
                    whole_step=dict(GBps=B * bpg["total"] / (step_ms * 1e-3) / 1e9,
                                    frac=B * bpg["total"] / (step_ms * 1e-3) / 1e9 / peaks["hbm"]),
                    how="CUDA events around a graph of %d back-to-back launches over rotating batches x %d replays" % (ring, reps))
    kt = per_kernel_times(torch, hp, reps)
    fl = kernel_flops(w)
    N, G, F = w["N"], w["G"], w["F"]
    kbytes = dict(fwd=8 * N + 4 * G * N + 4 * F * N, bwd_dx=8 * N + 8 * F * N + 4 * G * N, bwd_dh=8 * N + 4 * F * N + 4 * G * N)
    dom = max(kt, key=lambda k: kt[k]["ms"])
    per = {}
    # fp16 flops the tensor pipe actually executes per graph and kernel (each of the three kernels issues the forward's MMA
    # volume: 128-row block-diagonal hops, 3 / 2 MMAs per tap / hop product in the fp32-parity mode)
    issued_fwd = tensor_flops_per_graph(dict(w, train=False, layers=1))[0]
    for k, v in kt.items():
        tf = B * fl[k] / (v["ms"] * 1e-3) / 1e12
        gb = B * kbytes[k] / (v["ms"] * 1e-3) / 1e9
        itf = B * issued_fwd / (v["ms"] * 1e-3) / 1e12
        per[k] = dict(ms=v["ms"], launches=v["launches"], useful_tflops=tf, tensor_frac=tf / peaks["tf_burst"],
                      issued_fp16_tflops=itf, issued_tensor_frac=itf / peaks["tf_burst"],
                      algorithmic_GBps=gb, hbm_frac=gb / peaks["hbm"])
    names = dict(fwd="tc5_wide_kernel<fwd>", bwd_dx="tc5_wide_kernel<dX>", bwd_dh="tc5_wide_dh_kernel")
    total_fl = sum(fl[k] for k in kt)
    step_tf = B * total_fl / (step_ms * 1e-3) / 1e12
    step_gb = B * bpg["total"] / (step_ms * 1e-3) / 1e9
    return dict(bound="tensor", achieved=per[dom]["useful_tflops"], peak=peaks["tf_burst"], unit="TFLOP/s",
                frac=per[dom]["tensor_frac"], traffic=traffic_tab.get("%s:%s" % (cfg_name, dom)),
                kernel=names[dom], kernel_ms=per[dom]["ms"],
                algorithmic_flops_per_launch=B * fl[dom], algorithmic_bytes_per_launch=B * kbytes[dom],
                hbm=dict(achieved=per[dom]["algorithmic_GBps"], peak=peaks["hbm"], frac=per[dom]["hbm_frac"]),
                per_kernel=per,
                whole_step=dict(useful_tflops=step_tf, tensor_frac=step_tf / peaks["tf_sustained"], GBps=step_gb,
                                hbm_frac=step_gb / peaks["hbm"]),
                issued_over_useful=tensor_flops_per_graph(w)[0] / max(tensor_flops_per_graph(w)[1], 1),
                peak_source=peaks["src"] + ": dense bf16 burst for a kernel timed alone, sustained for the whole step; hbm_gbs",
                note=("achieved = USEFUL flops (SURVEY 8d: dense hops 2(K-1)GN^2 + taps 2NKGF per pass) of the dominant kernel / "
                      "its duration; single fp16 plane per operand: 1 MMA per product, bound 2e-3, NOT the parity mode"
                      if w.get("prec", "fp32") != "fp32" else
                      "achieved = USEFUL fp32-equivalent flops (SURVEY 8d: dense hops 2(K-1)GN^2 + taps 2NKGF per pass) of the "
                      "dominant kernel / its duration; fp32 parity costs 3 half-precision MMAs per tap product (fp16 hi/lo "
                      "split), so at most ~1/3 of the dense peak is reachable in this mode"),
                how="CUDA events around %d back-to-back launches x %d replays per kernel, other outputs switched off" % (ring, reps))


def dp_check(torch, dist, hp, world):
    """N > 1: every rank holds the same data (identical seeds), so the exchanged bucket must equal world x the local
    one, and all ranks must end with bit-identical gradients."""
    i = 0
    st = hp.stream()
    hp.fwd(i, st)
    hp.bwd(i, st)
    local = hp.grads.clone()
    if getattr(hp, "px", None) is not None:
        hp.bwd_dp(i, st)
    else:
        dist.all_reduce(hp.grads)
    torch.cuda.synchronize()
    got = hp.grads.clone()
    den = float((world * local).abs().max())
    err = float((got - world * local).abs().max()) / max(den, 1e-30)
    chk = got.double().sum().reshape(1)
    first = got[:64].clone()
    allc = [torch.empty_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    allf = [torch.empty_like(first) for _ in range(world)]
    dist.all_gather(allf, first)
    same = all(torch.equal(allc[0], c) for c in allc) and all(torch.equal(allf[0], f) for f in allf)
    ok = bool(err <= 1e-6 and same and torch.isfinite(got).all())
    if getattr(hp, "px", None) is not None:
        try:
            hp.px.status()
        except Exception:
            ok = False
    return dict(ok=ok, max_rel_err_vs_world_x_local=err, bit_identical_across_ranks=bool(same))


def side_measurement(torch, dist, name, w2, dev, peaks, cpu_budget):
    hp2 = HotPath(w2, dev, ring_size(w2))
    small = w2["B"] * bytes_per_graph(w2)["total"] < L2_BYTES
    st2 = 400 if small else 20
    ms2 = timed_steps(torch, hp2, st2, 3, 1, dist, True)
    step_ms = ms2 / st2
    rec = dict(workload=w2["desc"], value=w2["B"] * st2 / (ms2 * 1e-3), unit="graphs/s", ms_per_step=step_ms,
               steps=st2, config=config_dict(w2), roofline=roofline_of(torch, w2, hp2, name, step_ms, peaks))
    del hp2
    torch.cuda.empty_cache()
    if "prec" in w2:      # a precision variant of another config: the CPU reference is that config's
        rec["precision"] = w2["prec"]
        rec["cpu_baseline"] = "same workload as cfg3: see the headline's cpu_baseline"
        return rec
    cb, _, _ = time_cpu(w2, 50, 1, budget_s=cpu_budget)
    rec["cpu_baseline"] = cb
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true", help="launch every step from Python (no CUDA graph)")
    ap.add_argument("--nccl", action="store_true", help="N > 1: plain NCCL all-reduce instead of the fused peer exchange")
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements of the other configs")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline work")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one to DIR/<name>.npy (float32; a fixed "
                         "sample of the graphs where the batch is large) so that two builds can be compared")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    w = WORKLOADS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps or 20
        warmup = args.warmup if args.warmup is not None else 3
        cb, dt, sb = time_cpu(w, steps, warmup, budget_s=120.0)
        line = dict(metric=METRIC, value=cb["value"], unit="graphs/s", n_gpus=args.gpus, steps=steps, warmup=warmup,
                    ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                    data="synthetic", impl="reference", config=config_dict(w),
                    cpu_baseline=cb, gpu_launches=0,
                    e2e=dict(value=cb["value"], unit="graphs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    small = w["B"] * bytes_per_graph(w)["total"] < L2_BYTES
    steps = args.steps or (4000 if small else 20)
    warmup = args.warmup if args.warmup is not None else 5
    warmup = max(warmup, 3)
    peaks = load_peaks()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ring = ring_size(w)
    hp = HotPath(w, dev, ring)
    collective = "none"
    if world > 1 and w["train"]:
        collective = "NCCL all-reduce of the flat [dH|db] bucket every step"
        if not args.nccl:
            try:
                import gnnfc
                hp.enable_peer_exchange(gnnfc.PeerExchange(hp.grads.numel(), dev))
                collective = ("fused into the gradient-reduction kernel: one-shot all-reduce of the flat [dH|db] bucket "
                              "over NVLink peer memory (symmetric memory, P2P stores of {value, epoch} words)")
            except Exception as ex:   # symmetric memory unavailable on this box: the NCCL collective still is
                sys.stderr.write("bench: peer exchange unavailable (%s); using NCCL\n" % str(ex)[:160])
    use_graph = not args.no_graph
    ms = timed_steps(torch, hp, steps, warmup, world, dist, use_graph)
    launches = hp.launches_per_step * steps
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * w["B"] * steps / (ms_max * 1e-3)
    clocks = sampler.stop() if rank == 0 else None   # sampled over warm-up + the timed region of the headline
    if args.dump_outputs and rank == 0:
        dump_outputs(hp, steps, args.dump_outputs)

    dpc = dp_check(torch, dist, hp, world) if (world > 1 and w["train"]) else None

    bpg = bytes_per_graph(w)
    roofline = roofline_of(torch, w, hp, args.config, ms_max / steps, peaks)
    del hp
    torch.cuda.empty_cache()

    # end-to-end through the module API with host buffers
    e2e_n = max(3, min(steps, 200 if small else 10))
    e_ms, h2d, d2h, _ = e2e_steps(torch, w, dev, e2e_n, 3, world, dist, use_graph)
    te = torch.tensor([e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = dict(value=world * w["B"] * e2e_n / (float(te.item()) * 1e-3), unit="graphs/s",
               h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, steps=e2e_n,
               api="gnnfc.GraphFilterBatch.addPositions/forward + loss.backward%s; pinned host inputs, H2D double-buffered "
                   "on a copy stream every step, loss copied to pinned host every step and read by the host"
                   % (" captured once with torch.cuda.graph and replayed" if getattr(e2e_steps, "graphed", False) else ""))
    torch.cuda.empty_cache()

    extra = {}
    if rank == 0 and world == 1 and not args.no_extra:
        for name in ("cfg2", "cfg2_x64", "cfg3", "cfg3_f16", "cfg4", "cfg1"):
            if name == args.config:
                continue
            try:
                extra[name] = side_measurement(torch, dist, name, WORKLOADS[name], dev, peaks, 4.0)
            except Exception as ex:  # side measurement must never break the headline line
                extra[name] = dict(error=str(ex)[:200])
        try:
            extra["cfg5"] = csr_workload(torch, dev, cpu_budget=4.0)
        except Exception as ex:
            extra["cfg5"] = dict(error=str(ex)[:200])

    cpu = None
    if rank == 0 and world == 1:
        cpu, _, _ = time_cpu(w, 50, 1, budget_s=args.cpu_budget)
    if rank == 0:
        line = dict(metric=METRIC, value=value, unit="graphs/s", n_gpus=world, steps=steps, warmup=warmup,
                    ms_per_step=ms_max / steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic",
                    config=config_dict(w),
                    details=dict(global_batch=world * w["B"],
                                       precision="fp32-equivalent split products on the tensor cores (fp16 hi/lo or bf16x3 / 3xTF32, "
                                                 "fp32 accumulate), <=1e-5 of the fp64 reference",
                                       upstream_gradient="resident synthetic dY",
                                       l2=("one batch = %.0f MB (> 126 MB L2)" % (w["B"] * bpg["total"] / 1e6)) if ring == 1 else
                                          ("inputs rotate through a ring of %d distinct batches = %.0f MB (> 126 MB L2)"
                                           % (ring, ring * w["B"] * bpg["total"] / 1e6)),
                                       launch="CUDA graph replay" if use_graph else "python loop",
                                       collective=collective),
                    roofline=roofline, cpu_baseline=cpu, e2e=e2e, gpu_launches=launches, clocks=clocks, extra=extra)
        if dpc is not None:
            line["dp_check"] = dpc
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
