#!/usr/bin/env python
"""Contract benchmark: GAT layer fwd+bwd edges/sec at the ogbn-proteins shape.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one forward + backward of the GATConv sparse section (logits -> leaky_relu
-> edge-softmax -> dropout -> SpMM -> scaling; SURVEY.md section 8d) over the whole
synthetic graph; dense fc projections are excluded from `value` (they stay cuBLAS) and
included in `e2e`, which goes through the reference-facing `GATConv.forward(graph,
feat_src, feat_edge)` with HOST input buffers.

N > 1: the same graph is 1-D partitioned on destination rows (strong scaling); every
rank all-gathers the source table halo, runs its rows, and the gradient halo is
reduce-scattered back (bot_b200/partition.py).

--impl reference: the oracle port of the reference math (pure torch, CPU) on a bounded
sample of the same workload, on the host cores of this box (DGL itself is not
installable offline: DESIGN.md).

--dump-outputs DIR: after the timed steps, the results of the last one (the layer output and
the gradients of its inputs) are written as DIR/<name>.npy; the inputs are seeded, so two
builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The contract is ONE JSON line on stdout, but libraries print there too (NCCL's version banner: this image sets
# NCCL_DEBUG=VERSION).  main() points file descriptor 1 at stderr for the whole run; the JSON line goes to the real stdout.
_REAL_STDOUT = None


def claim_stdout():
    """Called by main() only (importing this module for its constants must not touch the caller's stdout)."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    text = json.dumps(line) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, text.encode())


import torch  # noqa: E402

SLOPE = 0.2
# BASELINE.json configs (SURVEY.md section 8 table).  `proteins` is the north-star / headline shape; the others are
# measured with the same code path at their own flags (`--shape`), N=1 and partitioned.
SHAPES = {
    "proteins": dict(n=132534, e=39561252, H=6, D=80, er=True, ee=True, edge_drop=0.1, attn_p=0.0, symm=False, in_feats=480,
                     desc="attn_dst + edge-feature logits (8-dim raw edge feats -> 16-dim edge emb), edge_drop=0.1 (training)",
                     ref="src/ogbn-proteins/gat.py:320-327, models.py:209-221"),
    "products": dict(n=2449029, e=61859140, H=4, D=120, er=True, ee=False, edge_drop=0.1, attn_p=0.0, symm=False, in_feats=480,
                     desc="attn_dst, no edge features, edge_drop=0.1 (training)",
                     ref="src/ogbn-products/gat.py:379-386, models.py:211-223"),
    "reddit": dict(n=232965, e=114615892, H=4, D=64, er=False, ee=False, edge_drop=0.0, attn_p=0.1, symm=True, in_feats=256,
                   desc="source-only logits, symmetric norm, attn_drop=0.1 drawn in-kernel (training)",
                   ref="src/no-sampling/run.py:978, models.py:683-694"),
    "arxiv": dict(n=169343, e=2484941, H=3, D=250, er=False, ee=False, edge_drop=0.0, attn_p=0.1, symm=True, in_feats=750,
                  desc="source-only logits, symmetric norm, attn_drop=0.1 drawn in-kernel (training); too small to shard: "
                       "replicas only", ref="src/no-sampling/run.py:1017"),
}
EDGE_FEATS, EDGE_EMB = 8, 16
# kept for importers (tests): the headline shape
N_NODES, N_EDGES, HEADS, HID = SHAPES["proteins"]["n"], SHAPES["proteins"]["e"], SHAPES["proteins"]["H"], SHAPES["proteins"]["D"]
EDGE_DROP = SHAPES["proteins"]["edge_drop"]


def metric_name(shape):
    return f"GAT layer fwd+bwd edges/sec (ogbn-{shape} shape)" if shape != "reddit" else "GAT layer fwd+bwd edges/sec (Reddit shape)"


METRIC = metric_name("proteins")


def workload_name(shape, n_nodes, n_edges):
    c = SHAPES[shape]
    return (f"{shape}-shape GATConv layer: N={n_nodes} E={n_edges} H={c['H']} D={c['D']} fp32, {c['desc']}, "
            f"uniform random edges ({c['ref']})")


def algorithmic_bytes(E, N_s, N_d, H, D, er=True, ee=True):
    """SURVEY.md section 8(d) gather/streaming model.  Returns (fwd, bwd) bytes per layer pass."""
    R, h = 4 * H * D, 4 * H
    x = (h + 4) if ee else 0
    e_r = 1 if er else 0
    fwd = E * (4 + h + R + x) + N_d * (8 + h * e_r + R + 2 * h)
    bwd = E * ((4 + h + R + x + h) + (8 + 2 * h + R)) + N_d * (8 + 2 * R + 2 * h + 2 * h * e_r) + N_s * (8 + R + h)
    return fwd, bwd


def performed_bytes(E, N_s, N_d, H, D, er=True, ee=True):
    """Bytes of the passes this engine actually performs (DESIGN.md section 4): the forward gather, ONE backward
    gather (the reference's dst-major re-gather for grad_a is eliminated: the dots ride on the src pass) and the
    per-edge record streams.  = forward + the src-pass bracket of SURVEY 8(d) + the node pass."""
    bf, bb = algorithmic_bytes(E, N_s, N_d, H, D, er, ee)
    R, h = 4 * H * D, 4 * H
    x = (h + 4) if ee else 0
    b_dst = E * (4 + h + R + x + h) + N_d * (8 + R + 2 * h + 2 * h)
    return bf, bb - b_dst


# ----------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self, timeout=3.0):
        # nvidia-smi needs a few hundred ms before its first line: do not start the timed region without it
        t = time.time()
        while self.proc is not None and not self.lines and time.time() - t < timeout:
            time.sleep(0.01)
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # the sampler runs from before the warm-up; only samples that arrived inside the timed region count
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        inside = [ln for (t, ln) in self.lines if t0 <= t <= t1]
        window = "timed region"
        if not inside:
            inside, window = [ln for (_, ln) in self.lines], "whole run (no sample fell inside the timed region)"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ----------------------------------------------------------------------------
# synthetic inputs
# ----------------------------------------------------------------------------
def synth_edges(n_nodes, n_edges, device, seed=0, power_law=0.0):
    """SURVEY.md section 8d generator: uniform random COO; power_law > 0 draws dst proportional to rank^-power_law."""
    g = torch.Generator(device=device).manual_seed(seed)
    src = torch.randint(0, n_nodes, (n_edges,), device=device, generator=g)
    if power_law > 0:
        w = torch.arange(1, n_nodes + 1, device=device, dtype=torch.float64) ** (-power_law)
        cdf = torch.cumsum(w / w.sum(), 0)
        u = torch.rand(n_edges, device=device, dtype=torch.float64, generator=g)
        dst = torch.searchsorted(cdf, u).clamp(max=n_nodes - 1)
    else:
        dst = torch.randint(0, n_nodes, (n_edges,), device=device, generator=g)
    return src, dst


# ----------------------------------------------------------------------------
# CPU arm: the oracle port of the reference math on a bounded sample
# ----------------------------------------------------------------------------
def cpu_port_run(shape, steps, warmup, n_edges=None, budget_s=200.0):
    """fwd+bwd of the same layer math, same flags, on the host (oracle port, non-materialising form,
    oracle/gat_ref.py gat_sparse_big_*).  A step processes a uniform edge subsample of the workload over ALL nodes,
    sized so that the whole run stays within ``budget_s``.  Returns dict(value, unit, cores, kind, sample, ms_per_step)."""
    from oracle import gat_ref

    c = SHAPES[shape]
    n, H, D = c["n"], c["H"], c["D"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if n_edges is None:
        # ~0.45 us per edge and step at H*D = 480 on 16 cores (measured: 4.3 s for 9.9 M edges); scale to the budget
        per_edge = 0.45e-6 * (H * D) / 480.0 * (16.0 / max(cores, 1))
        n_edges = int(min(c["e"], max(1_000_000, budget_s / max(steps + warmup, 1) / per_edge)))
    src, dst = synth_edges(n, n_edges, "cpu", seed=0)
    bg = gat_ref.BigGraph(src, dst, n, n)
    g = torch.Generator().manual_seed(1)
    ft = torch.randn(n, H, D, generator=g)
    el = torch.randn(n, H, generator=g)
    er = torch.randn(n, H, generator=g) if c["er"] else None
    ee = torch.randn(n_edges, H, generator=g) if c["ee"] else None
    gout = torch.randn(n, H, D, generator=g)
    cs = ds = None
    if c["symm"]:
        cs = torch.bincount(src, minlength=n).float().clamp(min=1).pow(-0.5)
        ds = torch.bincount(dst, minlength=n).float().clamp(min=1).pow(0.5)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            keep = mul = None
            if c["edge_drop"] > 0:     # models.py:529-532: exactly int(E*p) random edges dropped
                keep = torch.ones(n_edges, dtype=torch.bool)
                keep[torch.randperm(n_edges, generator=g)[: int(n_edges * c["edge_drop"])]] = False
            if c["attn_p"] > 0:        # models.py:537/544: nn.Dropout on the attention
                mul = (torch.rand(n_edges, H, generator=g) >= c["attn_p"]).float() / (1.0 - c["attn_p"])
            out, saved = gat_ref.gat_sparse_big_forward(bg, ft, el, er, ee, SLOPE, keep, mul, cs, ds)
            gat_ref.gat_sparse_big_backward(bg, saved, gout, SLOPE, c["er"], c["ee"], keep, cs, ds)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    frac = n_edges / c["e"]
    return {"value": n_edges / t, "unit": "edges/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"same layer math and flags (edge-drop draw / dropout mask included) on a {n_edges}-edge uniform subsample "
                      f"({frac:.2f} of the workload's edges) over all {n} nodes, fwd+bwd, {len(times)} timed steps, "
                      f"oracle/gat_ref.py gat_sparse_big_* (segment_reduce + per-head sparse CSR matmul), torch {torch.__version__} CPU, "
                      f"{torch.get_num_threads()} threads",
            "ms_per_step": t * 1e3, "edges_per_step": n_edges}


def cora_cpu_reference(steps=20, warmup=3):
    """BASELINE config 1 / SURVEY 8d: the full 2-layer Cora-shape GAT (2,708 nodes, 10,556 raw edges -> self loops,
    1,433 feats, 8 heads x 8, 7 classes, edge_drop 0.5; src/no-sampling/run.py:895) forward + backward on the host,
    restated on the oracle (oracle/modules_ref.py gatconv_v1) — the reference's own CPU-runnable case."""
    from oracle import graph_ref, modules_ref

    torch.set_num_threads(os.cpu_count() or 1)
    n, e, f_in, n_cls, H, D = 2708, 10556, 1433, 7, 8, 8
    src, dst = graph_ref.synthetic_coo(n, e, 0)
    src, dst = graph_ref.add_self_loop(*graph_ref.remove_self_loop(src, dst), n)
    src, dst = torch.from_numpy(src), torch.from_numpy(dst)
    E = src.numel()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, f_in, generator=g)
    sd0 = {"fc.weight": torch.randn(H * D, f_in, generator=g) * 0.05, "attn_l": torch.randn(1, H, D, generator=g) * 0.1,
           "res_fc.weight": torch.randn(H * D, f_in, generator=g) * 0.05}
    sd1 = {"fc.weight": torch.randn(n_cls, H * D, generator=g) * 0.1, "attn_l": torch.randn(1, 1, n_cls, generator=g) * 0.1,
           "res_fc.weight": torch.randn(n_cls, H * D, generator=g) * 0.1}
    params = [t.requires_grad_(True) for sd in (sd0, sd1) for t in sd.values()]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        keeps = []
        for _ in range(2):
            keep = torch.ones(E, dtype=torch.bool)
            keep[torch.randperm(E, generator=g)[: int(E * 0.5)]] = False
            keeps.append(keep)
        h = modules_ref.gatconv_v1(sd0, src, dst, n, n, x, num_heads=H, out_feats=D, keep=keeps[0]).flatten(1)
        h = torch.relu(h)
        out = modules_ref.gatconv_v1(sd1, src, dst, n, n, h, num_heads=1, out_feats=n_cls, keep=keeps[1]).mean(1)
        out.square().mean().backward()
        for p_ in params:
            p_.grad = None
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return {"workload": f"2-layer GAT, Cora shape (N={n}, E={E} with self loops, {f_in} feats, {H}x{D} -> 1x{n_cls}, edge_drop 0.5), "
                        "whole model fwd+bwd on the host (oracle/modules_ref.py over oracle/gat_ref.py), run.py:895",
            "ms_per_step": round(t * 1e3, 3), "edges_per_s": 2 * E / t, "cores": torch.get_num_threads(), "kind": "port"}


def common_config(shape, n_nodes, n_edges, world):
    """`config` of the JSON line — identical for both arms (the driver compares them)."""
    par = "single GPU" if world == 1 else (f"1-D dst-row partition x{world}, halo all-gather + gradient reduce-scatter over NVLink (peer-memory pulls or NCCL: `graph.halo_exchange`)"
                                           if shape != "arxiv" else f"{world} independent replicas (too small to shard)")
    return {"workload": workload_name(shape, n_nodes, n_edges), "shape": shape,
            "l2": "inputs_exceed_l2 (no flush between iterations: the per-step working set is >= 20x the 126 MB L2)",
            "parallelism": par,
            "timed": "edge-drop mask draw (exactly int(E*p) edges) + per-edge operand staging + fused fwd + bwd (node / src / "
                     "edge passes); per-edge operands are resident in the graph's canonical edge order (what the layer's own "
                     "edge-logit kernels emit from canonically stored edata); no instrumentation inside the timed region"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_port_run(args.shape, args.steps, max(args.warmup, 1))
    c = SHAPES[args.shape]
    line = {
        "impl": "reference", "metric": metric_name(args.shape), "value": r["value"], "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(args.shape, c["n"], c["e"], int(os.environ.get("WORLD_SIZE", "1"))),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------
def pin_to_gpu_numa(local_rank, world):
    """Multi-GPU runs: bind this rank's threads to the CPUs NVML reports as local to its GPU BEFORE any pinned host
    buffer is allocated (first touch puts the pages on that NUMA node), so that every rank's H2D stream stays on its own
    socket / PCIe root (round 1: the end-to-end leg did not scale from 2 to 4 GPUs).  Only narrows the set the process is
    already allowed to run on; any failure leaves the affinity untouched.  Returns what was done, for the JSON line."""
    if world <= 1 or os.environ.get("BOTGAT_NO_PIN") == "1" or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local_rank
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                idx = int(ids[local_rank])
        handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpu + 63) // 64)
        local = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        want = sorted(local & allowed)
        # several ranks may share one socket: leave each its share of that socket's allowed CPUs
        if len(want) >= 2:
            os.sched_setaffinity(0, want)
            return {"gpu": idx, "cpus": len(want), "of_allowed": len(allowed)}
        return {"gpu": idx, "cpus": 0, "of_allowed": len(allowed), "note": "no allowed CPU is local to this GPU: affinity unchanged"}
    except Exception as ex:   # NVML missing / restricted container: not an error for the benchmark
        return {"error": repr(ex)[:120]}


def run_ours(args):
    import torch.distributed as dist

    import bot_b200
    from bot_b200 import _lib, functional
    from bot_b200.functional import gat_fused

    shape = args.shape
    c = SHAPES[shape]
    H, D = c["H"], c["D"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl ours) needs a CUDA device: bot_b200 has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the results of one process: run it without torch.distributed")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_affinity = pin_to_gpu_numa(local_rank, world)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    replicas = world > 1 and shape == "arxiv"     # too small to shard: N independent replicas, no collective

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_nodes, n_edges = args.nodes or c["n"], args.edges or c["e"]
    src, dst = synth_edges(n_nodes, n_edges, dev, seed=0 if not replicas else rank)
    gen = torch.Generator(device=dev).manual_seed(1)

    layer = None
    if world == 1 or replicas:
        graph = bot_b200.Graph(src, dst, n_nodes)
        graph.create_formats_()
    else:
        from bot_b200 import partition

        layer = partition.PartitionedGraph(src, dst, n_nodes)
        graph = layer.local
        graph.create_formats_()
    full_src, full_dst = (src, dst) if (world == 1 and not args.no_parity) else (None, None)
    cs_l = ds_l = cs_own = None
    if c["symm"]:   # clamp(out_deg,1)^-0.5 on the gathered rows, clamp(in_deg,1)^+0.5 on the outputs (models.py:500-505, 550-555)
        if layer is None:
            cs_l, ds_l = graph.deg_scale("out", -0.5), graph.deg_scale("in", 0.5)
        else:
            cs_full = torch.bincount(src, minlength=n_nodes).float().clamp(min=1).pow(-0.5)
            ds_full = torch.bincount(dst, minlength=n_nodes).float().clamp(min=1).pow(0.5)
            cs_own = layer.owned_slice(cs_full).contiguous()
            with torch.no_grad():
                cs_l = layer.halo_gather(cs_own).contiguous()
            ds_l = layer.owned_slice(ds_full).contiguous()
            del cs_full, ds_full
    del src, dst
    E_local = graph.number_of_edges()
    n_src_l, n_dst_l = graph.number_of_src_nodes(), graph.number_of_dst_nodes()
    info = graph._info

    # ---------------- device-resident leg (value) ----------------
    n_own = n_dst_l if layer is not None else n_nodes
    if layer is not None and layer.plan == "dense" and layer.exchange in ("p2p", "auto") and layer._p2p_usable(H, D, 0):
        # the projected rows are produced straight into this rank's slice of the peer-memory exchange table
        hx = layer.halo_buffers(H, D)
        with torch.no_grad():
            hx.own_ft.normal_(generator=gen)
            hx.own_el.normal_(generator=gen)
        ft_own, el_own = hx.own_ft.detach().requires_grad_(True), hx.own_el.detach().requires_grad_(True)
    else:
        ft_own = torch.randn(n_own, H, D, device=dev, generator=gen).requires_grad_(True)
        el_own = torch.randn(n_own, H, device=dev, generator=gen).requires_grad_(True)
    er = torch.randn(n_dst_l, H, device=dev, generator=gen).requires_grad_(True) if c["er"] else None
    # edge logits as the layer's own producers emit them: one 32-byte record per edge (E, pad_heads(H)), in the graph's
    # CANONICAL edge order (static edata is stored canonically, bot_b200.graph.EdgeFrame)
    ee = torch.randn(E_local, functional.pad_heads(H), device=dev, generator=gen).requires_grad_(True) if c["ee"] else None
    gout = torch.randn(n_dst_l, H, D, device=dev, generator=gen)
    leaves = [t for t in (ft_own, el_own, er, ee) if t is not None]

    seeds = iter(range(1, 1 << 30))

    def step_resident(keep_grads=False, seed=None):
        sd = next(seeds) if seed is None else seed
        # the reference's draw: exactly int(E * p) uniformly random edges dropped (models.py:136-139 / 528-532)
        keep = functional.edge_drop_keep(E_local, int(E_local * c["edge_drop"]), sd, dev) if c["edge_drop"] > 0 else None
        if layer is None:
            out = gat_fused(graph, ft_own, el_own, er, ee, keep, None, cs_l, ds_l, SLOPE, c["attn_p"], sd, edge_order="canonical")
        else:
            out = layer.gat(ft_own, el_own, er, ee, keep, None, cs_l, ds_l, SLOPE, c["attn_p"], sd, edge_order="canonical")
        out.backward(gout)
        if keep_grads:
            return out.detach(), keep
        for t in leaves:
            t.grad = None

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    launches0 = lib.botgat_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark_begin()
    barrier()
    e0.record()
    for i in range(args.steps):
        last = step_resident(keep_grads=bool(args.dump_outputs) and i == args.steps - 1)
    e1.record()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.botgat_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    total_edges = n_edges * (world if replicas else 1)
    value = total_edges / (ms_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": last[0], "grad_ft": ft_own.grad, "grad_el": el_own.grad,
                                         "grad_er": None if er is None else er.grad}, {"grad_ee": None if ee is None else ee.grad})
        del last
        for t in leaves:
            t.grad = None

    # per-kernel durations: a SECOND, instrumented pass of the same steps (CUDA events around every ABI call, the backward
    # issued as three calls) — outside the headline's timed region
    kt = functional.KernelTimer()
    functional.timer = kt
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        step_resident()
    e1.record()
    torch.cuda.synchronize()
    functional.timer = None
    ms_instr = e0.elapsed_time(e1)
    ktot = kt.totals()

    # ---------------- roofline of the dominant kernel ----------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, hbm_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        hbm_peak, hbm_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md); MEASURED_PEAKS.json absent"
    l2_peak = None
    l2path = os.path.join(ROOT, "profiles", "l2_peak.json")
    if os.path.exists(l2path):
        l2_peak = float(json.load(open(l2path))["l2_read_gbs"])
    bf, b_src = performed_bytes(E_local, n_src_l, n_dst_l, H, D, c["er"], c["ee"])
    alg = {"gat_fwd": bf, "gat_bwd_src": b_src}
    # the gathers are served by the L2 when one head's (N x D) slab of the gathered table fits it (DESIGN.md section 3):
    # then the L2 -> SM bandwidth is the bound that applies; otherwise (products) the rows come from DRAM
    slab_mb = max(n_src_l, n_dst_l) * D * 4 / 2**20
    l2_bound = l2_peak is not None and slab_mb <= 64.0
    kernels = {}
    for name, (n, tot) in ktot.items():
        avg = tot / n
        k = {"launches": n, "avg_ms": round(avg, 4), "share_of_instrumented_step": round(tot / ms_instr, 4)}
        if name in alg:
            k["algorithmic_bytes"] = alg[name]
            k["achieved_GBs"] = round(alg[name] / (avg * 1e-3) / 1e9, 1)
            k["frac_of_hbm_peak"] = round(k["achieved_GBs"] / hbm_peak, 4)
            if l2_peak:
                k["frac_of_l2_peak"] = round(k["achieved_GBs"] / l2_peak, 4)
        kernels[name] = k
    dom = max((n for n in kernels if n in alg), key=lambda n: kernels[n]["avg_ms"] * kernels[n]["launches"])
    # DRAM bytes per launch from ncu, only if a capture of THIS shape and GPU count is committed (tools/profile_round.sh)
    traffic, dram_step = None, None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath)).get(shape, {}).get(str(world), {})
        traffic = tj.get(dom)
        if tj.get("_step_total"):
            dram_step = {"bytes_per_step": tj["_step_total"], "GBs": round(tj["_step_total"] / (ms_step * 1e-3) / 1e9, 1),
                         "frac_of_hbm_peak": round(tj["_step_total"] / (ms_step * 1e-3) / 1e9 / hbm_peak, 4),
                         "source": tj.get("_source")}
    peak = l2_peak if l2_bound else hbm_peak
    step_bytes = bf + b_src
    roofline = {"bound": "l2" if l2_bound else "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_GBs"], "peak": peak,
                "unit": "GB/s", "frac": round(kernels[dom]["achieved_GBs"] / peak, 4), "traffic": traffic,
                "peak_source": "profiles/l2_peak.json (L2 -> SM read bandwidth measured on this pool with tools/l2peak.cu)"
                if l2_bound else hbm_src,
                "algorithmic_bytes_per_launch": alg[dom],
                "hbm": {"peak": hbm_peak, "frac": kernels[dom]["frac_of_hbm_peak"], "peak_source": hbm_src},
                "whole_step": {"performed_bytes": step_bytes, "achieved_GBs": round(step_bytes / (ms_step * 1e-3) / 1e9, 1),
                               "frac_of_bound_peak": round(step_bytes / (ms_step * 1e-3) / 1e9 / peak, 4),
                               "frac_of_hbm_peak": round(step_bytes / (ms_step * 1e-3) / 1e9 / hbm_peak, 4),
                               "dram": dram_step,
                               "note": "bytes of the passes actually performed (forward gather + ONE backward gather + node pass); "
                                       "SURVEY 8d's figure additionally counts the reference's dst-major re-gather, which this "
                                       "engine eliminates"},
                "note": ("achieved = SURVEY 8d gather-model bytes of the kernel's own pass / its CUDA-event time.  bound = l2: every "
                         f"(N x D) head slab of the gathered table ({slab_mb:.0f} MB) is L2-resident by construction, so the "
                         "model's bytes are L2 -> SM traffic and the HBM fraction (`hbm`) exceeds 1; `traffic` = DRAM bytes ncu "
                         "measured for this launch, or null when no capture of this shape / GPU count is committed")
                if l2_bound else "achieved = SURVEY 8d gather-model bytes of the kernel's own pass / its CUDA-event time; the "
                                 f"gathered head slab ({slab_mb:.0f} MB) exceeds the L2, rows come from DRAM"}

    # ---------------- value parity of THIS run against the row-subsample oracle (checker only) ----------------
    parity = None
    if world == 1 and rank == 0 and not args.no_parity:
        parity = parity_check(graph, full_src, full_dst, n_nodes, c, ft_own, el_own, er, ee, gout, cs_l, ds_l, step_resident, dev)
        for t in leaves:
            t.grad = None
    del full_src, full_dst

    del ft_own, el_own, er, ee, gout, leaves
    torch.cuda.empty_cache()

    e2e = None if args.no_e2e else run_e2e(args, shape, c, graph, layer, world, rank, dev, n_nodes, n_edges, n_own, E_local, cs_l,
                                           ds_l, cs_own, barrier, seeds, replicas)

    # secondary number: the same layer on a heavy-tailed graph (dst ~ rank^-0.8; the hottest row has ~2 % of all edges)
    skew = None
    if world == 1 and not args.no_skew and shape == "proteins":
        s2, d2 = synth_edges(n_nodes, n_edges, dev, seed=0, power_law=0.8)
        g2 = bot_b200.Graph(s2, d2, n_nodes)
        g2.create_formats_()
        del s2, d2
        gen2 = torch.Generator(device=dev).manual_seed(2)
        t_ft = torch.randn(n_nodes, H, D, device=dev, generator=gen2).requires_grad_(True)
        t_el = torch.randn(n_nodes, H, device=dev, generator=gen2).requires_grad_(True)
        t_er = torch.randn(n_nodes, H, device=dev, generator=gen2).requires_grad_(True)
        t_ee = torch.randn(n_edges, functional.pad_heads(H), device=dev, generator=gen2).requires_grad_(True)
        t_go = torch.randn(n_nodes, H, D, device=dev, generator=gen2)

        def step_skew():
            keep = functional.edge_drop_keep(n_edges, int(n_edges * c["edge_drop"]), next(seeds), dev)
            gat_fused(g2, t_ft, t_el, t_er, t_ee, keep, None, None, None, SLOPE, 0.0, 0, edge_order="canonical").backward(t_go)
            for t in (t_ft, t_el, t_er, t_ee):
                t.grad = None

        for _ in range(2):
            step_skew()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            step_skew()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        skew = {"dst_distribution": "rank^-0.8", "max_in_degree": int(g2._info.max_in_deg), "ms_per_step": round(ms, 3),
                "value": n_edges / (ms * 1e-3), "unit": "edges/s", "split_row_slots": int(g2._info.n_slots_in)}
        del g2, t_ft, t_el, t_er, t_ee, t_go
        torch.cuda.empty_cache()

    cpu_baseline = cora = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_port_run(shape, steps=2, warmup=1, budget_s=25.0)
        cpu_baseline = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cora = cora_cpu_reference()

    if rank == 0:
        cfg = common_config(shape, n_nodes, n_edges, world)
        line = {
            "metric": metric_name(shape), "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if replicas else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "roofline": roofline, "kernels": kernels, "instrumented_ms_per_step": round(ms_instr / args.steps, 4),
            "graph": {"canonical_edge_order": bool(info.in_eid_identity), "transpose_tiles": [int(info.tiles_src), int(info.tiles_dst)],
                      "split_row_slots": [int(info.n_slots_in), int(info.n_slots_out)],
                      "halo_exchange": None if layer is None else (layer.exchange if layer.plan == "dense" else "sparse all-to-all")},
            "parity": parity, "cpu_baseline": cpu_baseline, "config1_cora_cpu_reference": cora, "e2e": e2e, "skew_variant": skew,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if host_affinity is not None:
            line["host_affinity_rank0"] = host_affinity
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, node_arrays, edge_arrays, max_rows=8192, max_edges=1 << 19, max_bytes=64 << 20):
    """--dump-outputs: write every array that is not None as <out_dir>/<name>.npy in float32.  Node-indexed arrays
    longer than ``max_rows`` keep the same seeded sample of rows, edge-indexed ones longer than ``max_edges`` the same
    seeded sample of edges (canonical edge order), so that the files stay small (about 50 MB at every shape) and two
    runs with the same arguments write the same rows."""
    import numpy as np

    out = {}
    for arrays, cap in ((node_arrays, max_rows), (edge_arrays, max_edges)):
        arrays = {k: v for k, v in arrays.items() if v is not None}
        if not arrays:
            continue
        n = next(iter(arrays.values())).shape[0]
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values if n > cap else None
        for name, t in arrays.items():
            out[name] = (t if idx is None else t[idx.to(t.device)]).detach().float().cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > max_bytes:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {max_bytes}-byte cap")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def parity_check(graph, src, dst, n_nodes, c, ft, el, er, ee, gout, cs, ds, step, dev, n_v=400, n_u=6):
    """One more (untimed) step of the resident leg, compared on a random sample of rows with the fp64 row-subsample
    oracle (oracle/gat_rows.py — the CHECKER; nothing on the measured path touches it)."""
    from oracle import gat_rows

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import philox_attn_mul, rel_err

    H = c["H"]
    sd = 424242
    out, keep = step(keep_grads=True, seed=sd)
    torch.cuda.synchronize()
    perm = graph.edge_perm()
    if perm is not None:        # the resident operands are in canonical order: show the oracle the COO in that order
        src, dst = src[perm], dst[perm]
    rs = torch.Generator().manual_seed(7)
    V = torch.randperm(n_nodes, generator=rs)[:n_v].to(dev)
    U = torch.randperm(n_nodes, generator=rs)[:n_u].to(dev)
    W = torch.unique(torch.cat([V, gat_rows.adjacent_dst(src, dst, n_nodes, U)]))
    sub = gat_rows.build_sub(src, dst, n_nodes, n_nodes, W, ft=ft, el=el, er=er, ee=ee, keep=keep, src_scale=cs, dst_scale=ds, gout=gout)
    if c["attn_p"] > 0:
        sub["attn_mul"] = philox_attn_mul(sd, 0, H, c["attn_p"], eids=sub["eid"].numpy()).double()
    ref = gat_rows.eval_explicit(sub, SLOPE)
    Wd, Ud, comp = sub["W"].to(dev), sub["U"].to(dev), sub["complete"]
    errs = {"out": rel_err(out[Wd], ref["out"]),
            "grad_ft": rel_err(ft.grad[Ud][comp.to(dev)], ref["grad_ft"][comp]),
            "grad_el": rel_err(el.grad[Ud][comp.to(dev)], ref["grad_el"][comp])}
    if er is not None:
        errs["grad_er"] = rel_err(er.grad[Wd], ref["grad_er"])
    if ee is not None:
        errs["grad_ee"] = rel_err(ee.grad[sub["eid"].to(dev)][:, :H], ref["grad_ee"])
    return {"parity_max_rel": max(errs.values()), "forward_max_rel": errs["out"],
            "grad_max_rel": max(v for k, v in errs.items() if k != "out"), "per_tensor": errs,
            "tolerance": {"forward": 1e-5, "grad": 1e-4}, "ok": errs["out"] <= 1e-5 and all(v <= 1e-4 for v in errs.values()),
            "rows_checked": {"dst": int(W.numel()), "src": int(comp.sum()), "edges": int(sub["e_src"].numel())},
            "checker": "oracle/gat_rows.py eval_explicit (fp64) on all in-edges of the sampled rows; metric max|x-ref|/max|ref|"}


def run_e2e(args, shape, c, graph, layer, world, rank, dev, n_nodes, n_edges, n_own, E_local, cs_l, ds_l, cs_own, barrier, seeds,
            replicas):
    """The same metric through the reference-facing module call with HOST buffers: every step copies its inputs from
    pinned host memory (bot_b200.HostFeed, double-buffered) and reads its loss back."""
    import torch.distributed as dist

    import bot_b200
    from bot_b200 import functional

    H, D, F_in = c["H"], c["D"], c["in_feats"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.manual_seed(0)
    v2 = shape in ("proteins", "products")
    if v2:
        from bot_b200.ogbn_proteins import GATConv

        conv = GATConv(F_in, EDGE_EMB if c["ee"] else 0, D, n_heads=H, edge_drop=c["edge_drop"]).to(dev)
        enc = torch.nn.Linear(EDGE_FEATS, EDGE_EMB).to(dev) if c["ee"] else None      # the model's per-layer edge_encoder[i]
    else:
        from bot_b200.no_sampling import GATConv

        conv = GATConv(F_in, D, num_heads=H, attn_drop=c["attn_p"], use_symmetric_norm=True).to(dev)
        conv.attn_dropout_mode = "fused"
        enc = None
    conv.train()
    params = list(conv.parameters()) + (list(enc.parameters()) if enc is not None else [])
    host = [torch.randn(n_own, F_in).pin_memory()]
    if c["ee"]:
        # RAW 8-dim edge features of this rank's edges, stored in the graph's canonical edge order (static data: permuted
        # once when it was assigned, bot_b200.graph.EdgeFrame); the layer's fused encoder turns them into logits on the GPU
        host.append(torch.rand(E_local, EDGE_FEATS).pin_memory())
    h2d = sum(t.numel() * 4 for t in host)

    def layer_call(x, fe):
        if layer is None:
            if v2:
                fe_arg = None if fe is None else bot_b200.EdgeEmbedding(fe.wait(), enc, canonical=True)
                return conv(graph, x, fe_arg)
            return conv(graph, x.wait() if isinstance(x, bot_b200.Deferred) else x)
        # partitioned: the module's body spelled out around PartitionedGraph.gat (projections of the OWNED rows only)
        x = x.wait() if isinstance(x, bot_b200.Deferred) else x
        sd = next(seeds)
        keep = functional.edge_drop_keep(E_local, int(E_local * c["edge_drop"]), sd, dev) if c["edge_drop"] > 0 else None
        if v2:
            ft = conv.src_fc(x).view(-1, H, D)
            resid = conv.dst_fc(x).view(-1, H, D)
            el, er = conv.attn_src_fc(x), conv.attn_dst_fc(x)
            ee = bot_b200.EdgeEmbedding(fe.wait(), enc, canonical=True).logits(conv.attn_edge_fc.weight) if fe is not None else None
            return layer.gat(ft, el, er, ee, keep, None, None, None, SLOPE, 0.0, 0, edge_order="canonical") + resid
        ft = conv.fc(x).view(-1, H, D)
        el = torch.einsum("nhd,hd->nh", ft, conv.attn_l[0]) * cs_own.unsqueeze(-1)      # el from the scaled ft, models.py:517
        return layer.gat(ft, el, None, None, keep, None, cs_l, ds_l, SLOPE, c["attn_p"], sd, edge_order="canonical") \
            + conv.res_fc(x).view(-1, H, D)

    def finish(y):
        loss = y.square().mean()
        loss.backward()
        if world > 1 and not replicas:
            flat = torch.cat([p.grad.flatten() for p in params if p.grad is not None])
            dist.all_reduce(flat)                      # data-parallel weight gradients
        for p in params:
            p.grad = None
        return float(loss.item())  # device -> host read of the step's result

    def run_fed(k):
        # bot_b200.HostFeed: the copies of step i+1 are enqueued before step i's layer and run beside it
        feed = bot_b200.HostFeed(dev, depth=2)
        feed.submit(*host)
        for i in range(k):
            if i + 1 < k:
                feed.submit(*host)
            got = feed.take(requires_grad=(0,))
            finish(layer_call(got[0], got[1] if len(got) > 1 else None))

    def run_serial(k):
        # copy and layer of the same step back to back (how the reference's loop is written)
        for _ in range(k):
            feed = bot_b200.HostFeed(dev, depth=1)
            feed.submit(*host)
            got = feed.take(requires_grad=(0,))
            finish(layer_call(got[0], got[1] if len(got) > 1 else None))

    def timed(run, k):
        barrier()
        e0.record()
        run(k)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / k

    w_e2e = max(1, min(args.warmup, 3))
    unp = None
    if world == 1:
        run_serial(w_e2e)
        k_serial = max(1, min(args.steps, 5))
        ms_serial = timed(run_serial, k_serial)
        unp = {"ms_per_step": round(ms_serial, 3), "value": n_edges / (ms_serial * 1e-3), "steps": k_serial,
               "note": "same call with each step's copy issued inside the step (no prefetch)"}
        torch.cuda.empty_cache()
    run_fed(w_e2e)
    k_e2e = max(1, args.steps)
    ms_e2e = timed(run_fed, k_e2e)
    h2d_total = h2d
    if world > 1:
        t = torch.tensor([float(h2d)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        h2d_total = int(t.item())
    total_edges = n_edges * (world if replicas else 1)
    call = ("bot_b200.ogbn_proteins.GATConv.forward(graph, feat_src, EdgeEmbedding(raw efeat, edge_encoder))" if shape == "proteins" else
            "bot_b200.ogbn_products.GATConv.forward(graph, feat_src)" if shape == "products" else
            "bot_b200.no_sampling.GATConv.forward(graph, feat)")
    model_line = None
    if world == 1 and shape == "proteins" and not args.no_e2e_model:
        del conv, enc, params
        torch.cuda.empty_cache()
        model_line = run_e2e_model(args, c, graph, dev, n_nodes, n_edges, host[1])
    return {"value": total_edges / (ms_e2e * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": 4 * world,
            "model": model_line,
            "ms_per_step": round(ms_e2e, 3), "steps": k_e2e,
            "call": call + " + backward" + ("" if world == 1 else ", partitioned: every rank projects its OWNED rows, runs "
                    "PartitionedGraph.gat (halo all-gather / gradient reduce-scatter inside), all-reduces the weight gradients") +
                    f"; per step every rank copies feat_src ({n_own} x {F_in})" + (f" and the RAW edge features ({E_local} x {EDGE_FEATS}, "
                    "canonical edge order)" if c["ee"] else "") + " from pinned host memory through bot_b200.HostFeed (double-buffered: step "
                    "i+1's copy is enqueued before step i's layer) and reads its loss back; graph structure resident (the reference "
                    "moves the graph once, run.py:539); dense nn.Linear projections included; max over ranks",
            "unpipelined": unp}


def run_e2e_model(args, c, graph, dev, n_nodes, n_edges, host_efeat):
    """The same end-to-end measurement one level up: the reference's whole 6-layer proteins model
    (src/ogbn-proteins/models.py:230-264 through bot_b200.ogbn_proteins.GAT.forward), one full-graph training step per
    iteration, node and RAW edge features copied from pinned host memory every step, loss read back.  The copy
    (1.27 GB, ~23 ms) amortises over six layers here."""
    import torch.nn.functional as F

    import bot_b200
    from bot_b200.ogbn_proteins import GAT

    n_layers, n_tasks, node_feats = 6, 112, 8
    torch.manual_seed(0)
    model = GAT(node_feats, EDGE_FEATS, n_tasks, n_layers, c["H"], c["D"], EDGE_EMB, F.relu, 0.25, 0.1, 0.0, c["edge_drop"]).to(dev)
    model.train()
    host = [torch.randn(n_nodes, node_feats).pin_memory(), host_efeat]
    labels = (torch.rand(n_nodes, n_tasks, device=dev) > 0.5).float()      # resident, like the reference's labels (gat.py:62)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run(k):
        feed = bot_b200.HostFeed(dev, depth=2)
        feed.submit(*host)
        for i in range(k):
            if i + 1 < k:
                feed.submit(*host)
            x, fe = feed.take()
            graph.srcdata["feat"] = x.wait()
            graph.edata.put_canonical("feat", fe.wait())      # static features, stored canonically on the host
            loss = F.binary_cross_entropy_with_logits(model(graph), labels)
            loss.backward()
            model.zero_grad(set_to_none=True)
            float(loss.item())

    run(2)
    k = max(2, min(args.steps, 5))
    torch.cuda.synchronize()
    e0.record()
    run(k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    peak = torch.cuda.max_memory_allocated() / 2**30
    del model, labels
    graph.srcdata.pop("feat", None)
    torch.cuda.empty_cache()
    return {"call": f"bot_b200.ogbn_proteins.GAT.forward(graph) + binary_cross_entropy_with_logits + backward: {n_layers} layers, "
                    f"{c['H']} heads x {c['D']}, edge encoder fused per layer, full graph (N={n_nodes}, E={n_edges}); per step "
                    f"node features ({n_nodes} x {node_feats}) and RAW edge features ({n_edges} x {EDGE_FEATS}) copied from pinned "
                    "host memory (HostFeed, double-buffered), loss read back",
            "ms_per_step": round(ms, 3), "steps": k, "layers": n_layers,
            "value": n_layers * n_edges / (ms * 1e-3), "unit": "layer-edges/s (edges x layers per second)",
            "h2d_bytes_per_step": sum(t.numel() * 4 for t in host), "d2h_bytes_per_step": 4, "peak_mem_GB": round(peak, 1)}


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="proteins", choices=list(SHAPES),
                    help="BASELINE.json config to run (default: the headline ogbn-proteins shape)")
    ap.add_argument("--nodes", type=int, default=0, help="override the shape's node count (developer runs)")
    ap.add_argument("--edges", type=int, default=0, help="override the shape's edge count (developer runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-skew", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="developer runs: skip the end-to-end leg")
    ap.add_argument("--no-e2e-model", action="store_true", help="skip the whole-model end-to-end line (proteins shape, 1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's layer output and input gradients (seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
