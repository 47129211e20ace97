#!/usr/bin/env python
"""GripNet hot-path benchmark: fwd+bwd edges/s per epoch on synthetic supergraphs shaped like the reference's.

    python bench.py --gpus N --steps K --warmup W                 # this repo (CUDA, sm_100a), BASELINE metric
    python bench.py --impl reference --steps K --warmup W          # the reference's CPU path (oracle port)
    python bench.py --workload aminer|freebase-d|pose2|scaled ...  # the other BASELINE configs (their own metric label)

One "step" = one training epoch's forward + loss + backward over the whole supergraph (the reference trains
full-batch, GripNet-pose.py:113-144; optimiser excluded, SURVEY §8d).  edges/s = E_epoch / t_step with E_epoch
the input edges traversed by the message-passing layers plus the decoder's edge evaluations (pose:
2*E_gg + E_gd + E_dd + 2*E_dd = 4 081 044).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs in HBM, the whole step replayed
from one CUDA graph); `e2e` = the same step driven with HOST buffers: the epoch's inputs are copied from pinned
host memory each step and the loss + scores are read back.  The default (pose) line also carries
`config5`: BASELINE config 5 (10 M nodes / ~520 M edges, destination-partitioned over the N GPUs of the run)
timed right after the headline workload, and at N > 1 `loss_check`: the partitioned loss against a single-GPU
replay of the same scaled supergraph on rank 0.

The reference arm imports `synthdata` (neutral generators) and `oracle` only — never `gripnet_b200` — so its
process does not map the product's library.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: NCCL's own version / INFO lines go to a file instead
if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
    os.environ["NCCL_DEBUG_FILE"] = "/tmp/nccl_debug_%h_%p.log"

import numpy as np  # noqa: E402
import torch  # noqa: E402

UNIT = "edges/s"
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 64 * 1000 * 1000
METRICS = {
    "pose": "GripNet fwd+bwd edges/sec per epoch (pose-0 shape)",
    "pose2": "GripNet fwd+bwd edges/sec per epoch (pose-2 shape, R=1097)",
    "aminer": "GripNet fwd+bwd edges/sec per epoch (aminer shape)",
    "freebase-d": "GripNet fwd+bwd edges/sec per epoch (freebase-d shape)",
    "scaled": "GripNet fwd+bwd edges/sec per epoch (scaled 10 M-node supergraph, config 5)",
    "scaled-small": "GripNet fwd+bwd edges/sec per epoch (small chain, smoke test of config 5)",
}


def workload_desc(workload, scale=1):
    """ONE description per (workload, scale): both arms print exactly this string in `config.workload`."""
    if workload == "pose":
        base = ("pose-0-shaped synthetic supergraph (n_g=19081,E_gg=1431224,n_d=645,E_gd=18596,R=16,E_dd=400000), "
                "GripNet-pose model gg[32,16,16]->gd(64->16|32)->dd RGCN[48,32]->DistMult(80,16); one step = "
                "fwd+loss+bwd of one full-batch epoch")
        return base if scale == 1 else base + f"; nodes and edges of every supervertex scaled x{scale} (weak scaling)"
    if workload == "pose2":
        return ("pose-2-shaped synthetic supergraph (config 4: n_g=19081,E_gg=1431224,n_d=645,E_gd=18596,R=1097 "
                "power-law relations, E_dd~8.3M over a pool of 63473 drug pairs), GripNet-pose model; one step = "
                "fwd+loss+bwd of one full-batch epoch")
    if workload == "aminer":
        return ("aminer-shaped synthetic NC supergraph (config 2: n_p=200000,E_pp=2000000,n_a=150000,E_pa=600000,"
                "E_aa=1500000,C=8), pp[128,64,64]->pa(256->64|64)->aa[128,128,32]->mcip(288,8); one step = "
                "fwd+loss+bwd of one full-batch epoch")
    if workload == "freebase-d":
        return ("freebase-d-shaped synthetic NC supergraph (config 3: n_p=n_q=300000,E_pp=E_qq=3000000,n_a=100000,"
                "E_pa=E_qa=1000000,E_aa=1000000,C=8), pp/qq[256,128,128]->pa/qa(512->128)->mean3->aa[128,32]->"
                "mcip(32,8); one step = fwd+loss+bwd of one full-batch epoch")
    if workload == "scaled":
        return ("scaled synthetic supergraph chain A->B->C (config 5: R-MAT degrees, N=(4M,4M,2M) nodes, "
                "200M+200M+20M intra + 50M+50M inter edges), ChainModel hid=64, node classification on C; one step = "
                "fwd+loss+bwd of one full-batch epoch")
    return "small synthetic supergraph chain A->B->C (smoke test of config 5), ChainModel hid=64"


# ------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port (reference semantics, torch-CPU, all host threads).
# Imports synthdata + oracle only.
# ------------------------------------------------------------------------------------------
def _cpu_inputs(workload, scale):
    import synthdata
    from oracle import port, synth
    if workload == "pose":
        g = synthdata.pose_graph_scaled(scale)
        return g, synth.pose_params(g, bias_jitter=False), port.pose_forward, synthdata.pose_edges_per_epoch(g)
    if workload == "pose2":
        g = synthdata.pose2_graph()
        return g, synth.pose_params(g, bias_jitter=False), port.pose_forward, synthdata.pose_edges_per_epoch(g)
    if workload == "aminer":
        g = synthdata.aminer_full()
        return g, synth.aminer_params(g, bias_jitter=False), port.aminer_forward, nc_edges_per_epoch(g)
    if workload == "freebase-d":
        g = synthdata.freebase_d_full()
        return g, synth.freebase_d_params(g, bias_jitter=False), port.freebase_d_forward, nc_edges_per_epoch(g)
    raise SystemExit(f"bench.py: the CPU arm has no port of workload {workload!r} (config 5 has no single-host "
                     "reference: the reference is single-device and the graph is a scaling construct)")


def nc_edges_per_epoch(g):
    """Input edges traversed by one forward of the NC models: 2 GCN layers on every intra-supervertex graph
    with two layers (pp, qq; aa has 2 in the aminer model, 1 in freebase-d) + the bipartite edges."""
    e = 2 * g["pp_edge_index"].shape[1] + g["pa_edge_index"].shape[1]
    if "qq_edge_index" in g:
        e += 2 * g["qq_edge_index"].shape[1] + g["qa_edge_index"].shape[1] + g["aa_edge_index"].shape[1]
    else:
        e += 2 * g["aa_edge_index"].shape[1]
    return e


def cpu_reference_run(workload, steps, warmup, state_dict=None, scale=1, budget_s=100.0):
    """Time the reference's CPU path (oracle/port.py: index_select -> message -> index_add + autograd) on the
    workload (pose scaled `scale`-fold like the CUDA arm at N = scale GPUs).  Full epochs; at most `steps` of
    them and at most ~`budget_s` seconds of timed work (never fewer than 2)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g, p, forward, e_epoch = _cpu_inputs(workload, scale)
    if state_dict is not None:
        p = {k: v.detach().cpu().clone() for k, v in state_dict.items()}
    p = {k: v.requires_grad_(True) for k, v in p.items()}
    cache = {}
    times = []
    i = 0
    while True:
        for v in p.values():
            v.grad = None
        t0 = time.perf_counter()
        out = forward(p, g, cache)
        out[0].backward()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        i += 1
        if len(times) >= steps or (len(times) >= 2 and sum(times) + dt > budget_s):
            break
    t = sum(times) / len(times)
    return {"value": e_epoch / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} full epochs (fwd+loss+bwd, {e_epoch} edges each) after {warmup} warm-up, "
                      f"mean {t * 1e3:.0f} ms/epoch, torch-CPU on {cores} threads",
            "ms_per_step": t * 1e3, "loss": float(out[0].detach()), "steps_run": len(times), "edges": e_epoch}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scale = max(1, int(os.environ.get("WORLD_SIZE", args.gpus))) if args.workload == "pose" else 1
    r = cpu_reference_run(args.workload, args.steps, max(args.warmup, 1), scale=scale)
    line = {
        "impl": "reference", "metric": METRICS[args.workload], "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps_run"], "requested_steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_desc(args.workload, scale), "edges_per_step": r["edges"],
                   "arm": "reference path on host cores: oracle port of gripnet/*.py (torch-CPU index_select + "
                          "index_add + autograd), PyG cannot be installed here"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.4)                      # nvidia-smi start-up: first sample before the timed region
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is None:
            return
        time.sleep(0.1)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) >= 9:
                self.rows.append(f)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def committed_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each kernel, extracted from the committed
    `ncu --set full` capture of this command by profiles/extract_traffic.py -> profiles/traffic.json."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.isfile(path):
        return {}
    with open(path) as f:
        return json.load(f).get(workload, {})


def timed_steps(step, n, flush):
    """Run `step` n times; CUDA events around every step on the current stream, L2 flushed in between."""
    evs = []
    for _ in range(n):
        if flush is not None:
            flush.zero_()                       # > L2: the next step starts from HBM
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def dump_outputs(out_dir, named):
    """Write each (name, tensor) of `named` to out_dir/<name>.npy as float32, DUMP_BYTES in all at most.  The
    budget is shared out smallest array first; an array larger than its share is replaced by a sample of its
    rows: a sorted choice without replacement from numpy's default_rng(0) that depends on the row count only,
    so two builds of the project dump the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    named = sorted(named, key=lambda kv: kv[1].numel())
    left = DUMP_BYTES
    for i, (name, t) in enumerate(named):
        share = left // (len(named) - i)
        t = t.detach()
        if t.dim() > 0 and t.numel() * 4 + 256 > share:
            row_bytes = 4 * (t.numel() // max(t.size(0), 1))
            k = max(0, (share - 256) // row_bytes)
            rows = np.sort(np.random.default_rng(0).choice(t.size(0), size=k, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, t.float().cpu().numpy())
        left -= os.path.getsize(path)


def e2e_pipelined(io, step, n_steps, flush):
    """End-to-end steps with the PCIe copies double-buffered: the host->device copy of step i+1's inputs (copy
    stream 1, pinned host -> device staging slot) and the device->host read of step i-1's results (copy stream 2,
    device staging slot -> pinned host) overlap the compute of step i; the step itself starts with a device copy
    staging -> the graph's static input and ends with a device copy of its outputs into a staging slot.  Returns
    the device time of ALL n_steps (one event pair around the whole loop, L2 flushes included: every copy of every
    step lies inside the timed region)."""
    cur = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    in_dev, in_host = io["in_dev"], io["in_host"]
    stage_in = [torch.empty_like(in_dev) for _ in range(2)]
    probe = io["pick"](step.outputs)
    stage_out = [[torch.empty_like(t) for t in probe] for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]       # staging slot filled from the host
    ev_used = [torch.cuda.Event() for _ in range(2)]     # staging slot consumed by the step
    ev_res = [torch.cuda.Event() for _ in range(2)]      # results of a step are in the output staging slot
    ev_out = [torch.cuda.Event() for _ in range(2)]      # output staging slot read back to the host
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def issue_h2d(i):
        k = i % 2
        with torch.cuda.stream(s_in):
            if i >= 2:
                s_in.wait_event(ev_used[k])
            stage_in[k].copy_(in_host[i % len(in_host)], non_blocking=True)
            ev_in[k].record(s_in)

    start.record(cur)
    s_in.wait_event(start)
    s_out.wait_event(start)
    issue_h2d(0)
    for i in range(n_steps):
        k = i % 2
        if i + 1 < n_steps:
            issue_h2d(i + 1)
        flush.zero_()
        cur.wait_event(ev_in[k])
        in_dev.copy_(stage_in[k], non_blocking=True)
        ev_used[k].record(cur)
        outs = io["pick"](step.replay())
        if i >= 2:
            cur.wait_event(ev_out[k])                    # the read-back of step i-2 has left this slot
        for dst, src in zip(stage_out[k], outs):
            dst.copy_(src, non_blocking=True)
        ev_res[k].record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_res[k])
            for host, src in zip(io["out_host"], stage_out[k]):
                host.copy_(src, non_blocking=True)
            ev_out[k].record(s_out)
    cur.wait_event(ev_out[(n_steps - 1) % 2])
    if n_steps >= 2:
        cur.wait_event(ev_out[n_steps % 2])
    end.record(cur)
    torch.cuda.synchronize()
    return start.elapsed_time(end)


def _sync_replicated(model, row_partitioned):
    """Replicated parameters must be identical on every rank: broadcast rank 0's."""
    import torch.distributed as dist
    for k, v in model.named_parameters():
        if k not in row_partitioned:
            dist.broadcast(v.data, src=0)


# ------------------------------------------------------------------------------------------
# workloads of this repo's arm.  Every builder returns a dict:
#   model, fwd() -> outputs (outputs[0] = loss), dynamic (static input buffers rewritten per step), edges,
#   io (pinned-host <-> device plumbing of the e2e leg), loss_of(outputs) -> the global loss tensor,
#   kernels() -> the isolated-kernel roofline probes, row_partitioned parameter names
# ------------------------------------------------------------------------------------------
def build_pose(args, world, rank, dev, dctx, workload="pose"):
    """pose-0 at N=1; at N>1 the pose-shaped supergraph scaled N-fold (weak scaling) and destination-
    partitioned over the N ranks (SURVEY.md §8e): every rank owns 1/N of the rows of every supervertex and
    1/N of the decoder edge lists; operand rows move over NVLink peer memory."""
    import synthdata
    from gripnet_b200.pipelines import PoseModel, shard_pose, to_device
    g = synthdata.pose2_graph() if workload == "pose2" else synthdata.pose_graph_scaled(world, seed=1111)
    e_epoch = synthdata.pose_edges_per_epoch(g)
    torch.manual_seed(1111)
    if dctx is None:
        model = PoseModel(g["n_g"], g["n_d"], g["n_rel"]).to(dev)
        data = to_device(g, dev)
        neg_static = data["neg_edge_index"].clone()
    else:
        data = shard_pose(g, dctx, dev)
        torch.manual_seed(1111 + rank)
        model = PoseModel(data["n_g"], data["n_d"], g["n_rel"]).to(dev)
        model.dmt.dist_ctx = dctx
        _sync_replicated(model, ("gg.embedding", "gd.target_feat"))
        neg_static = data["neg_edge_index_local"].clone()
    n_d = g["n_d"]
    e_loc = neg_static.size(1)
    rs = np.random.RandomState(99 + rank)
    n_sets = 4
    neg_host = [torch.from_numpy(np.stack([rs.randint(0, n_d, e_loc), rs.randint(0, n_d, e_loc)]).astype(np.int64))
                .pin_memory() for _ in range(n_sets)]

    def fwd():
        return model(data, neg_static)

    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    host_scores = torch.empty(2 * e_loc, dtype=torch.float32).pin_memory()

    def loss_of(outs):
        return (dctx.loss_value if (dctx is not None and dctx.defer_grad_reduce) else outs[0]).detach().view(1)

    io = dict(in_dev=neg_static, in_host=neg_host,
              pick=lambda outs: [loss_of(outs), outs[2].detach(), outs[3].detach()],
              out_host=[host_loss, host_scores[:e_loc], host_scores[e_loc:]])

    def kernels():
        """Isolated-kernel probes: (name, launches per step, algorithmic bytes per launch, callable)."""
        from gripnet_b200 import ops
        from gripnet_b200.graph import pair_struct
        gg = model.gg.conv_list[0]._graph
        F = 16
        x = torch.randn(gg.fwd.n_cols, F, device=dev)
        out = torch.empty(gg.n_dst, F, device=dev)
        bias = torch.zeros(F, device=dev)
        nnz, n = gg.fwd.nnz, gg.n_dst
        probes = [("spmm_kernel (GCN SpMM over the gg graph, F=16)", 4,
                   nnz * (4 + 4 + 4 * F) + n * (8 + 4 * F),
                   lambda: ops.spmm(gg.fwd, ops.M(x), ops.M(out), F, bias=bias, relu=True))]
        # decoder probes on this rank's edge lists
        pos = data["dd_edge_index_local"] if dctx is not None else data["dd_edge_index"]
        et = data["dd_edge_type_local"] if dctx is not None else data["dd_edge_type"]
        n_z = (dctx.world * dctx.block(n_d)) if dctx is not None else n_d
        D, R, E = 80, g["n_rel"], pos.size(1)
        z = torch.randn(n_z, D, device=dev) * 0.3
        w = torch.randn(R, D, device=dev)
        coef = torch.randn(E, device=dev)
        ps = pair_struct(pos, et, n_z, R)
        probes.append(("distmult_fwd_batch_kernel (DistMult scores, one edge list)", 2, E * (24 + 8 * D + 4),
                       lambda: ops._distmult_fwd(z, w, pos, et, True)))
        probes.append(("pair_walk_batch_kernel (DistMult backward, one gather pass per edge list)", 2,
                       2 * E * (8 + 4 + 4 * D) + n_z * R * 4 * D,
                       lambda: ops._pair_walk(ps, coef, z)))
        return probes

    return dict(model=model, data=data, graph=g, fwd=fwd, dynamic=[neg_static], edges=e_epoch, io=io,
                output_names=("loss", "z", "pos_score", "neg_score"),
                host_loss=host_loss, loss_of=loss_of, h2d_bytes=int(neg_static.numel() * 8),
                d2h_bytes=int(4 + 2 * e_loc * 4), kernels=kernels,
                row_partitioned=("gg.embedding", "gd.target_feat") if dctx is not None else (),
                e2e_note="negatives from pinned host memory each step; loss and pos/neg scores read back")


def build_nc(args, world, rank, dev, dctx, workload):
    """BASELINE configs 2 and 3 (single GPU): aminer-shaped and freebase-d-shaped node classification."""
    import synthdata
    from gripnet_b200.pipelines import AminerModel, FreebaseDModel, to_device
    if dctx is not None:
        raise SystemExit(f"bench.py: workload {workload} is a single-GPU configuration")
    g = synthdata.aminer_full() if workload == "aminer" else synthdata.freebase_d_full()
    e_epoch = nc_edges_per_epoch(g)
    torch.manual_seed(1111)
    if workload == "aminer":
        model = AminerModel(g["n_p"], g["n_a"], g["n_class"]).to(dev)
    else:
        model = FreebaseDModel(g["n_p"], g["n_q"], g["n_a"], g["n_class"]).to(dev)
    data = to_device(g, dev)
    labels_static = data["train_node_class"]
    labels_host = [labels_static.cpu().pin_memory()]
    n_lab, n_class = labels_static.numel(), g["n_class"]

    def fwd():
        return model(data)

    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    host_scores = torch.empty(n_lab * n_class, dtype=torch.float32).pin_memory()
    io = dict(in_dev=labels_static, in_host=labels_host,
              pick=lambda outs: [outs[0].detach().view(1), outs[2].detach().view(-1)],
              out_host=[host_loss, host_scores])

    def kernels():
        from gripnet_b200 import ops
        pp = model.pp.conv_list[0]._graph
        F = model.pp.conv_list[0].out_channels
        x = torch.randn(pp.fwd.n_cols, F, device=dev)
        out = torch.empty(pp.n_dst, F, device=dev)
        bias = torch.zeros(F, device=dev)
        nnz, n = pp.fwd.nnz, pp.n_dst
        launches = 4 if workload == "aminer" else 8          # fwd + bwd of two layers (pp; pp and qq)
        return [(f"spmm_kernel (GCN SpMM over the pp graph, F={F})", launches,
                 nnz * (4 + 4 + 4 * F) + n * (8 + 4 * F),
                 lambda: ops.spmm(pp.fwd, ops.M(x), ops.M(out), F, bias=bias, relu=True))]

    return dict(model=model, data=data, graph=g, fwd=fwd, dynamic=[], edges=e_epoch, io=io, host_loss=host_loss,
                output_names=("loss", "z", "score"),
                loss_of=lambda outs: outs[0].detach().view(1), h2d_bytes=int(n_lab * 8),
                d2h_bytes=int(4 + n_lab * n_class * 4), kernels=kernels, row_partitioned=(),
                e2e_note="labels from pinned host memory each step; loss and class scores read back")


def build_chain(args, world, rank, dev, dctx, workload="scaled"):
    """BASELINE config 5: ~10 M nodes / ~520 M edges, three supervertices.  Partitioned runs stream the
    generator through per-rank filters: no rank holds a global edge list or builds a global CSR."""
    import synthdata
    from gripnet_b200.pipelines import ChainModel, chain_edges_per_epoch, shard_chain_streamed
    make = synthdata.chain_small if workload == "scaled-small" else synthdata.chain_full
    if dctx is None:
        data = make(dev)
    else:
        data = shard_chain_streamed(make, dctx, dev)
    e_epoch = chain_edges_per_epoch(data)
    torch.manual_seed(1111 + rank)
    n_class = data["n_class"]
    model = ChainModel(data["n_a"], data["n_b"], data["n_c"], n_class).to(dev)
    if dctx is not None:
        model.mcip.dist_ctx = dctx
        _sync_replicated(model, ("aa.embedding", "ab.target_feat", "bc.target_feat"))
    labels_static = data["train_node_class"]
    labels_host = [labels_static.cpu().pin_memory()]
    n_lab = labels_static.numel()
    torch.cuda.empty_cache()

    def fwd():
        return model(data)

    def loss_of(outs):
        return (dctx.loss_value if (dctx is not None and dctx.defer_grad_reduce) else outs[0]).detach().view(1)

    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    host_scores = torch.empty(max(n_lab * n_class, 1), dtype=torch.float32).pin_memory()
    io = dict(in_dev=labels_static, in_host=labels_host,
              pick=lambda outs: [loss_of(outs), outs[2].detach().view(-1)], out_host=[host_loss, host_scores[:n_lab * n_class]])

    def kernels():
        from gripnet_b200 import ops
        aa = model.aa.conv_list[0]._graph
        F = 64
        x = torch.randn(aa.fwd.n_cols, F, device=dev)
        out = torch.empty(aa.n_dst, F, device=dev)
        bias = torch.zeros(F, device=dev)
        nnz, n = aa.fwd.nnz, aa.n_dst
        return [(f"spmm_kernel (GCN SpMM over this rank's rows of the aa graph, F={F})", 8,
                 nnz * (4 + 4 + 4 * F) + n * (8 + 4 * F),
                 lambda: ops.spmm(aa.fwd, ops.M(x), ops.M(out), F, bias=bias, relu=True))]

    return dict(model=model, data=data, graph=None, fwd=fwd, dynamic=[], edges=e_epoch, io=io, host_loss=host_loss,
                output_names=("loss", "z", "score"),
                loss_of=loss_of, h2d_bytes=int(n_lab * 8), d2h_bytes=int(4 + n_lab * n_class * 4), kernels=kernels,
                row_partitioned=("aa.embedding", "ab.target_feat", "bc.target_feat") if dctx is not None else (),
                e2e_note="labels from pinned host memory each step; loss and class scores read back")


def build_workload(args, workload, world, rank, dev, dctx):
    if workload in ("pose", "pose2"):
        return build_pose(args, world, rank, dev, dctx, workload)
    if workload in ("aminer", "freebase-d"):
        return build_nc(args, world, rank, dev, dctx, workload)
    return build_chain(args, world, rank, dev, dctx, workload)


def capture_step(w, dctx, args, world, rank):
    """The whole step (forward + loss + backward + the partitioned run's gradient reduction) as ONE CUDA graph."""
    import gripnet_b200 as gb
    from gripnet_b200.capture import CapturedStep
    model = w["model"]
    replicated = [v for k, v in model.named_parameters() if k not in w.get("row_partitioned", ())]

    def post_backward():
        if dctx is not None:
            dctx.reduce_gradients(replicated)

    if not args.eager:
        try:
            return CapturedStep(w["fwd"], model.parameters(), dynamic_inputs=w["dynamic"], warmup=max(args.warmup, 3),
                                post_backward=post_backward), "whole step replayed from one CUDA graph"
        except Exception as e:  # pragma: no cover - a refused capture must not take the line down at N > 1
            if world == 1:
                raise
            sys.stderr.write(f"bench.py: CUDA-graph capture failed on rank {rank} ({type(e).__name__}: {e}); "
                             "running eagerly\n")
            torch.cuda.synchronize()

    class _Eager:
        def __init__(self):
            self.outputs = None
            self.launches_per_replay = 0

        def replay(self):
            for p in model.parameters():
                p.grad = None
            before = gb.launch_count()
            self.outputs = w["fwd"]()
            self.outputs[0].backward()
            post_backward()
            self.launches_per_replay = gb.launch_count() - before
            return self.outputs

    step = _Eager()
    for _ in range(max(args.warmup, 3)):
        step.replay()
    return step, "eager launches (no CUDA graph)"


def kernel_rooflines(w, step_ms, workload, flush, peaks, peak_src):
    """Time each probe kernel alone (CUDA events, cold L2) and rank them by their share of the step."""
    traffic = committed_traffic(workload)
    rows = []
    for name, launches, alg_bytes, fn in w["kernels"]():
        for _ in range(3):
            fn()
        us = statistics.mean(timed_steps(fn, 20, flush)) * 1e3
        achieved = alg_bytes / (us * 1e-6) / 1e9
        key = name.split(" ")[0]
        dram = traffic.get(key)
        rows.append({"kernel": name, "launches_per_step": launches, "us_per_launch": us,
                     "share_of_step": launches * us * 1e-3 / step_ms, "bound": "hbm",
                     "algorithmic_bytes": alg_bytes, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": dram,
                     "frac_dram": (dram / (us * 1e-6) / 1e9 / peaks["hbm_gbs"]) if dram else None})
    rows.sort(key=lambda r: -r["share_of_step"])
    top = dict(rows[0])
    top["peak_source"] = peak_src
    top["note"] = ("time-dominant probe kernel of the step (launches x isolated time); timed alone with CUDA events, "
                   "L2 flushed before every launch (burst peak applies).  `frac` counts ALGORITHMIC bytes (SURVEY §8d: "
                   "every gathered row as HBM traffic); `frac_dram` uses the measured dram__bytes of the committed ncu "
                   "capture: operands that fit the 126 MB L2 are served from L2, so frac_dram << frac by design")
    return top, rows


def time_workload(args, workload, world, rank, dev, dctx, steps, flush, with_e2e=True, dump_dir=None):
    """Build, capture and time one workload; with `dump_dir`, rank 0 writes what the last timed step computed
    (the model's outputs and every parameter gradient) there.  Returns (record, w, step)."""
    import torch.distributed as dist
    import gripnet_b200 as gb  # noqa: F401
    w = build_workload(args, workload, world, rank, dev, dctx)
    step, execution = capture_step(w, dctx, args, world, rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step.replay()
    barrier()
    with ClockSampler(dev.index or 0) as clk:
        t_wall0 = time.perf_counter()
        times = timed_steps(step.replay, steps, flush)
        barrier()
        t_wall = time.perf_counter() - t_wall0
    dev_ms = sum(times)
    loss_dev = float(w["loss_of"](step.outputs).cpu()[0])
    if dump_dir is not None and rank == 0:
        outs = [w["loss_of"](step.outputs)] + list(step.outputs[1:])
        grads = [("grad." + k, p.grad) for k, p in w["model"].named_parameters() if p.grad is not None]
        dump_outputs(dump_dir, list(zip(w["output_names"], outs)) + grads)

    io = w["io"]
    e2e_mode, e2e_ms = "pipelined", None
    if with_e2e:
        def e2e_step():
            io["in_dev"].copy_(io["in_host"][0], non_blocking=True)
            outs = io["pick"](step.replay())
            for host, src in zip(io["out_host"], outs):
                host.copy_(src, non_blocking=True)

        # double-buffered copies on every rank; the ranks AGREE on the outcome (MIN over ranks of the per-rank
        # check below), so either all of them keep the pipelined number or all of them time the serial loop
        e2e_want = os.environ.get("GRIPNET_BENCH_E2E", "pipelined")
        if e2e_want == "pipelined" and not args.eager:
            good, detail = 1, ""
            try:
                e2e_pipelined(io, step, 4, flush)                    # warm-up of the pipeline
                torch.cuda.synchronize()
                e2e_ms = e2e_pipelined(io, step, steps, flush)
                # check: the loss read back by the LAST pipelined step == that step's inputs run synchronously
                pipelined_loss = float(w["host_loss"][0])
                io["in_dev"].copy_(io["in_host"][(steps - 1) % len(io["in_host"])])
                torch.cuda.synchronize()
                sync_loss = float(io["pick"](step.replay())[0].cpu()[0])
                if not abs(pipelined_loss - sync_loss) <= 1e-6 * max(abs(sync_loss), 1e-30):
                    good, detail = 0, f"loss {pipelined_loss} vs {sync_loss}"
            except Exception as e:  # pragma: no cover - never let the e2e variant take the bench line down
                good, detail = 0, f"{type(e).__name__}: {e}"
                torch.cuda.synchronize()
            if good != 1:
                sys.stderr.write(f"bench.py: pipelined e2e rejected on rank {rank} ({detail})\n")
            if world > 1:
                agree = torch.tensor([good], device=dev, dtype=torch.int32)
                dist.all_reduce(agree, op=dist.ReduceOp.MIN)
                good = int(agree.item())
            if good != 1:
                if rank == 0:
                    sys.stderr.write("bench.py: timing the serial end-to-end loop instead\n")
                e2e_ms = None
            barrier()
        if e2e_ms is None:
            e2e_mode = "serial"
            for _ in range(3):
                e2e_step()
            barrier()
            e2e_ms = sum(timed_steps(e2e_step, steps, flush))
            barrier()
    # ---- max over ranks (the same global step runs on every rank: value = global edges / slowest rank)
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms if e2e_ms is not None else 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = float(t[0]), (float(t[1]) if e2e_ms is not None else None)
    rec = {"dev_ms": dev_ms, "e2e_ms": e2e_ms, "e2e_mode": e2e_mode, "execution": execution, "clocks": clk.summary(),
           "wall_s": t_wall, "loss": loss_dev, "edges": w["edges"], "launches": int(step.launches_per_replay),
           "steps": steps}
    return rec, w, step


def gather_global_state(model, row_partitioned, dims, dctx):
    """state_dict of the GLOBAL model on every rank: row-partitioned parameters all-gathered block by block."""
    import torch.distributed as dist
    out = {}
    for k, v in model.state_dict().items():
        if k in row_partitioned:
            n = dims[k]
            b = dctx.block(n)
            pad = torch.zeros((b,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
            pad[: v.size(0)].copy_(v)
            full = torch.empty((dctx.world * b,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
            dist.all_gather_into_tensor(full, pad)
            out[k] = full[:n].clone()
        else:
            out[k] = v.detach().clone()
    return out


def partitioned_loss_check(w, rec, dctx, dev, rank, workload):
    """Rank 0 replays the SAME global supergraph with the gathered parameters through the single-GPU path and
    compares the loss of the partitioned step with it (every rank takes part in the parameter gather)."""
    from gripnet_b200 import graph as G
    from gripnet_b200.pipelines import ChainModel, PoseModel, to_device
    g = w["graph"]
    if workload in ("pose", "pose2"):
        dims = {"gg.embedding": g["n_g"], "gd.target_feat": g["n_d"]}
    else:
        dims = {"aa.embedding": w["data"]["n_a_global"], "ab.target_feat": w["data"]["n_b_global"],
                "bc.target_feat": w["data"]["n_c_global"]}
    state = gather_global_state(w["model"], w["row_partitioned"], dims, dctx)
    if rank != 0:
        return None
    t0 = time.perf_counter()
    G.clear_cache()
    with torch.no_grad():
        if workload in ("pose", "pose2"):
            ref = PoseModel(g["n_g"], g["n_d"], g["n_rel"]).to(dev)
            ref.load_state_dict(state)
            loss = float(ref(to_device(g, dev))[0])
        else:
            import synthdata
            gg = (synthdata.chain_small if workload == "scaled-small" else synthdata.chain_full)(dev)
            ref = ChainModel(gg["n_a"], gg["n_b"], gg["n_c"], gg["n_class"]).to(dev)
            ref.load_state_dict(state)
            loss = float(ref(gg)[0])
            del gg
    del ref
    G.clear_cache()
    torch.cuda.empty_cache()
    part = rec["loss"]
    return {"partitioned": part, "single_gpu_replay": loss, "rel_err": abs(part - loss) / max(abs(loss), 1e-30),
            "tolerance": 1e-5, "ok": abs(part - loss) <= 1e-5 * max(abs(loss), 1e-30),
            "seconds": time.perf_counter() - t0,
            "note": "rank 0 rebuilt the global supergraph, loaded the all-gathered parameters into the single-GPU "
                    "model and ran its forward; same static negatives / labels"}


def config5_record(args, world, rank, dev, dctx, flush, peaks):
    """BASELINE config 5 at this run's N: ms/step, edges/s and the fraction of the per-rank roofline
    max(local SpMM bytes / HBM, gathered bytes / NVLink) of SURVEY §8e."""
    from gripnet_b200 import graph as G
    steps = max(2, min(args.steps, 5))
    rec, w, step = time_workload(args, "scaled", world, rank, dev, dctx, steps, flush, with_e2e=False)
    ms = rec["dev_ms"] / steps
    # per-rank algorithmic bytes of one step: every SpMM launch fwd and bwd (E'(8+4F) + N(8+4F)), F = 64 / 32
    model = w["model"]
    spmm_bytes, gathered, halo_used = 0, 0, 0
    halo = []
    for name, layers in (("aa", 2), ("ab", 1), ("bb", 2), ("bc", 1), ("cc", 2)):
        mod = getattr(model, name)
        convs = list(mod.conv_list) if hasattr(mod, "conv_list") else [mod.conv]
        for c in convs:
            gr = c._graph
            F = c.out_channels
            for csr, plan in ((gr.fwd, getattr(gr, "fwd_halo", None)), (gr.bwd, getattr(gr, "bwd_halo", None))):
                spmm_bytes += csr.nnz * (8 + 4 * F) + csr.n_rows * (8 + 4 * F)
                if world > 1:       # rows that enter this GPU per launch: the referenced halo rows, or whole blocks
                    rows_in = sum(plan.recv_counts) if plan is not None else (world - 1) * (csr.n_cols // world)
                    gathered += rows_in * F * 4
                    halo_used += plan is not None
        if world > 1 and hasattr(convs[0]._graph, "halo_fraction"):
            halo.append(round(convs[0]._graph.halo_fraction(), 4))
    t_hbm = spmm_bytes / (peaks["hbm_gbs"] * 1e9)
    t_link = gathered / 770e9
    ideal_ms = max(t_hbm, t_link) * 1e3
    out = {"workload": workload_desc("scaled"), "metric": METRICS["scaled"], "n_gpus": world, "scaling": "strong",
           "ms_per_step": ms, "edges_per_step": rec["edges"], "value": rec["edges"] / (ms * 1e-3), "unit": UNIT,
           "steps": steps, "launches_per_step": rec["launches"], "loss": rec["loss"], "execution": rec["execution"],
           "roofline": {"per_rank_spmm_bytes": spmm_bytes, "per_rank_gathered_bytes": gathered,
                        "hbm_ms": t_hbm * 1e3, "nvlink_ms": t_link * 1e3, "ideal_ms": ideal_ms,
                        "frac": ideal_ms / ms,
                        "note": "SURVEY §8e: max(local SpMM algorithmic bytes / measured HBM peak, gathered operand "
                                "bytes / 770 GB/s NVLink) over all SpMM launches of the step, per rank"},
           "prep": "per-rank: every rank filtered the streamed generator to its own edges and sorted only those "
                   "(no global edge list, no global CSR)" if world > 1 else "single GPU",
           "remote_operand_rows_referenced": halo or None,
           "exchange": None if world == 1 else
           (f"halo-packed rows over NVLink peer memory (gn_peer_halo_push) for {halo_used} SpMM operands per step, "
            "full slot all-gather (NVLS multicast) for the others")}
    if world > 1 and args.check_config5:
        out["loss_check"] = partitioned_loss_check(w, rec, dctx, dev, rank, "scaled")
    del w, step
    G.clear_cache()
    torch.cuda.empty_cache()
    return out


def run_cuda(args):
    import torch.distributed as dist
    import gripnet_b200 as gb  # noqa: F401
    from gripnet_b200 import graph as G

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (gripnet_b200 has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dctx = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from gripnet_b200.parallel import DistContext
        dctx = DistContext(defer_grad_reduce=True)       # ONE exchange for all weight gradients + the loss per step
    workload = args.workload
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev)
    peaks, peak_src = measured_peaks()

    rec, w, step = time_workload(args, workload, world, rank, dev, dctx, args.steps, flush,
                                 dump_dir=args.dump_outputs)
    model, e_epoch = w["model"], w["edges"]
    dev_ms, e2e_ms = rec["dev_ms"], rec["e2e_ms"]
    value = e_epoch * args.steps / (dev_ms * 1e-3)
    e2e_value = e_epoch * args.steps / (e2e_ms * 1e-3)
    roofline, all_kernels = kernel_rooflines(w, dev_ms / args.steps, workload if world == 1 else None, flush, peaks,
                                             peak_src)

    # ---- whole training epoch (SURVEY §8d: "optimiser excluded (reported separately)"): negative draw + fwd +
    #      loss + bwd + fused Adam + per-relation AUPRC/AUROC/AP, one CUDA graph, nothing crosses PCIe
    train_epoch = None
    state0 = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}     # the timed steps' parameters
    if world == 1 and workload == "pose" and not args.no_train_epoch:
        from gripnet_b200.training import PoseTrainer
        trainer = PoseTrainer(model, dict(w["data"]), lr=0.01, seed=1111, with_metrics=True, eager=args.eager)
        for _ in range(3):
            trainer.train_epoch()
        torch.cuda.synchronize()
        n_ep = min(args.steps, 100)
        t_ms = statistics.mean(timed_steps(trainer.train_epoch, n_ep, flush))
        train_epoch = {"ms_per_epoch": t_ms, "edges_per_s": e_epoch / (t_ms * 1e-3), "epochs_timed": n_ep,
                       "launches_per_epoch": trainer.launches_per_epoch, "loss_after": float(trainer.loss.detach()),
                       "train_auprc_auroc_ap": trainer.record.mean(dim=1).cpu().tolist(),
                       "includes": "on-device negative sampling (Philox) + (node, relation) structure rebuild, fwd, "
                                   "loss, bwd, fused multi-tensor Adam (lr 0.01), per-relation AUPRC/AUROC/AP; " +
                                   ("eager launches" if args.eager else "one CUDA graph per epoch") +
                                   ", L2 flushed between epochs"}
        del trainer

    loss_check = None
    if world > 1 and workload in ("pose", "scaled-small") and not args.no_loss_check:
        loss_check = partitioned_loss_check(w, rec, dctx, dev, rank, workload)
    exchange = None
    if dctx is not None:
        exchange = {"peer_gathers": dctx.peer_gathers, "nccl_gathers": dctx.nccl_gathers,
                    "peer_reductions": dctx.peer_reductions, "nccl_reductions": dctx.nccl_reductions,
                    "arena": dctx.arena is not None,
                    "nvls_multicast": bool(dctx.arena is not None and dctx.arena.multicast)}

    # ---- BASELINE config 5 at this N (default pose run only): free the headline workload first
    config5 = None
    if workload == "pose" and not args.no_config5:
        del step
        w_keep = {k: w[k] for k in ("h2d_bytes", "d2h_bytes", "e2e_note")}
        w.clear()
        model = None
        G.clear_cache()
        from gripnet_b200 import parallel
        parallel.clear_registry()
        torch.cuda.empty_cache()
        dctx5 = None
        if world > 1:
            from gripnet_b200.parallel import DistContext
            dctx5 = DistContext(defer_grad_reduce=True)
        try:
            config5 = config5_record(args, world, rank, dev, dctx5, flush, peaks)
        except Exception as e:  # pragma: no cover - the headline line must survive a failure of the extra leg
            if world > 1:
                raise
            config5 = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.synchronize()
        w = w_keep

    if rank == 0:
        cpu = None
        if world == 1 and workload in ("pose",) and not args.no_cpu_baseline:
            cpu = cpu_reference_run(workload, 3, 1, state0)
            cpu_loss = cpu.pop("loss")
            for k in ("ms_per_step", "steps_run", "edges"):
                cpu.pop(k)
            cpu["loss_check"] = {"cpu_port": cpu_loss, "note": "same parameters and graph, its own fixed negatives"}
        par = "single GPU"
        if world > 1:
            par = (f"destination-partitioned x{world}: per-rank graph prep (each rank sorts only the edges of its own "
                   "rows); SpMM operands exchanged by " +
                   ("gn_peer_allgather (P2P stores into the peers' symmetric-memory gather buffers over NVLink), "
                    "weight gradients + loss and the decoder's dz reduced by gn_peer_push + gn_slot_sum (rank-ordered "
                    "sums over peer memory, no NCCL in the step)" if exchange["arena"] else
                    "NCCL all-gather / all-reduce"))
        line = {
            "metric": METRICS[workload], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if workload.startswith("scaled") else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_desc(workload, world if workload == "pose" else 1),
                       "edges_per_step": e_epoch, "parallelism": par,
                       "l2": "flushed between timed steps (write of a 252 MiB buffer, outside the event pair)",
                       "execution": rec["execution"]},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": w["h2d_bytes"],
                    "d2h_bytes_per_step": w["d2h_bytes"], "ms_per_step": e2e_ms / args.steps,
                    "note": w["e2e_note"] + ("; copies double-buffered on two copy streams (H2D of step i+1 and D2H "
                                             "of step i-1 overlap step i), one event pair around all steps, L2 "
                                             "flushes inside the timed region" if rec["e2e_mode"] == "pipelined" else
                                             "; copies and step serialised on one stream")},
            "gpu_launches": int(rec["launches"] * args.steps),
            "launches_per_step": int(rec["launches"]),
            "clocks": rec["clocks"], "roofline": roofline, "roofline_kernels": all_kernels, "loss": rec["loss"],
            "wall_s_timed_region": rec["wall_s"],
        }
        if exchange is not None:
            line["exchange"] = exchange
        if loss_check is not None:
            line["loss_check"] = loss_check
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if train_epoch is not None:
            line["train_epoch"] = train_epoch
        if config5 is not None:
            line["config5"] = config5
        print(json.dumps(line), flush=True)
    if world > 1:
        # NCCL teardown with captured graphs alive can block forever: drain, rendezvous, leave
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="pose", choices=sorted(METRICS),
                    help="pose: BASELINE metric workload (pose-0 at N=1, scaled N-fold and partitioned at N>1; the line "
                         "also carries config 5 as `config5`); pose2 / aminer / freebase-d: configs 4 / 2 / 3 (N=1); "
                         "scaled: config 5 alone (10 M nodes / 520 M edges chain)")
    ap.add_argument("--no-train-epoch", action="store_true", help="skip the whole-training-epoch leg")
    ap.add_argument("--no-config5", action="store_true", help="skip the config-5 sub-record of the default run")
    ap.add_argument("--no-loss-check", action="store_true", help="skip the single-GPU replay of the partitioned loss")
    ap.add_argument("--check-config5", action="store_true",
                    help="also replay config 5 on rank 0 alone and compare the loss (tens of seconds, ~40 GB)")
    ap.add_argument("--eager", action="store_true", help="do not capture the step into a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, embeddings, scores and every "
                         "parameter gradient; rank 0's in a multi-GPU run) as DIR/<name>.npy in float32, 64 MB in all "
                         "at most; an array over its share holds a fixed seeded sample of its rows")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs is not None:
        ap.error("--dump-outputs applies to the CUDA arm (--impl cuda) only")
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
