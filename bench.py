"""bench.py - TwoWL forward+backward target-links/s on synthetic graphs (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload rmat|collab|cora] [--hidden H]
                    [--impl ours|reference] [--dump-outputs DIR]

One *step* = LocalWLNet.forward + binary_cross_entropy_with_logits + backward on one batch
(reference TwoWL/model/train.py:36-38) through the drop-in API of link-prediction-gnn_b200/TwoWL.
`value`  : whole-job target links/s with every input already resident in HBM (device-timed, CUDA events).
`e2e`    : the same through the reference-facing call sequence of train.py:18-38 starting from HOST
           buffers: pinned-host batch ids/labels -> H2D -> double / sample_block -> forward -> loss ->
           backward -> D2H of the loss, all inside the timed region.
`roofline`: the dominant kernel's algorithmic bytes / its CUDA-event time, against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle port of the reference path (oracle/twowl_oracle.py) on a bounded sample.
`same_config`: BOTH arms on ONE configuration the reference can run as written (configs[1]: the Cora-scale graph, hidden 64,
           the same host-generated graph, weights and batches) - the only GPU-over-CPU ratio a reader should quote.
`strong`  (N > 1): the same step with ONE batch whose pair rows are cut into row blocks over the ranks (twowl_b200.rowshard,
           north_star's partition), next to the target-link data-parallel `value`.
`--impl reference` times that CPU path alone (the reference is pure Python/torch-CPU; its hot loop is
restated 1:1 by the oracle, which is pinned to the reference by tests/golden).
`--dump-outputs DIR` writes what the last timed step computed - loss, logits and every parameter gradient - as
DIR/<name>.npy (float32). Graph, weights and batches are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {
    # name: (rmat scale, edge samples, (a,b,c,d), default hidden)
    "rmat": (20, 16_000_000, (0.57, 0.19, 0.19, 0.05), 64),     # configs[3]: R-MAT 1M nodes / 16M edges
    "collab": (18, 1_300_000, (0.57, 0.19, 0.19, 0.05), 128),   # configs[2]: ogbl-collab scale
    "cora": (None, 5278, None, 64),                             # configs[1]: 2708 nodes, uniform
}


# ------------------------------------------------------------------------------ synthetic graphs (input generation)

def make_graph(workload, seed, device, scale_override=None, samples_override=None):
    """-> dict(n, pos [2,E], pred [2,P], pos1 [R,2]) in the reference's doubled layout (SURVEY 8(d)); the generators live in
    TwoWL/operators/synthetic.py."""
    from TwoWL.operators.synthetic import rmat_edges, synthetic_link_graph
    from TwoWL.utils import double
    scale, samples, abcd, _ = WORKLOADS[workload]
    if workload == "cora":
        n = 2708
        g = torch.Generator(device=device).manual_seed(seed + 1)
        s = torch.randint(0, n, (samples,), generator=g, device=device)
        d = torch.randint(0, n, (samples,), generator=g, device=device)
    else:
        s, d, n = rmat_edges(scale_override or scale, samples_override or samples, abcd, seed, device)
    sg = synthetic_link_graph(n, s, d, seed)
    pos, pred = double(sg["pos_und"]), double(sg["neg_und"])
    pos1 = torch.cat((pos.t(), pred.t()), dim=0).contiguous()
    return dict(n=n, pos=pos, pred=pred, pos1=pos1, und=pos.shape[1] // 2)


def draw_batch(und, n_pred_und, nb, step, replicate=False):
    """Host-side batch draw, as train.py:18-23: nb positive + nb negative undirected ids (pinned). Under torchrun every
    rank takes its own disjoint slice of ONE seeded global permutation per step (twowl_b200.dist.shard_batch)."""
    from twowl_b200 import dist as D
    i1 = D.shard_batch(und, nb, step, seed=1, replicate=replicate).pin_memory()
    i2 = D.shard_batch(n_pred_und, nb, step, seed=2, replicate=replicate).pin_memory()
    y = torch.cat((torch.ones(nb), torch.zeros(nb))).unsqueeze(-1).pin_memory()
    return i1, i2, y


# ------------------------------------------------------------------------------ clocks

class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region, in-process through NVML (pynvml) every
    50 ms - forking nvidia-smi from a process with a CUDA context stalls the launching thread for tens of ms."""

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _run(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((clk, rs))
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        if self.h is not None:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.h is not None:
            self.t.join(timeout=2)

    def summary(self):
        if self.h is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = [k for k, b in bits.items() if any(r & b for _, r in self.rows)]
        return {"sm_mhz": statistics.median(c for c, _ in self.rows), "sm_max_mhz": int(self.max), "reasons": reasons,
                "samples": len(self.rows), "how": "pynvml, 50 ms period, timed region only"}


# ------------------------------------------------------------------------------ CPU baseline (oracle port)

def cpu_baseline_sample(workload, hidden, seed=0, steps=2, budget_s=25.0):
    """The reference CPU path (oracle port: vectorised get_ei2/sample_block + LocalWLNet fwd/BCE/bwd with
    PyG semantics, torch CPU, all host threads) on a bounded sample of the same workload family."""
    from oracle import twowl_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    rng = np.random.default_rng(seed)
    if workload == "cora":
        n, und = 2708, rng.integers(0, 2708, size=(2, 5278))
        desc = "full cora-scale graph (2708 nodes, 5278 edge samples)"
    else:
        scale = 11 if workload == "rmat" else 12
        ef = 16 if workload == "rmat" else 5
        n = 1 << scale
        a, b, c, _ = WORKLOADS[workload][2]
        s = np.zeros(n * ef, dtype=np.int64)
        d = np.zeros(n * ef, dtype=np.int64)
        for _ in range(scale):
            r = rng.random(n * ef)
            s = s * 2 + (r >= a + b)
            d = d * 2 + (((r >= a) & (r < a + b)) | (r >= a + b + c))
        perm = rng.permutation(n)
        und = np.stack([perm[s], perm[d]])
        desc = f"R-MAT scale {scale} (same a,b,c,d; {n} nodes, {n * ef} edge samples) - the explicit [2,T] index the " \
               f"reference needs does not fit host RAM at the full size"
    pos, pred = O.synthetic_split(n, und, seed)
    E = pos.shape[1]
    nb = max(2, (E // 2) // 10)
    idx1 = O.double(rng.permutation(E // 2)[:nb], for_index=True)
    idx2 = O.double(rng.permutation(pred.shape[1] // 2)[:nb], for_index=True) + E
    pos1 = torch.from_numpy(np.concatenate([pos.T, pred.T]))
    y = torch.cat((torch.ones(nb), torch.zeros(nb))).unsqueeze(-1)
    ei2 = O.get_ei2(n, pos, pred)
    sd = O.init_state_dict(int(O.degree(pos, n).max()), hidden, hidden, 1, 1, seed=0)
    times, sb_times = [], []
    t_all = time.perf_counter()
    for it in range(steps + 1):
        t0 = time.perf_counter()
        ei_new, x_new, ei2_new = O.sample_block(idx1, n, pos, ei2)
        t1 = time.perf_counter()
        O.fwd_bwd(sd, torch.from_numpy(x_new), torch.from_numpy(ei_new), pos1, torch.from_numpy(np.concatenate([idx1, idx2])),
                  ei2_new, y)
        t2 = time.perf_counter()
        if it > 0:                      # first iteration = warm-up
            times.append(t2 - t1)
            sb_times.append(t1 - t0)
        if time.perf_counter() - t_all > budget_s and len(times) >= 1:
            break
    med = statistics.median(times)
    return {"value": 2 * nb / med, "unit": "target-links/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{desc}; T={ei2.shape[1]} wedges, {2 * nb} target links/step, hidden {hidden}, "
                      f"fwd+bwd median of {len(times)} = {med * 1e3:.1f} ms (+ sample_block {statistics.median(sb_times) * 1e3:.1f} ms)",
            "ms_per_step": med * 1e3, "links_per_step": 2 * nb}


def same_config_cora(dev, hidden=64, steps=20, warmup=5, cpu_steps=5):
    """BASELINE configs[1] on BOTH arms: one host-generated Cora-scale graph (2708 nodes, 5278 uniform edge samples, seed 0),
    the same doubled layout, weights (oracle init, seed 0) and per-step batches (10 % of the undirected edges + as many
    negatives, train.py:16-23). CPU = the oracle port of the reference path (explicit [2,T] index, sample_block, forward, BCE,
    backward: train.py:32-38) on all host threads; GPU = the drop-in API, device-resident (`value`), from host buffers with the
    loss read back every step (`e2e`), and with the step replayed as one CUDA graph (`graph_value`)."""
    from oracle import twowl_oracle as O
    import TwoWL.model.model as model
    import TwoWL.utils as U
    n = 2708
    rng = np.random.default_rng(0)
    pos, pred = O.synthetic_split(n, rng.integers(0, n, size=(2, 5278)), 0)
    E, P = pos.shape[1], pred.shape[1]
    nb = max(2, (E // 2) // 10)
    batches = [(rng.permutation(E // 2)[:nb], rng.permutation(P // 2)[:nb]) for _ in range(steps + warmup)]
    pos1 = np.concatenate([pos.T, pred.T])
    y = torch.cat((torch.ones(nb), torch.zeros(nb))).unsqueeze(-1)
    sd = O.init_state_dict(int(O.degree(pos, n).max()), hidden, hidden, 1, 1, seed=0)
    # ---- CPU arm
    torch.set_num_threads(os.cpu_count() or 1)
    ei2 = O.get_ei2(n, pos, pred)
    pos1_t = torch.from_numpy(pos1)
    cpu_ms = []
    for i in range(cpu_steps + 1):
        i1, i2 = batches[i]
        t0 = time.perf_counter()
        idx1 = O.double(i1, for_index=True)
        idx2 = O.double(i2, for_index=True) + E
        ei_new, x_new, ei2_new = O.sample_block(idx1, n, pos, ei2)
        O.fwd_bwd(sd, torch.from_numpy(x_new), torch.from_numpy(ei_new), pos1_t, torch.from_numpy(np.concatenate([idx1, idx2])), ei2_new, y)
        if i > 0:
            cpu_ms.append((time.perf_counter() - t0) * 1e3)
    cpu_med = statistics.median(cpu_ms)
    # ---- GPU arm
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    dpos, dpred, dpos1, dy = d(pos), d(pred), d(pos1), y.to(dev)
    dei2 = U.get_ei2(n, dpos, dpred)
    mod = model.LocalWLNet(sd["emb.0.weight"].shape[0] - 1, False, None, hidden, hidden, 1, 1, 0., 0., 0., 0., 0., 0.)
    mod.load_state_dict(sd)
    mod = mod.to(dev).train()
    host = [(torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()) for a, b in batches]

    def prepare(b):
        i1, i2 = (t.to(dev, non_blocking=True) for t in b)
        idx1 = U.double(i1, for_index=True)
        idx2 = U.double(i2, for_index=True) + E
        ei_new, x_new, ei2_new = U.sample_block(idx1, n, dpos, dei2)
        return x_new, ei_new, torch.cat((idx1, idx2)), ei2_new

    def step(inp):
        for p_ in mod.parameters():
            p_.grad = None
        loss = torch.nn.functional.binary_cross_entropy_with_logits(mod(inp[0], inp[1], dpos1, inp[2], inp[3]), dy)
        loss.backward()
        return loss

    inputs = [prepare(b) for b in host]
    for i in range(warmup):
        step(inputs[i])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        step(inputs[warmup + i])
    b.record()
    torch.cuda.synchronize()
    res_ms = a.elapsed_time(b) / steps
    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    a.record()
    for i in range(steps):
        loss = step(prepare(host[warmup + i]))
        host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    b.record()
    torch.cuda.synchronize()
    e2e_ms = a.elapsed_time(b) / steps
    graph_ms = None
    try:
        from twowl_b200.graphed import GraphedTrainStep
        del loss, inputs
        mod2 = model.LocalWLNet(sd["emb.0.weight"].shape[0] - 1, False, None, hidden, hidden, 1, 1, 0., 0., 0., 0., 0., 0.)
        mod2.load_state_dict(sd)      # a fresh module: no gradient accumulators that the eager steps created on another stream
        mod2 = mod2.to(dev).train()
        gs = GraphedTrainStep(mod2, n, dpos, dpos1, dei2, n_block=2 * nb, n_links=2 * nb)
        gin = []
        for bb in host:
            i1, i2 = (t.to(dev) for t in bb)
            idx1 = U.double(i1, for_index=True)
            gin.append((idx1, torch.cat((idx1, U.double(i2, for_index=True) + E))))
        for i in range(warmup):
            gs(gin[i][0], gin[i][1], dy)
        torch.cuda.synchronize()
        a.record()
        for i in range(steps):
            gs(gin[warmup + i][0], gin[warmup + i][1], dy)
        b.record()
        torch.cuda.synchronize()
        graph_ms = a.elapsed_time(b) / steps
    except Exception as ex:   # the replayed step is an extra; the eager numbers above stand without it
        graph_ms = f"unavailable: {type(ex).__name__}: {ex}"[:200]
    links = 2 * nb
    gpu = {"value": links / (res_ms * 1e-3), "ms_per_step": res_ms, "e2e": links / (e2e_ms * 1e-3), "e2e_ms_per_step": e2e_ms}
    if isinstance(graph_ms, float):
        gpu["graph_value"], gpu["graph_ms_per_step"] = links / (graph_ms * 1e-3), graph_ms
    else:
        gpu["graph_value"] = graph_ms
    return {"workload": "cora", "nodes": n, "E": E, "R": E + P, "wedges_T": int(ei2.shape[1]), "hidden": hidden,
            "target_links_per_step": links, "unit": "target-links/s",
            "step": "double + sample_block + forward + BCE + backward (train.py:29-38) on the same graph, weights and batches",
            "gpu": gpu,
            "cpu": {"value": links / (cpu_med * 1e-3), "ms_per_step": cpu_med, "cores": torch.get_num_threads(), "kind": "port",
                    "steps": len(cpu_ms)},
            "e2e_ratio": (links / (e2e_ms * 1e-3)) / (links / (cpu_med * 1e-3))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _, _, _, dh = WORKLOADS[args.workload]
    hidden = args.hidden or dh
    cb = cpu_baseline_sample(args.workload, hidden, steps=max(args.steps, 1), budget_s=120.0)
    line = {"impl": "reference", "metric": "twowl_fwd_bwd_target_links_per_s", "value": cb["value"], "unit": "target-links/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "hidden": hidden, "sample": cb["sample"]},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "target-links/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DUMP_BYTES = 60 << 20          # array data; with the .npy headers a dump stays under 64 MB


def dump_outputs(arrays, out_dir):
    """Write every float32 array as out_dir/<name>.npy, at most DUMP_BYTES in all. Smaller arrays are written whole; an array
    larger than an equal share of what is left keeps that share of its elements, at positions drawn with a fixed seed (sorted,
    from the flattened array): the same positions on every run with the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    left, sampled = DUMP_BYTES // 4, []
    by_size = sorted(arrays.items(), key=lambda kv: kv[1].size)
    for i, (name, a) in enumerate(by_size):
        keep = min(a.size, left // (len(by_size) - i))
        left -= keep
        if keep < a.size:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
            sampled.append(name)
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"dump-outputs: {len(arrays)} arrays ({total / 2**20:.1f} MiB) -> {out_dir}"
          + (f"; sampled: {', '.join(sampled)}" if sampled else ""), file=sys.stderr)


# ------------------------------------------------------------------------------ our arm

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rmat", choices=list(WORKLOADS))
    ap.add_argument("--hidden", type=int, default=0)
    ap.add_argument("--scale", type=int, default=0, help="override the R-MAT scale (debug)")
    ap.add_argument("--samples", type=int, default=0, help="override the R-MAT edge samples (debug)")
    ap.add_argument("--pair-path", default="auto", choices=["auto", "structured", "explicit"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inplace-backward", action="store_true", help="reuse the forward's [R,C] buffers in the backward (ops.INPLACE_BACKWARD)")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the row-sharded (strong scaling) measurement")
    ap.add_argument("--graph", action="store_true",
                    help="replay the step (edge blocking + forward + BCE + backward) as ONE captured CUDA graph "
                         "(twowl_b200.graphed): for the launch-bound small workloads")
    ap.add_argument("--shard", default="links", choices=["links", "rows"],
                    help="multi-GPU: 'links' = every rank steps its own disjoint slice of the target links (weak scaling, the "
                         "default); 'rows' = ONE step whose pair rows are cut into row blocks over the ranks (strong scaling, "
                         "twowl_b200.rowshard)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's loss, logits and parameter gradients as DIR/<name>.npy (float32, at most "
                         "64 MB in all: larger outputs keep a fixed seeded sample of their elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from twowl_b200 import ops
    import TwoWL.model.model as model
    import TwoWL.utils as U

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL's kernels on a high-priority stream: the row-sharded step overlaps the all-reduce of one node range with the
        # gather kernel of the next, and a pending collective should take the SM resources a finished gather frees before the
        # next gather's CTAs do (TWOWL_NCCL_HIGH_PRIO=0 turns it off)
        opts = None
        if os.environ.get("TWOWL_NCCL_HIGH_PRIO", "1") != "0":
            try:
                opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            except Exception:   # noqa: BLE001 - an older torch without the option
                opts = None
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    hidden = args.hidden or WORKLOADS[args.workload][3]
    args.warmup = max(args.warmup, 3)
    if args.inplace_backward or (args.workload == "rmat" and hidden >= 128 and not args.scale):
        ops.INPLACE_BACKWARD = True    # dO over O, dH over H: the 3 x [R,C] footprint that lets hidden 128 fit one GPU at R = 60 M

    # ---- dataset (resident, like the reference's `dataset` object after .to(device)) ----
    g = make_graph(args.workload, 0, dev, args.scale or None, args.samples or None)
    n, pos, pred, pos1 = g["n"], g["pos"], g["pred"], g["pos1"]
    E, P = pos.shape[1], pred.shape[1]
    x_full = U.degree(pos, n)
    max_x = int(x_full.max().item())
    explicit = args.pair_path == "explicit"
    ei2 = U.get_ei2(n, pos, pred) if explicit else U.get_ei2_implicit(n, pos, pred)
    from twowl_b200 import dist as D

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def measure(rows: bool, keep_outputs: bool = False):
        """One measurement of K steps. rows = False: every rank steps its own disjoint slice of the target links (data parallel,
        weak scaling); rows = True: ONE batch per step, its pair rows cut into row blocks over the ranks (strong scaling).
        keep_outputs: also return the last timed step's loss, logits and gradients as host arrays."""
        nb = max(2, g["und"] // 10)
        if world > 1 and not rows:         # the slices of the ranks are disjoint: cap the global batch at the id range
            nb = min(nb, g["und"] // world, (P // 2) // world)
        L = 2 * nb
        torch.manual_seed(0)
        mod = model.LocalWLNet(max_x, False, None, hidden, hidden, 1, 1, 0., 0., 0., 0., 0., 0.).to(dev).train()
        mod.pair_path = args.pair_path
        if rows:
            from twowl_b200.rowshard import RowShard
            mod.row_shard = RowShard()
        params = list(mod.parameters())

        def sync_grads():
            if world > 1:
                D.allreduce_grads(params)   # one NCCL all-reduce of the flat gradient buffer, written back into .grad

        gstep = None
        if args.graph:
            if rows or explicit:
                raise SystemExit("--graph covers the structured single-process step (not --shard rows / --pair-path explicit)")
            from twowl_b200.graphed import GraphedTrainStep
            gstep = GraphedTrainStep(mod, n, pos, pos1, ei2, n_block=2 * nb, n_links=L)

        def prepare(batch, eager=False):
            i1, i2, y = (t.to(dev, non_blocking=True) for t in batch)
            idx1 = U.double(i1, for_index=True)
            idx2 = U.double(i2, for_index=True) + E
            if gstep is not None and not eager:  # edge blocking happens inside the captured step
                return idx1, torch.cat((idx1, idx2)), y
            ei_new, x_new, ei2_new = U.sample_block(idx1, n, pos, ei2)
            return x_new, ei_new, torch.cat((idx1, idx2)), ei2_new, y

        kept = {}

        def fwd_bwd(inp, keep=False):
            """keep: also hold on to this step's loss and logits in `kept` (--dump-outputs)."""
            if len(inp) == 3:
                loss = gstep(*inp)
                sync_grads()
                if keep:
                    kept.update(loss=loss, logits=gstep.logits)
                return loss
            x_new, ei_new, idx, ei2_new, y = inp
            for p_ in mod.parameters():
                p_.grad = None
            out = mod(x_new, ei_new, pos1, idx, ei2_new)
            loss = torch.nn.functional.binary_cross_entropy_with_logits(out, y)
            loss.backward()
            sync_grads()
            if keep:
                kept.update(loss=loss, logits=out)
            return loss

        batches = [draw_batch(g["und"], P // 2, nb, i, replicate=rows) for i in range(args.steps + args.warmup)]
        # ---- device-resident timing: K steps of fwd+bwd, inputs prepared beforehand ----
        inputs = [prepare(b) for b in batches]
        for i in range(args.warmup):
            fwd_bwd(inputs[i])
        barrier()
        launches0 = ops.launches()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        with ClockSampler(local) as clocks:
            for i in range(args.steps):
                l2_flush.fill_(i & 255)     # evict L2 between timed steps (inputs also exceed L2 at rmat/collab size)
                ev[i][0].record()
                fwd_bwd(inputs[args.warmup + i], keep=keep_outputs and i + 1 == args.steps)
                ev[i][1].record()
            barrier()
        launches = ops.launches() - launches0
        step_ms = [a.elapsed_time(b) for a, b in ev]
        outputs = None
        if keep_outputs:                # copied now: the next steps overwrite the gradients (and a replayed graph its logits)
            named = list(kept.items()) + [("grad." + k, p.grad) for k, p in mod.named_parameters() if p.grad is not None]
            outputs = {k: v.detach().float().cpu().numpy() for k, v in named}
            kept.clear()
        # ---- the same K steps once more with CUDA events around every kernel group (roofline); kept out of the timed
        #      region above because two extra events per op are not free for the launch-bound small workloads ----
        if gstep is not None:   # a replayed graph has no per-op events: the per-kernel roofline comes from the eager path
            inputs = [prepare(b, eager=True) for b in batches]
        ops.profile_start()
        for i in range(args.steps):
            l2_flush.fill_(i & 255)
            fwd_bwd(inputs[args.warmup + i])
        barrier()
        prof = ops.profile_stop()
        total_ms = D.max_over_ranks(sum(step_ms), dev)
        del inputs

        # ---- sample_block alone (per-step, on the path; reported separately as SURVEY 8(d) asks) ----
        sb_ev = []
        for i in range(min(5, args.steps)):
            i1, i2, y = (t.to(dev) for t in batches[i])
            idx1 = U.double(i1, for_index=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            U.sample_block(idx1, n, pos, ei2)
            b.record()
            sb_ev.append((a, b))
        torch.cuda.synchronize()
        sb_ms = statistics.median(a.elapsed_time(b) for a, b in sb_ev)

        # ---- end to end from host buffers: H2D batch -> sample_block -> fwd -> loss -> bwd -> D2H loss ----
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
        e0.record()
        for i in range(args.steps):
            loss = fwd_bwd(prepare(batches[args.warmup + i]))
            host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()   # the reference reads loss.item() every step (train.py:47)
        e1.record()
        barrier()
        e2e_ms = D.max_over_ranks(e0.elapsed_time(e1), dev)
        h2d = sum(t.numel() * t.element_size() for t in batches[0])
        links = L * (1 if rows else world) * args.steps
        comm = None
        if rows:
            from twowl_b200 import rowshard
            comm = rowshard.comm_summary()
        del mod, gstep
        return dict(total_ms=total_ms, e2e_ms=e2e_ms, launches=launches, prof=prof, sb_ms=sb_ms, links=links, L=L, h2d=h2d,
                    clocks=clocks.summary(), comm=comm, outputs=outputs)

    rows_main = args.shard == "rows" and world > 1
    m = measure(rows_main, keep_outputs=bool(args.dump_outputs) and rank == 0)
    strong = None
    if world > 1 and not rows_main and not args.graph and not explicit and not args.no_strong:
        # north_star's partition, measured in the same run: one batch per step, pair rows cut over the ranks
        from twowl_b200 import graph as G
        G.clear_cache()
        torch.cuda.empty_cache()
        ms_ = measure(True)
        ops_ms = {}
        for name, _, ms in ms_["prof"]:
            ops_ms[name] = ops_ms.get(name, 0.0) + ms
        strong = {"scaling": "strong", "value": ms_["links"] / (ms_["total_ms"] * 1e-3), "unit": "target-links/s",
                  "per_op_ms_per_step_rank0": {k: round(v / args.steps, 3) for k, v in sorted(ops_ms.items(), key=lambda kv: -kv[1])},
                  "ms_per_step": ms_["total_ms"] / args.steps, "target_links_per_step": ms_["L"],
                  "e2e": {"value": ms_["links"] / (ms_["e2e_ms"] * 1e-3), "ms_per_step": ms_["e2e_ms"] / args.steps},
                  "gpu_launches": ms_["launches"], "collectives": ms_["comm"],
                  "parallelism": f"rows{world}: ONE batch per step, its pair rows cut into {world} row blocks (twowl_b200.rowshard)"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total_ms, e2e_ms, prof, launches = m["total_ms"], m["e2e_ms"], m["prof"], m["launches"]
    if args.dump_outputs:
        dump_outputs(m["outputs"], args.dump_outputs)

    # ---- roofline of the dominant kernel ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    by_op = {}
    for name, nbytes, ms in prof:
        d = by_op.setdefault(name, [0, 0.0, 0.0])
        d[0] += 1
        d[1] += nbytes
        d[2] += ms
    tot_kernel_ms = sum(d[2] for d in by_op.values()) or 1.0
    top = max(by_op.items(), key=lambda kv: kv[1][2]) if by_op else ("none", [1, 0.0, 1.0])
    tname, (tcnt, tbytes, tms) = top[0], top[1]
    achieved = (tbytes / tcnt) / (tms / tcnt * 1e-3) / 1e9 if tms > 0 else 0.0
    agg_bytes = sum(d[1] for d in by_op.values())
    traffic = traffic_table(f"{args.workload}/hidden{hidden}")

    def dram(name, avg_ms):
        t = traffic.get(name)
        return None if t is None or avg_ms <= 0 else round(t / (avg_ms * 1e-3) / 1e9 / peak, 4)

    per_op = {}
    for k, v in sorted(by_op.items(), key=lambda kv: -kv[1][2]):
        gbps = v[1] / (v[2] * 1e-3) / 1e9 if v[2] > 0 else None
        e = {"n": v[0], "ms": round(v[2], 3), "GBps": round(gbps, 1) if gbps else None, "frac": round(gbps / peak, 4) if gbps else None,
             "frac_dram": dram(k, v[2] / v[0])}
        if gbps and gbps > 1.2 * peak:
            e["l2_served"] = True   # algorithmic bytes count every gathered row as read; above the DRAM peak they came from L2
        per_op[k] = e
    roofline = {"bound": "hbm", "kernel": tname, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic.get(tname), "frac_dram": dram(tname, tms / tcnt),
                "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed "
                                  "ncu --set full capture, used only while the kernel's source file hashes to what was captured",
                "peak_source": peak_src,
                "launches": tcnt, "avg_ms": round(tms / tcnt, 4), "share_of_kernel_time": round(tms / tot_kernel_ms, 4),
                "algorithmic_bytes_per_launch": int(tbytes / tcnt),
                "note": "achieved / frac = algorithmic bytes (every gathered row counted as read, SURVEY 8(d)) / measured time; rows "
                        "served from L1/L2 make it exceed what DRAM moved - frac_dram = measured DRAM bytes / the same time / peak",
                "all_kernels_algorithmic_GBps": round(agg_bytes / (tot_kernel_ms * 1e-3) / 1e9, 1),
                "per_op": per_op}

    cb = sc = None
    if not args.no_cpu_baseline and world == 1:   # the CPU legs run at N = 1 only
        cb = cpu_baseline_sample(args.workload, hidden)
        cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cb["note"] = "a bounded sample of the workload family, NOT the GPU arm's graph: see same_config for a like-for-like ratio"
        sc = same_config_cora(dev)

    links, L = m["links"], m["L"]
    par = (f"rows{world}: ONE batch per step, its pair rows cut into {world} row blocks (twowl_b200.rowshard)") if rows_main else (
        f"dp{world}: target links sharded over ranks (disjoint slices of one global batch per step), graph replicated, one "
        "all-reduce of the parameter gradients")
    line = {
        "metric": "twowl_fwd_bwd_target_links_per_s", "value": links / (total_ms * 1e-3), "unit": "target-links/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "strong" if rows_main else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "nodes": n, "undirected_edges": g["und"], "E": E, "R": E + P,
                   "hidden": hidden, "depth1": 1, "depth2": 1, "target_links_per_step": L, "pair_path": args.pair_path,
                   "wedges_T": ei2.shape[1] if explicit else None, "cuda_graph": bool(args.graph), "inplace_backward": bool(ops.INPLACE_BACKWARD), "l2": "256 MiB flush write between timed steps; "
                   "activations exceed L2", "parallelism": par},
        "clocks": m["clocks"],
        "e2e": {"value": links / (e2e_ms * 1e-3), "unit": "target-links/s", "h2d_bytes_per_step": m["h2d"],
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps, "includes": "H2D batch ids+labels, double, "
                "sample_block, forward, BCE, backward, D2H loss"},
        "sample_block_ms": m["sb_ms"],
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": cb,
        "same_config": sc,
    }
    if rows_main:
        line["collectives"] = m["comm"]
    if strong is not None:
        line["strong"] = strong
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------ measured DRAM traffic (ncu)

_OP_SOURCE = {"pair_conv": "pair_conv.cu", "pair_dw_gn": "dw_tc.cu", "pair_dw": "dw_tc.cu", "seg_reduce": "agg.cu",
              "pair_init_fwd": "pair_ops.cu", "gn2_readout_fwd": "norm.cu", "gn2_readout_bwd_prepare": "norm.cu"}


def source_sha16(op):
    """sha256 (16 hex digits) of the CUDA source file the op's kernel lives in + common.cuh: what a traffic capture is stamped with."""
    import hashlib
    h = hashlib.sha256()
    for f in (_OP_SOURCE.get(op, ""), "common.cuh"):
        path = os.path.join(ROOT, "link-prediction-gnn_b200", "csrc", f)
        if f and os.path.isfile(path):
            h.update(open(path, "rb").read())
    return h.hexdigest()[:16]


def traffic_table(config_key):
    """{op: measured DRAM bytes per launch} for this workload / width from profiles/traffic.json (written by
    tools/capture_traffic.py from an `ncu --set full` capture). An entry is used only if the kernel's source still hashes to the
    stamp taken at capture time: a changed kernel reports traffic null instead of a stale constant."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}
    out = {}
    for op, per_cfg in tj.items():
        e = per_cfg.get(config_key) if isinstance(per_cfg, dict) else None
        if e and e.get("source_sha16") == source_sha16(op):
            out[op] = e["bytes_per_launch"]
    return out


if __name__ == "__main__":
    main()
