#!/usr/bin/env python
"""bench.py — edges/s through the fused gather-message-scatter layer (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

Workload (N=1 default) = BASELINE.json configs[1]: RGCN, synthetic Erdos-Renyi graph, 1M nodes /
20M edges / 4 edge types, hidden_dim=256, one B200.  A "step" is ONE message-passing layer forward
over the whole batch (every edge sends one message); value = edges / step time.  Inputs (1 GB node
table) exceed the 126 MB L2, so no flush is needed between timed iterations.

Printed JSON line keys: see the task contract; `roofline` is the algorithmic bytes of the layer
(SURVEY.md §8d formula) over the device time of the layer, against MEASURED_PEAKS.json;
`cpu_baseline` is the torch-CPU restatement of the reference op sequence (oracle/torch_cpu_port.py)
on a bounded edge sample; `e2e` goes through the public layer API with pinned HOST buffers
(H2D of node states + adjacency, prepare, layer, D2H of the result inside the timed region).
Multi-GPU: every rank processes its own batch of the same shape (partitions of a disjoint-graph
batch need no collective, SURVEY.md §8e) -> "scaling": "weak".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs; the default (N=1) bench line is cfg2, the others are recorded with --workload.
    "cfg2": dict(V=1_000_000, E=[5_000_000] * 4, H=256, kind="rgcn", graph="er",
                 desc="RGCN synthetic Erdos-Renyi 1M nodes / 20M edges / 4 edge types, hidden_dim=256 "
                      "(BASELINE.json configs[1])"),
    "cfg1": dict(V=8000, E=[8000, 115_200, 115_200], H=320, kind="rgcn", graph="ppi",
                 desc="RGCN PPI-shaped hidden_dim=320, 3 edge types, 8000 nodes (BASELINE.json configs[0])"),
    "cfg3": dict(V=2_000_000, E=[20_000_000] * 3, H=128, kind="rgat", graph="powerlaw", params=dict(num_heads=4),
                 desc="RGAT 4-head synthetic power-law 2M nodes / 60M edges / 3 edge types, hidden_dim=128 "
                      "(BASELINE.json configs[2])"),
    "cfg4": dict(V=500_000, E=[500_000, 600_000, 250_000, 50_000, 100_000], H=128, kind="ggnn", graph="er",
                 desc="GGNN QM9-shaped 500k nodes / 1.5M edges / 5 edge types, hidden_dim=128 (BASELINE.json configs[3])"),
    "cfg5_shard": dict(V=2_000_000, E=[5_333_333] * 6, H=320, kind="gnn_film", graph="er",
                       desc="GNN-FiLM 1/8 shard of BASELINE.json configs[4]: 2M nodes / 32M edges / 6 edge types, hidden_dim=320"),
    "cfg5": dict(V=16_000_000, E=[42_666_666] * 6, H=320, kind="gnn_film", graph="er",
                 desc="GNN-FiLM synthetic 16M nodes / 256M edges / 6 edge types, hidden_dim=320, target-range sharded over "
                      "8 GPUs with one all-gather per layer (BASELINE.json configs[4]; sharded leg only)"),
    "h320": dict(V=1_000_000, E=[6_666_667] * 3, H=320, kind="rgcn", graph="er",
                 desc="RGCN synthetic Erdos-Renyi 1M nodes / 20M edges / 3 edge types, hidden_dim=320 "
                      "(north_star hidden size on a graph that exceeds L2)"),
    "tiny": dict(V=20_000, E=[100_000] * 4, H=256, kind="rgcn", graph="er", desc="smoke-sized cfg2"),
}
METRIC = "edges/sec (fused gather-msg-scatter)"
E2E_DEPTH = int(os.environ.get("TFGNN_B200_E2E_DEPTH", "3"))   # steps in flight in the end-to-end leg (runtime.HostPipeline)
DUMP_ARRAY_BYTES = 16 << 20   # --dump-outputs, per workload: the three workloads of a default run stay under DUMP_TOTAL_BYTES
DUMP_TOTAL_BYTES = 64 << 20


def dump_rows(V, H):
    """Rows of a [V, H] float32 layer output that --dump-outputs writes: all of them when they fit DUMP_ARRAY_BYTES, else a
    fixed seeded sample in ascending order, so that every run (and every build) writes the same rows."""
    n = DUMP_ARRAY_BYTES // (4 * H)
    if V <= n:
        return np.arange(V, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(V, size=n, replace=False))


def write_outputs(dirname, outputs):
    """One DIR/<workload>.npy per measured workload: the sampled rows of its last timed layer call."""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_TOTAL_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_TOTAL_BYTES}-byte limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(dirname, f"{name}.npy"), a)


def algorithmic_bytes(kind, V, E_list, D, H, params):
    """SURVEY.md §8d: sum_l E_l*(8+4*D_g) + 4VH + 4*sum(weights) [+4LV normalise] [+4VD target input]
    [+8VH GGNN GRU reads]; D_g = D (H + K source scores for RGAT)."""
    L, M = len(E_list), sum(E_list)
    if kind == "rgat":
        K = params["num_heads"]
        return M * (8 + 4 * (H + K)) + 4 * V * H + 4 * L * (D * H + 2 * H) + 4 * V * D
    b = M * (8 + 4 * D) + 4 * V * H + 4 * L * D * H
    if params.get("normalize_by_num_incoming"):
        b += 4 * L * V
    if kind == "gnn_film":
        b += 4 * L * D * 2 * H + 4 * V * D
    if kind == "ggnn":
        b += 8 * V * H + 4 * (2 * H * 3 * H + 6 * H)
    return b


def dense_flops(kind, V, E_list, D, H, params):
    """fp32-equivalent FLOPs of the node-level contractions of one layer in the formulation the kernels use (DESIGN.md §3):
    RGCN/GGNN messages 2*V*L*D*H, + GGNN GRU 2*V*(D+H)*3H, RGAT projection 2*V*L*D*H, GNN-FiLM messages + gamma + beta =
    3 * 2*V*L*D*H.  Each product costs three tf32 MMAs (3xTF32) on the tensor cores."""
    L = len(E_list)
    base = 2.0 * V * L * D * H
    if kind == "ggnn":
        return base + 2.0 * V * (D + H) * 3 * H
    if kind == "gnn_film":
        return 3.0 * base
    return base


def load_tensor_peak():
    """Measured dense tf32 peak = half the measured bf16 cuBLAS peak of MEASURED_PEAKS.json (TFLOP/s), else nominal 1100/... fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["bf16_tflops"]) / 2.0, "measured bf16_tflops / 2 (MEASURED_PEAKS.json)"
    return 1590.0 / 2.0, "fallback bf16 1.59 PFLOP/s / 2 (B200_PROFILING.md)"


def make_inputs(wl, seed):
    rng = np.random.default_rng(seed)
    V, H = wl["V"], wl["H"]
    adjs = []
    for l, E in enumerate(wl["E"]):
        if wl["graph"] == "ppi" and l == 0:
            ids = np.arange(V, dtype=np.int32)
            adjs.append(np.stack([ids, ids], axis=1))
        elif wl["graph"] == "powerlaw":
            # target in-degrees ~ Zipf(2.1) capped at 1e5 (SURVEY.md §8d), sources uniform
            deg = np.minimum(rng.zipf(2.1, size=V), 100_000).astype(np.float64)
            tgt = rng.choice(V, size=E, p=deg / deg.sum()).astype(np.int32)
            src = rng.integers(0, V, size=E, dtype=np.int32)
            adjs.append(np.stack([src, tgt], axis=1))
        else:
            adjs.append(rng.integers(0, V, size=(E, 2), dtype=np.int32))
    h = rng.random((V, H), dtype=np.float32) * 2.0 - 1.0           # U(-1,1): post-tanh range
    lim = np.sqrt(6.0 / (H + H))
    weights = [((rng.random((H, H), dtype=np.float32) * 2.0 - 1.0) * lim).astype(np.float32) for _ in wl["E"]]
    return h, adjs, weights


def load_traffic(workload, path):
    """DRAM bytes per launch of the dominant kernel.  NOT measured in this run (ncu replays kernels; a number printed
    under a profiler is never a bench value): a STATIC figure from the committed ncu --set full capture of the same
    command, labelled with the file and the commit it was taken at.  (None, reason) when no capture exists."""
    for fname in ("traffic_r2.json", "traffic_r1.json"):
        p = os.path.join(ROOT, "profiles", fname)
        try:
            with open(p) as f:
                e = json.load(f).get(f"{workload}:{path}")
        except Exception:
            continue
        if e is not None:
            src = f"static, from {e.get('source', 'profiles/' + fname)} @ {e.get('commit', 'round-1 kernel')}"
            return int(e["dram_bytes_read"]) + int(e["dram_bytes_write"]), src
    return None, "no ncu --set full capture committed for this workload/path"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.

    NVML (nvidia-ml-py) polled from a thread every 10 ms; `nvidia-smi -lms` in a subprocess if NVML cannot be
    loaded.  Samples are stamped with time.monotonic() and only those between begin() and end() are reported
    (all samples since start() if the window caught none, noted in "window")."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None
        self.thread = None
        self.samples = []          # (t, sm_mhz, max_mhz, reasons tuple)
        self.t_begin = None
        self.t_end = None
        self._stop = False

    def _nvml_loop(self, nv, handle):
        bits = []
        for name, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
            alt = attr.replace("ClocksEventReason", "ClocksThrottleReason")
            val = getattr(nv, attr, getattr(nv, alt, None))
            if val is not None:
                bits.append((name, val))
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons",
                              getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None))
        mx = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM))
                mask = get_reasons(handle) if get_reasons else 0
                self.samples.append((time.monotonic(), sm, mx, tuple(n for n, b in bits if mask & b)))
            except Exception:
                pass
            time.sleep(0.010)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            idx = self.gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.gpu_index < len(ids) and ids[self.gpu_index].isdigit():
                    idx = int(ids[self.gpu_index])
            handle = nv.nvmlDeviceGetHandleByIndex(idx)
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def begin(self):
        self.t_begin = time.monotonic()

    def end(self):
        self.t_end = time.monotonic()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            rows = self.samples
            window = "timed region"
            if self.t_begin is not None and self.t_end is not None:
                inside = [r for r in rows if self.t_begin <= r[0] <= self.t_end]
                if inside:
                    rows = inside
                else:
                    window = "warm-up + timed region (no sample fell inside the timed region)"
            if rows:
                reasons = set()
                for r in rows:
                    reasons.update(r[3])
                out.update(sm_mhz=float(np.median([r[1] for r in rows])), sm_max_mhz=float(max(r[2] for r in rows)),
                           reasons=sorted(reasons), samples=len(rows), source="nvml, 10 ms poll", window=window)
            return out
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
        except Exception:
            return out
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, val in zip(names, r[5:9]):
                    if val.strip().lower() == "active":
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm), source="nvidia-smi -lms 50", window="warm-up + timed region")
        return out


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    return rank, world, local


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_ranks_true(flag, world):
    """Logical AND of a per-rank condition (collective)."""
    if world == 1:
        return bool(flag)
    import torch
    import torch.distributed as dist
    t = torch.tensor([1 if flag else 0], dtype=torch.int32, device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


# -------------------------------------------------------------------------------------------
def run_cpu_port(wl, h, adjs, weights, sample_edges, steps, warmup, threads):
    """Time the torch-CPU restatement of the reference op order on a bounded edge sample."""
    import torch
    from oracle.torch_cpu_port import rgcn_layer_reference_order
    torch.set_num_threads(threads)
    M = sum(a.shape[0] for a in adjs)
    frac = min(1.0, sample_edges / M)
    s_adjs = [torch.from_numpy(a[: max(1, int(round(a.shape[0] * frac)))]) for a in adjs]
    ht = torch.from_numpy(h)
    wt = [torch.from_numpy(w) for w in weights]
    m_sample = sum(int(a.shape[0]) for a in s_adjs)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        rgcn_layer_reference_order(ht, s_adjs, wt)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = float(sum(times))
    return m_sample * len(times) / total, m_sample, total / len(times)


def best_cpu_threads(wl, h, adjs, weights):
    """torch-CPU scaling of the gather / index_add ops is poor on many-core hosts (NUMA): calibrate a few
    thread counts on a small sample and use the fastest, as a user of the reference would."""
    total = os.cpu_count() or 1
    cands = sorted({c for c in (total, 64, 32, 16, 8) if c <= total}, reverse=True)
    M = sum(a.shape[0] for a in adjs)
    best, best_rate = total, 0.0
    for c in cands:
        rate, _, _ = run_cpu_port(wl, h, adjs, weights, min(M, 200_000), 1, 1, c)
        if rate > best_rate:
            best, best_rate = c, rate
    return best, best_rate, total


def reference_arm(args, wl, rank, world):
    """--impl reference: the reference's CPU path (restated port; TF is not installable here)."""
    if rank != 0:
        return
    if wl["kind"] != "rgcn":
        print(json.dumps({"impl": "reference", "unavailable": "timed CPU port exists for the RGCN workloads only"}))
        return
    h, adjs, weights = make_inputs(wl, seed=0)
    M = sum(a.shape[0] for a in adjs)
    # calibrate threads and rate on a small sample, then size the per-step sample so the run ends within ~2 minutes
    threads, rate, host_cores = best_cpu_threads(wl, h, adjs, weights)
    budget_s = 120.0
    sample = int(min(M, max(50_000, rate * budget_s / max(1, args.steps + args.warmup))))
    eps, m_sample, t_step = run_cpu_port(wl, h, adjs, weights, sample, args.steps, args.warmup, threads)
    sample_desc = (f"first {m_sample} of {M} edges (same V={wl['V']}, H={wl['H']}, L={len(wl['E'])}), 1 layer/step, "
                   f"torch-CPU restatement of the reference op order (TensorFlow absent); fastest of "
                   f"{{all,64,32,16,8}} threads on a {host_cores}-core host")
    line = {
        "impl": "reference", "metric": METRIC, "value": eps, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "sample": sample_desc},
        "cpu_baseline": {"value": eps, "unit": "edges/s", "cores": threads, "kind": "port", "sample": sample_desc},
        "e2e": {"value": eps, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------
KERNEL_OF = {
    "rgcn": "fused_rgcn_kernel (gather ring -> TMA -> 3xTF32 tcgen05.mma cta_group::2 -> epilogue from registers) + 1 weight-pack kernel",
    "ggnn": "fused_rgcn_kernel (messages) + gemm_tc_kernel over [agg | h] with the GRU gate math in its epilogue",
    "rgat": "gemm_tc_kernel (P = h W, attention score halves in its epilogue) + rgat_warp_kernel / hub kernels (online segment softmax + weighted sum)",
    "gnn_film": "edge_reduce_kernel (A_l) + gemm_tc_kernel (FiLM parameters, messages) with the modulation in the GEMM epilogue",
}


def build_layer(wl, rank, path="auto"):
    import torch
    from tf2_gnn_b200.layers import MessagePassingInput, get_message_passing_class
    kind, H, L = wl["kind"], wl["H"], len(wl["E"])
    layer_cls = get_message_passing_class(kind)
    params = layer_cls.get_default_hyperparameters()
    params.update(wl.get("params", {}))
    params.update(hidden_dim=H, b200_path=path)
    layer = layer_cls(params)
    torch.manual_seed(1234 + rank)
    layer.build(MessagePassingInput((None, H), tuple((None, 2) for _ in range(L))))  # Glorot-uniform weights
    return layer, params


class L2Flusher:
    """Writes a buffer larger than the 126 MB L2 between timed iterations (workloads whose inputs fit L2)."""

    def __init__(self, dev, nbytes=256 << 20):
        import torch
        self.buf = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)

    def __call__(self):
        self.buf.fill_(1.0)


def time_device_resident(layer, inp, prepared, steps, warmup, flush=None):
    """ms per layer call with inputs resident in HBM: CUDA events on the launching stream.  With `flush`, every
    iteration is timed on its own (the flush runs outside the event pair) and the times are summed."""
    import torch
    for _ in range(warmup):
        out = layer(inp, prepared=prepared)
    torch.cuda.synchronize()
    if flush is None:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            out = layer(inp, prepared=prepared)
            ev[i + 1].record()
        torch.cuda.synchronize()
        per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        return ev[0].elapsed_time(ev[-1]), per_step, out
    per_step = []
    for i in range(steps):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = layer(inp, prepared=prepared)
        e1.record()
        torch.cuda.synchronize()
        per_step.append(e0.elapsed_time(e1))
    return float(sum(per_step)), per_step, out


def time_e2e(layer, h_host, adj_host, out_host, steps, world, depth=2):
    """The public call with HOST buffers: every step copies its node states + adjacency lists from pinned host memory,
    builds the per-batch CSR, runs the layer and copies the new node states back to pinned host memory.  Steps are
    software-pipelined `depth` deep on CUDA streams (runtime.HostPipeline): D2H of step i overlaps H2D of step i+1."""
    import torch
    from tf2_gnn_b200.layers import MessagePassingInput
    from tf2_gnn_b200.runtime import HostPipeline
    host_inp = MessagePassingInput(h_host, tuple(adj_host))
    outs = [out_host] + [torch.empty_like(out_host).pin_memory() for _ in range(depth - 1)]
    pipe = HostPipeline(lambda b: layer(b), depth=depth)
    for i in range(2 * depth):
        pipe.submit(host_inp, outs[i % depth])
    pipe.drain()
    torch.cuda.synchronize()
    barrier(world)
    t0 = time.perf_counter()
    for i in range(steps):
        pipe.submit(host_inp, outs[i % depth])
    pipe.drain()
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0, world)
    return dt


def measure_workload(name, args, rank, world, local, dev, headline):
    """One workload: device-resident layer time (+ roofline), optional e2e.  Returns a dict."""
    import torch
    from tf2_gnn_b200 import _ffi
    from tf2_gnn_b200.layers import MessagePassingInput
    from tf2_gnn_b200.runtime import PreparedBatch
    wl = WORKLOADS[name]
    V, H, L = wl["V"], wl["H"], len(wl["E"])
    M = sum(wl["E"])
    kind = wl["kind"]
    h_np, adjs_np, w_np = make_inputs(wl, seed=rank)
    h_host = torch.from_numpy(h_np).pin_memory()
    adj_host = [torch.from_numpy(a).pin_memory() for a in adjs_np]
    layer, params = build_layer(wl, rank, args.path)
    if kind == "rgcn":
        layer.set_weights_from_oracle_dict({"edge_mlps": [[w] for w in w_np]})
    h_dev = h_host.to(dev)
    adj_dev = tuple(a.to(dev) for a in adj_host)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    prepared = PreparedBatch(adj_dev, V)
    torch.cuda.synchronize()
    prepare_first_ms = (time.perf_counter() - t0) * 1e3
    # steady-state prepare (pool warm): CUDA events around a second build of the same CSR
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    prepared2 = PreparedBatch(adj_dev, V)
    e1.record()
    torch.cuda.synchronize()
    prepare_wall_ms = (time.perf_counter() - t0) * 1e3
    prepare_dev_ms = e0.elapsed_time(e1)
    del prepared2
    inp = MessagePassingInput(h_dev, adj_dev)
    fits_l2 = V * H * 4 <= 126e6
    flush = L2Flusher(dev) if fits_l2 else None
    sampler = ClockSampler(local)
    if headline and rank == 0 and not args.no_clock_sampler:
        sampler.start()          # before the warm-up, so the poller is running when the timed region starts
    try:
        time_device_resident(layer, inp, prepared, 0, args.warmup, None)
        barrier(world)
        launches0 = _ffi.launch_count()
        sampler.begin()
        total_ms, per_step, out = time_device_resident(layer, inp, prepared, args.steps, 0, flush)
        sampler.end()
    finally:                     # the nvidia-smi poller must not outlive a failed run
        clocks = sampler.stop() if (headline and rank == 0) else None
    barrier(world)
    launches = _ffi.launch_count() - launches0
    total_ms = max_over_ranks(total_ms, world)
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = out.index_select(0, torch.from_numpy(dump_rows(V, H)).to(dev)).cpu().numpy()
    ms_per_step = total_ms / args.steps
    res = {"workload": wl["desc"], "nodes": V, "edges": M, "edge_types": L, "hidden_dim": H, "kind": kind,
           "ms_per_layer": ms_per_step, "edges_per_s": world * M / (ms_per_step * 1e-3),
           "step_ms_min_max": [min(per_step), max(per_step)], "gpu_launches": int(launches),
           "prepare_ms": prepare_dev_ms, "prepare_wall_ms": prepare_wall_ms, "prepare_first_call_ms": prepare_first_ms,
           "l2": ("flushed between timed iterations (256 MB write): node table fits the 126 MB L2" if fits_l2
                  else "no flush needed: node table exceeds the 126 MB L2"),
           "clocks": clocks}
    peak, peak_src = load_peaks()
    alg = algorithmic_bytes(kind, V, wl["E"], H, H, params)
    achieved = alg / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = load_traffic(name, args.path)
    res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                       "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                       "algorithmic_bytes_per_step": alg, "frac_of_nominal_8TBs": achieved / 8000.0,
                       "kernel": KERNEL_OF.get(kind, kind)}
    # the other roof: node-level contractions at fp32 accuracy on the tensor cores (3 tf32 MMAs per product)
    flops = dense_flops(kind, V, wl["E"], H, H, params)
    tf32_peak, tf32_src = load_tensor_peak()
    t_hbm_ms = alg / (peak * 1e9) * 1e3
    t_dense_ms = 3.0 * flops / (tf32_peak * 1e12) * 1e3
    res["roofline"]["dense"] = {"fp32_equiv_flops_per_step": flops, "tf32_mma_flops_per_step": 3.0 * flops,
                                "tf32_peak_tflops": tf32_peak, "tf32_peak_source": tf32_src,
                                "t_hbm_ms": t_hbm_ms, "t_dense_ms": t_dense_ms,
                                "binding": "tensor" if t_dense_ms > t_hbm_ms else "hbm",
                                "frac_of_binding_bound": max(t_hbm_ms, t_dense_ms) / ms_per_step}
    if not args.skip_e2e:
        out_host = torch.empty((V, H), dtype=torch.float32).pin_memory()
        e2e_steps = args.steps
        dt = time_e2e(layer, h_host, adj_host, out_host, e2e_steps, world, depth=E2E_DEPTH)
        res["e2e"] = {"value": world * M * e2e_steps / dt, "unit": "edges/s",
                      "h2d_bytes_per_step": int(h_host.numel() * 4 + sum(a.numel() * 4 for a in adj_host)),
                      "d2h_bytes_per_step": int(out_host.numel() * 4), "steps": e2e_steps,
                      "ms_per_step": dt / e2e_steps * 1e3, "pipeline_depth": E2E_DEPTH,
                      "what": "public layer call on pinned HOST buffers: H2D(node states + adjacency) -> CSR prepare -> "
                              f"layer -> D2H(new node states) every step; steps software-pipelined {E2E_DEPTH} deep on CUDA streams "
                              "(runtime.HostPipeline), wall clock over all steps"}
    res["_inputs"] = (h_np, adjs_np, w_np)
    res["_output"] = dumped
    return res


def measure_sharded(args, rank, world, local, dev):
    """SURVEY.md §8e case 2 under the bench clock: ONE graph (cfg2) strong-scaled over the N ranks by target range, one
    all-gather of the node-state shards per layer (NCCL over NVLink), checked against the unsharded layer on rank 0's rows."""
    import torch
    import torch.distributed as dist
    from tf2_gnn_b200.layers import MessagePassingInput
    from tf2_gnn_b200.runtime import PreparedBatch
    results = {}
    jobs = [("cfg2_strong", "cfg2")]
    if world == 8:
        jobs.append(("cfg5_full", "cfg5"))
    for key, name in jobs:
      try:
          wl = WORKLOADS[name]
          V, H, L = wl["V"], wl["H"], len(wl["E"])
          M = sum(wl["E"])
          if V % (world * 128) != 0:
              V = V // (world * 128) * (world * 128)   # equal shards on 128-row tile boundaries
          rows = V // world
          lo, hi = rank * rows, (rank + 1) * rows
          layer, params = build_layer(wl, 0, args.path)            # same weights on every rank
          gen = torch.Generator(device=dev)
          gen.manual_seed(99)
          if name == "cfg5":
              # each rank generates ITS shard of the ER graph directly: targets uniform in its range, sources uniform in
              # [0, V) (the full 256M-edge list never exists in one place); node states generated on the device
              g2 = torch.Generator(device=dev)
              g2.manual_seed(1000 + rank)
              adj_dev = []
              for E in wl["E"]:
                  e_loc = E // world
                  src = torch.randint(0, V, (e_loc,), generator=g2, device=dev, dtype=torch.int32)
                  tgt = torch.randint(lo, hi, (e_loc,), generator=g2, device=dev, dtype=torch.int32)
                  adj_dev.append(torch.stack([src, tgt], dim=1).contiguous())
              adj_dev = tuple(adj_dev)
              h_local = torch.rand((rows, H), generator=g2, device=dev) * 2 - 1
              m_total = sum(int(a.shape[0]) for a in adj_dev) * world
              full_check = None
          else:
              h_np, adjs_np, w_np = make_inputs(dict(wl, V=V), seed=0)   # the SAME graph on every rank
              if wl["kind"] == "rgcn":
                  layer.set_weights_from_oracle_dict({"edge_mlps": [[w] for w in w_np]})
              adj_dev = tuple(torch.from_numpy(a).to(dev) for a in adjs_np)
              h_local = torch.from_numpy(h_np[lo:hi]).to(dev)
              m_total = M
              full_check = (h_np, adjs_np)
          shard = PreparedBatch(adj_dev, V, target_range=(lo, hi))
          h_full = torch.empty((V, H), dtype=torch.float32, device=dev)

          def step():
              dist.all_gather_into_tensor(h_full, h_local)          # the one collective of the layer
              return layer(MessagePassingInput(h_full, adj_dev), prepared=shard)

          for _ in range(max(3, args.warmup)):
              out_local = step()
          torch.cuda.synchronize()
          barrier(world)
          n_it = args.steps
          ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
          # all-gather alone, layer alone, both (device time, max over ranks)
          ev[0].record()
          for _ in range(n_it):
              dist.all_gather_into_tensor(h_full, h_local)
          ev[1].record()
          torch.cuda.synchronize()
          ag_ms = max_over_ranks(ev[0].elapsed_time(ev[1]) / n_it, world)
          barrier(world)
          ev[0].record()
          for _ in range(n_it):
              out_local = step()
          ev[1].record()
          torch.cuda.synchronize()
          tot_ms = max_over_ranks(ev[0].elapsed_time(ev[1]) / n_it, world)
          ag_bytes = (world - 1) * rows * H * 4
          rec = {"workload": wl["desc"], "nodes": V, "edges": m_total, "target_rows_per_rank": rows,
                 "ms_per_layer": tot_ms, "edges_per_s": m_total / (tot_ms * 1e-3), "allgather_ms": ag_ms,
                 "allgather_bytes_received_per_rank": ag_bytes,
                 "allgather_GBps_per_rank": ag_bytes / (ag_ms * 1e-3) / 1e9 if ag_ms > 0 else None,
                 "overlap": "none: all_gather_into_tensor of the [V/N, H] shards, then the layer on the rank's target range",
                 "scaling": "strong"}
          if full_check is not None and rank == 0:
              h_np, adjs_np = full_check
              full = PreparedBatch(adj_dev, V)
              ref = layer(MessagePassingInput(torch.from_numpy(h_np).to(dev), adj_dev), prepared=full)
              mine = out_local
              diff = (ref[lo:hi] - mine).abs().max().item()
              rec["check"] = {"what": "rank 0's target rows of the sharded layer vs the unsharded layer on the same GPU",
                              "bitwise_equal": bool(torch.equal(ref[lo:hi], mine)), "max_abs_diff": diff,
                              "max_abs_ref": ref.abs().max().item()}
              del full, ref
          # ---- the all-gather fused into the layer kernel (peer stores over NVLink from the epilogue) ----
          if wl["kind"] == "rgcn":
              try:
                  from tf2_gnn_b200.sharding import PeerNodeTables
                  tables = PeerNodeTables(V, H)
                  n_layers = 4
                  tables.table(0)[lo:hi].copy_(h_local)
                  dist.all_gather_into_tensor(tables.table(0), h_local)      # the initial node states, once

                  def make_chain(use_mc):
                      def chain():
                          for k in range(n_layers):
                              layer.call_allgather(tables.table(k), shard, tables.replica_ptrs(k + 1), rank,
                                                   multicast_ptr=tables.multicast_ptr(k + 1) if use_mc else 0)
                              tables.barrier(k + 1)
                      return chain

                  def time_chain(chain):
                      for _ in range(3):
                          chain()
                      torch.cuda.synchronize()
                      barrier(world)
                      ev[0].record()
                      for _ in range(n_it):
                          chain()
                      ev[1].record()
                      torch.cuda.synchronize()
                      return max_over_ranks(ev[0].elapsed_time(ev[1]) / (n_it * n_layers), world)

                  have_mc = all_ranks_true(tables.multicast_ptr(0) != 0 and tables.multicast_ptr(1) != 0, world)
                  chain = make_chain(False)
                  fused_ms = time_chain(chain)
                  fz = {"ms_per_layer": fused_ms, "edges_per_s": m_total / (fused_ms * 1e-3), "layers_chained": n_layers,
                        "nvlink_bytes_stored_per_rank_per_layer": ag_bytes,
                        "nvlink_GBps_per_rank": ag_bytes / (fused_ms * 1e-3) / 1e9,
                        "what": "tfgnn_b200_rgcn_fwd_allgather: the fused kernel's epilogue stores each output tile into every "
                                "rank's node-state table (P2P stores over NVLink, symmetric memory); no collective call, one "
                                "signal exchange per layer"}
                  # the chained result against the same chain built from layer + NCCL all-gather (bitwise)
                  dist.all_gather_into_tensor(tables.table(0), h_local)      # fresh start: the timing loop iterated the states
                  torch.cuda.synchronize()
                  barrier(world)
                  chain()
                  torch.cuda.synchronize()
                  barrier(world)
                  h_a = h_local
                  full_t = torch.empty((V, H), dtype=torch.float32, device=dev)
                  for k in range(n_layers):
                      dist.all_gather_into_tensor(full_t, h_a)
                      h_a = layer(MessagePassingInput(full_t, adj_dev), prepared=shard)
                  dist.all_gather_into_tensor(full_t, h_a)
                  final = tables.table(n_layers)
                  torch.cuda.synchronize()
                  fz["bitwise_equal_to_nccl_chain"] = bool(torch.equal(final, full_t))
                  fz["max_abs_diff_to_nccl_chain"] = (final - full_t).abs().max().item()
                  if have_mc:
                      # the same through the switch's multicast: one multimem.st per 16 bytes instead of one store per peer
                      mc_chain = make_chain(True)
                      mc_ms = time_chain(mc_chain)
                      dist.all_gather_into_tensor(tables.table(0), h_local)
                      torch.cuda.synchronize()
                      barrier(world)
                      mc_chain()
                      torch.cuda.synchronize()
                      barrier(world)
                      fz["multicast"] = {"ms_per_layer": mc_ms, "edges_per_s": m_total / (mc_ms * 1e-3),
                                         "nvlink_bytes_stored_per_rank_per_layer": ag_bytes // max(world - 1, 1),
                                         "bitwise_equal_to_nccl_chain": bool(torch.equal(tables.table(n_layers), full_t)),
                                         "what": "multimem.st to the symmetric-memory multicast address: NVSwitch replicates"}
                  else:
                      fz["multicast"] = None
                  rec["fused_allgather"] = fz
                  del tables, full_t
              except Exception as e:
                  rec["fused_allgather"] = {"error": f"{type(e).__name__}: {e}"[:300]}
          results[key] = rec
          del shard, h_full, adj_dev, h_local, out_local
          torch.cuda.empty_cache()
          barrier(world)
      except Exception as e:   # same shapes on every rank: a failure (e.g. out of memory) is collective
        results[key] = {"workload": WORKLOADS[name]["desc"], "error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()
    return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--path", default="auto")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true", help="headline workload only")
    ap.add_argument("--skip-sharded", action="store_true", help="N > 1: no target-range sharded leg")
    ap.add_argument("--no-clock-sampler", action="store_true", help="do not poll nvidia-smi during the run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write each measured workload's last layer output as DIR/<workload>.npy "
                         "(float32; all rows, or a fixed seeded sample of 16 MB of rows when larger; rank 0 only) to "
                         "compare builds on identical seeded inputs")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    wl = WORKLOADS[args.workload]

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        world = int(os.environ.get("WORLD_SIZE", "1"))
        reference_arm(args, wl, rank, world)
        return

    import torch
    rank, world, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback exists)")
    from tf2_gnn_b200.build import build_library
    build_library()
    dev = torch.device("cuda", torch.cuda.current_device())

    head = measure_workload(args.workload, args, rank, world, local, dev, headline=True)
    h_np, adjs_np, w_np = head.pop("_inputs")
    outputs = {args.workload: head.pop("_output")}
    V, H, L, M, kind = head["nodes"], head["hidden_dim"], head["edge_types"], head["edges"], head["kind"]

    # ---- secondary workloads in the same run (north_star: hidden_dim 320; PPI-shaped batch) ----
    secondary = {}
    if not args.skip_secondary and args.workload == "cfg2" and world == 1:
        for name in ("h320", "cfg1"):
            torch.cuda.empty_cache()
            r = measure_workload(name, args, rank, world, local, dev, headline=False)
            r.pop("_inputs")
            r.pop("clocks")
            outputs[name] = r.pop("_output")
            secondary[name] = r

    # ---- target-range sharded leg (N > 1) --------------------------------------------------
    sharded = None
    if world > 1 and not args.skip_sharded and args.workload == "cfg2":
        torch.cuda.empty_cache()
        sharded = measure_sharded(args, rank, world, local, dev)

    if rank != 0:
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    cpu = None
    if not args.skip_cpu_baseline and kind == "rgcn":
        threads, _, host_cores = best_cpu_threads(wl, h_np, adjs_np, w_np)
        eps, m_sample, t_step = run_cpu_port(wl, h_np, adjs_np, w_np, min(M, 2_000_000), 2, 1, threads)
        cpu = {"value": eps, "unit": "edges/s", "cores": threads, "kind": "port",
               "sample": f"first {m_sample} of {M} edges on the full V={V} node table, 1 layer, 2 timed runs; "
                         f"torch-CPU restatement of the reference op order (TensorFlow absent); fastest thread "
                         f"count on a {host_cores}-core host"}
    line = {
        "metric": METRIC, "value": head["edges_per_s"], "unit": "edges/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_layer"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": head["workload"], "nodes": V, "edges": M, "edge_types": L, "hidden_dim": H,
                   "layers_per_step": 1, "path": args.path, "inputs_exceed_l2": V * H * 4 > 126e6,
                   "l2_flush": head["l2"],
                   "parallelism": f"dp{world} (independent batches of disjoint graphs, no collective; the target-range "
                                  f"sharded path is reported under 'sharded')",
                   "prepare_ms": head["prepare_ms"], "prepare_wall_ms": head["prepare_wall_ms"],
                   "prepare_first_call_ms": head["prepare_first_call_ms"]},
        "roofline": head["roofline"], "cpu_baseline": cpu, "e2e": head.get("e2e"),
        "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "step_ms_min_max": head["step_ms_min_max"],
        "secondary": secondary or None, "sharded": sharded,
    }
    print(json.dumps(line), flush=True)


def _shutdown():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    try:
        main()
    finally:
        _shutdown()
