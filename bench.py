#!/usr/bin/env python
"""bench.py -- headline benchmark of the weight-only matmul hot path on B200.

Metric (BASELINE.json): decode tokens/s, Llama-2-7B Q4_0, batch 1, 1 GPU, with the fraction of the measured HBM roofline.
A "step" = one decode token's worth of the hot path: every weight-only matmul of Llama-2-7B (32 x {QKV, o-proj,
gate/up+SiLU*mul, down} + lm_head = 6.607e9 Q4_0 weights = 3.716 GB of packed bytes), activations quantised to Q8_0 on
the device exactly as ne_compute_forward_mul_mat_q_f32 does, all captured in one CUDA graph.  Synthetic data:
W ~ N(0, 0.02^2) (torch.manual_seed(1234)), quantised to Q4_0 on the device by the library's own quantiser.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--fmt q4_0|int4g128] [--dump-outputs DIR]

--dump-outputs DIR writes what the timed path computed in its last timed step, as float32 DIR/<name>.npy: the logits and the
outputs of the last layer's matmul nodes (every layer writes the same buffers).  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.

Keys beyond the base contract: roofline{} (dominant kernel = the streaming GEMV, timed live with CUDA events on the
launching stream), cpu_baseline{} (the reference's own ggml Q4_0 x Q8_0 code, oracle/_ref, timed on this box's host cores
on a bounded sample), e2e{} (the same token through the host-buffer C-ABI, H2D/D2H inside the timed region).
N > 1: the 7B model fits one GPU, so ranks are independent replicas ("replicas only", DESIGN.md) -- no collective.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("OMP_PROC_BIND", "false")

N_EMBD, N_FF, N_LAYER, N_VOCAB = 4096, 11008, 32, 32000
# BASELINE.json's metric, verbatim.  `value` is its first component (decode tokens/s, batch 1, weight-only matmul path); the
# second (prefill tok/s with the tensor roofline) is reported under "prefill", the % of the HBM roofline under "roofline".
METRIC = "decode tokens/s + prefill tok/s Llama-2-7B Q4_0 @1 GPU; % HBM roofline"
try:
    with open(os.path.join(ROOT, "BASELINE.json")) as _f:
        METRIC = json.load(_f).get("metric", METRIC)
except (OSError, ValueError):
    pass


def dump_outputs(path, arrays):
    """arrays: name -> array; written as float32 .npy files under path (at most 64 MB in all)"""
    os.makedirs(path, exist_ok=True)
    arrays = {name: np.ascontiguousarray(a, dtype=np.float32) for name, a in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def shapes():
    """(name, n, k) of every matmul weight of one layer + lm_head (SURVEY.md 8: q,k,v,o 4096x4096; gate,up 11008x4096;
    down 4096x11008; lm_head 32000x4096)."""
    per_layer = [("wq", N_EMBD, N_EMBD), ("wk", N_EMBD, N_EMBD), ("wv", N_EMBD, N_EMBD), ("wo", N_EMBD, N_EMBD),
                 ("w1", N_FF, N_EMBD), ("w3", N_FF, N_EMBD), ("w2", N_EMBD, N_FF)]
    return per_layer, ("lm_head", N_VOCAB, N_EMBD)


# ----------------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(kernel_substr, path=None):
    """average dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernels whose name contains `kernel_substr`, from a
    committed `ncu --csv` launch list (cold-cache, serialised launches); (None, None) when the file is missing"""
    import csv
    path = path or os.path.join(ROOT, "profiles", "r02_launches_bench.csv")
    try:
        rows = list(csv.reader(open(path)))
    except OSError:
        return None, None
    hdr = next((r for r in rows if "Kernel Name" in r), None)
    if not hdr:
        return None, None
    ki, mi, vi, ii = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    per = {}
    for r in rows:
        if len(r) > vi and kernel_substr in r[ki] and r[mi] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            try:
                per[r[ii]] = per.get(r[ii], 0.0) + float(r[vi].replace(",", ""))
            except ValueError:
                pass
    if not per:
        return None, None
    return sum(per.values()) / len(per), f"ncu launch list {os.path.relpath(path, ROOT)} ({len(per)} launches of {kernel_substr})"


# ----------------------------------------------------------------------------------------------------------- reference arm
def host_threads():
    """usable host cores: scheduler affinity, capped by the cgroup CPU quota (a 128-CPU box may grant this container far
    fewer; oversubscribed OpenMP barriers would then make the reference look absurdly slow)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    env = os.environ.get("NS_REF_THREADS")
    return int(env) if env else n


class CpuReference:
    """The reference's ggml Q4_0 x Q8_0 matmul (oracle/_ref/libref_ggml.so = /root/reference headers compiled in place;
    falls back to the oracle port when _ref is absent), all host threads, on synthetic Llama-2-7B-shaped weights.
    To bound setup time only `distinct` layers of distinct weights are materialised and cycled (each layer's 114 MB
    exceeds typical L2; cycling 4 layers = 455 MB defeats L3 reuse)."""

    def __init__(self, distinct=4, seed=1234):
        import oracle
        self.o = oracle
        self.kind = "reference" if oracle.ref_ggml() is not None else "port"
        self.impl = "ref" if self.kind == "reference" else "oracle"
        rng = np.random.default_rng(seed)
        per_layer, lm = shapes()
        self.layers = []
        for _ in range(distinct):
            ws = {}
            for name, n, k in per_layer:
                w = (rng.standard_normal((n, k), dtype=np.float32) * np.float32(0.02))
                ws[name] = oracle.quantize_q4_0(w, self.impl)
            self.layers.append(ws)
        w = (rng.standard_normal((lm[1], lm[2]), dtype=np.float32) * np.float32(0.02))
        self.lm_head = oracle.quantize_q4_0(w, self.impl)
        self.x = rng.standard_normal((1, N_EMBD), dtype=np.float32)
        self.h = rng.standard_normal((1, N_FF), dtype=np.float32)
        self.threads = host_threads()

    def token(self, n_layers=N_LAYER):
        """all matmuls of one decode token (7 per layer, unfused, as the ggml path runs them) + lm_head; self.last keeps the
        last layer's outputs and the logits"""
        mm = lambda wq, a: self.o.mul_mat_q4_0_f32(wq, a, self.impl, nth=self.threads)
        out = {}
        for l in range(n_layers):
            ws = self.layers[l % len(self.layers)]
            for name in ("wq", "wk", "wv", "wo", "w1", "w3"):
                out["last_layer_" + name] = mm(ws[name], self.x)
            out["last_layer_w2"] = mm(ws["w2"], self.h)
        if n_layers == N_LAYER:
            out["logits"] = mm(self.lm_head, self.x)
        self.last = out

    def time_tokens(self, tokens, warmup=1):
        for _ in range(warmup):
            self.token()
        t0 = time.perf_counter()
        for _ in range(tokens):
            self.token()
        dt = time.perf_counter() - t0
        return tokens / dt, dt / tokens


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference()
    tps, spt = ref.time_tokens(args.steps, max(1, min(args.warmup, 2)))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ref.last)
    line = {
        "impl": "reference", "metric": METRIC, "value": tps, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": spt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int8xint4->f32 (q8_0 x q4_0)", "data": "synthetic N(0,0.02^2) weights, 4 distinct layers cycled",
        "config": {"workload": "llama2-7b q4_0 decode matmul path, batch 1, 225 unfused mul_mat per token", "parallelism": "cpu"},
        "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": ref.threads, "kind": ref.kind,
                         "sample": f"{args.steps} full tokens (32 layers x 7 matmuls + lm_head), {ref.threads} OpenMP threads, "
                                   "ne_vec_dot_q4_0_q8_0 built -O3 -mavx2 -mfma -mf16c"},
        "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------- tensor parallel leg
def run_tp(world, rank, hbm_peak, steps):
    """BASELINE config 5: Llama-2-70B INT4 g128, tensor parallel over `world` GPUs (strong scaling: the model is fixed, every rank
    holds 1/world of each matmul; q/k/v/gate/up N-split, o/down K-split + one sum all-reduce each, llama.cpp:121-124,592,693).
    All 80 layers' matmul nodes + the replicated lm_head per token, one CUDA graph per token, (a) NCCL all-reduce (b) the one-shot
    NVLink all-reduce of csrc/comm.cu (ns_comm_*).  Device time, max over ranks."""
    import torch
    import torch.distributed as dist
    import neural_speed_b200 as ns
    from neural_speed_b200 import tp
    E, FF, H, HKV, NL, V = 8192, 28672, 64, 8, 80, 32000
    if H % world or HKV % world:
        return {"skipped": f"n_head_kv {HKV} not divisible by {world}"}
    ctx = tp.TPContext(init=False)
    plan = tp.LlamaShardPlan(world, E, FF, H, HKV, 128)
    shapes = plan.shapes()
    kw = dict(group=128, wfmt=ns.W_S4, stype=ns.S_F32, comp=ns.COMP_INT8, asym=False)
    layers = [{name: ns.Weight.random(n, k, seed=1000 * rank + 7 * li + i, **kw) for i, (name, (_, n, k)) in enumerate(shapes.items())}
              for li in range(NL)]
    head = ns.Weight.random(V, E, seed=5, **kw)  # replicated, as the reference keeps it
    ns.lib().bestla_device_sync(None)
    bytes_rank = sum(w.algorithmic_bytes for lay in layers for w in lay.values()) + head.algorithmic_bytes
    eng = tp.TPLlamaMatmuls(plan, layers, ctx)
    x0 = torch.randn(1, E, device="cuda")
    logits = torch.zeros(1, V, device="cuda")
    res = {}
    # the one-shot NVLink exchange (cudaIpc peer mappings, csrc/comm.cu) is measured where it has been validated on hardware
    # (2 GPUs: tests/test_gpu_tp.py, profiles/r02_summary.md); NS_TP_ONESHOT=1 forces it at any world size
    modes = ("nccl", "nvlink_oneshot") if (world == 2 or os.environ.get("NS_TP_ONESHOT")) else ("nccl",)
    for mode in modes:
        if mode == "nvlink_oneshot":
            ctx.enable_p2p(E)
        stream = torch.cuda.Stream()
        xa, xb = x0.clone(), torch.empty_like(x0)

        def token():
            # every layer reads the same N(0,1) input: synthetic weights without the norms in between would overflow fp32 after a
            # few dozen residual adds; the stream still runs the 80 layers strictly one after the other
            cur = xb
            for li in range(NL):
                cur = eng.layer(li, xa, out=xb)
            ns.mul_mat(head, cur.data_ptr(), E, logits.data_ptr(), V, 1, queue=tp.current_queue(torch))
            return cur

        with torch.cuda.stream(stream):
            for _ in range(2):
                token()
            torch.cuda.synchronize()
            dist.barrier()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                y = token()
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                g.replay()
            e1.record(stream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            # the exchange alone: 2 x NL all-reduces of E floats, same graph mechanics
            t = torch.zeros(1, E, device="cuda")
            ga = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ga, stream=stream):
                for _ in range(2 * NL):
                    ctx.all_reduce(t)
            ga.replay()
            torch.cuda.synchronize()
            dist.barrier()
            e0.record(stream)
            for _ in range(10):
                ga.replay()
            e1.record(stream)
            torch.cuda.synchronize()
            ar_us = e0.elapsed_time(e1) * 1e3 / (10 * 2 * NL)
        tm = torch.tensor([ms, ar_us], device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms, ar_us = float(tm[0]), float(tm[1])
        res[mode] = {"finite": bool(torch.isfinite(y).all()), "ms_per_token": ms, "tokens_per_s": 1000.0 / ms, "per_gpu_GBps": bytes_rank / (ms * 1e-3) / 1e9,
                     "per_gpu_frac": bytes_rank / (ms * 1e-3) / 1e9 / hbm_peak, "allreduce_us": ar_us}
    best = max(res, key=lambda m: res[m]["tokens_per_s"])
    out = {"model": "llama2-70b int4 g128 (synthetic shards), batch 1, 80 layers + replicated lm_head, matmul path + 160 all-reduces of 32 KiB",
           "tp": world, "scaling": "strong", "tokens_per_s": res[best]["tokens_per_s"], "per_gpu_frac": res[best]["per_gpu_frac"],
           "allreduce_us": res[best]["allreduce_us"], "exchange": best, "per_rank_packed_bytes": int(bytes_rank), **res}
    del layers, head, eng
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import neural_speed_b200 as ns

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        import datetime
        # a rank that dies must not leave the others waiting for ten minutes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    torch.cuda.set_device(local)
    L = ns.lib()
    L.bestla_init()
    devh = L.bestla_create_device(False)
    queue = L.bestla_get_device_queue(devh)
    stream = torch.cuda.ExternalStream(queue)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    # ---- synthetic weights, quantised + repacked on the device
    torch.manual_seed(1234 + rank)
    per_layer, lm = shapes()

    def make_weight(n, k):
        w = torch.randn(n, k, device="cuda", dtype=torch.float32) * 0.02
        if args.fmt == "q4_0":
            rows = torch.empty(n * (k // 32) * 18, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            rc = L.ns_device_quantize_q4_0(C.c_void_p(w.data_ptr()), C.c_void_p(rows.data_ptr()), n, k, queue)
            assert rc == 0, ns.last_error()
            h = ns.Weight.from_q4_0_device(rows.data_ptr(), n, k, k // 32 * 18, queue)
            L.bestla_device_sync(queue)
            return h
        blob = ns.np_bestla_quantize(w.cpu().numpy(), "int4", 128, "sym", "fp32", "int8")
        return ns.Weight.from_blob(blob, queue)

    t_setup = time.perf_counter()
    n_layers = args.layers
    layers = [{name: make_weight(n, k) for name, n, k in per_layer} for _ in range(n_layers)]
    lm_head = make_weight(lm[1], lm[2])
    L.bestla_device_sync(queue)
    setup_s = time.perf_counter() - t_setup
    alg_bytes = sum(w.algorithmic_bytes for lay in layers for w in lay.values()) + lm_head.algorithmic_bytes
    n_weights = sum(w.n * w.k for lay in layers for w in lay.values()) + lm_head.n * lm_head.k

    # ---- device buffers (activations stay resident; synthetic post-norm-like N(0,1) inputs)
    x = torch.randn(1, N_EMBD, device="cuda")
    attn = torch.randn(1, N_EMBD, device="cuda")
    qkv = torch.zeros(3, 1, N_EMBD, device="cuda")
    o = torch.zeros(1, N_EMBD, device="cuda")
    tmp = torch.zeros(1, N_FF, device="cuda")
    ffn = torch.zeros(1, N_EMBD, device="cuda")
    logits = torch.zeros(1, N_VOCAB, device="cuda")
    ws_bytes = L.ns_device_workspace_bytes(4, N_FF)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    ws_x = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    ws_h = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    wsp = C.c_void_p(ws.data_ptr())

    dbg = os.environ.get("NS_SYNC_EACH") is not None

    def step_calls():
        """one token's matmuls: fused QKV, o-proj, fused gate/up+SiLU*mul -> down, lm_head"""
        for li, lay in enumerate(layers):
            if dbg:
                L.bestla_device_sync(queue)
                print("layer", li, flush=True)
            rc = L.ns_mul_qkv(lay["wq"].h, lay["wk"].h, lay["wv"].h, C.c_void_p(x.data_ptr()), N_EMBD, C.c_void_p(qkv.data_ptr()),
                              N_EMBD, 1, wsp, queue)
            rc |= L.ns_mul_mat(lay["wo"].h, C.c_void_p(attn.data_ptr()), N_EMBD, C.c_void_p(o.data_ptr()), N_EMBD, 1, None, None, 0,
                               wsp, queue)
            rc |= L.ns_ffn_silu(lay["w1"].h, lay["w2"].h, lay["w3"].h, C.c_void_p(x.data_ptr()), N_EMBD, C.c_void_p(tmp.data_ptr()),
                                C.c_void_p(ffn.data_ptr()), N_EMBD, 1, wsp, queue)
            assert rc == 0, ns.last_error()
        rc = L.ns_mul_mat(lm_head.h, C.c_void_p(x.data_ptr()), N_EMBD, C.c_void_p(logits.data_ptr()), N_VOCAB, 1, None, None, 0, wsp,
                          queue)
        assert rc == 0, ns.last_error()

    def gemv_only_calls():
        """the same GEMV launches against pre-quantised activations (dominant-kernel timing for the roofline)"""
        WP = C.c_void_p * 3
        for lay in layers:
            rc = L.ns_matmul_prepared(WP(lay["wq"].h, lay["wk"].h, lay["wv"].h), 3, 1, C.c_void_p(ws_x.data_ptr()),
                                      C.c_void_p(qkv.data_ptr()), N_EMBD, 1, None, 0, None, None, queue)
            rc |= L.ns_matmul_prepared(WP(lay["wo"].h, None, None), 1, 0, C.c_void_p(ws_x.data_ptr()), C.c_void_p(o.data_ptr()),
                                       N_EMBD, 1, None, 0, None, None, queue)
            rc |= L.ns_matmul_prepared(WP(lay["w1"].h, lay["w3"].h, None), 2, 2, C.c_void_p(ws_x.data_ptr()),
                                       C.c_void_p(tmp.data_ptr()), N_FF, 1, None, 0, None, None, queue)
            rc |= L.ns_matmul_prepared(WP(lay["w2"].h, None, None), 1, 0, C.c_void_p(ws_h.data_ptr()), C.c_void_p(ffn.data_ptr()),
                                       N_EMBD, 1, None, 0, None, None, queue)
            assert rc == 0, ns.last_error()
        rc = L.ns_matmul_prepared(WP(lm_head.h, None, None), 1, 0, C.c_void_p(ws_x.data_ptr()), C.c_void_p(logits.data_ptr()),
                                  N_VOCAB, 1, None, 0, None, None, queue)
        assert rc == 0, ns.last_error()

    # eager pass first (sizes nothing inside capture), then capture both graphs
    lc0 = L.ns_launch_count()
    step_calls()
    L.bestla_device_sync(queue)
    launches_per_step = int(L.ns_launch_count() - lc0)
    assert L.ns_prepare_activation(layers[0]["wq"].h, C.c_void_p(x.data_ptr()), N_EMBD, 1, C.c_void_p(ws_x.data_ptr()), queue) == 0
    assert L.ns_prepare_activation(layers[0]["w2"].h, C.c_void_p(tmp.data_ptr()), N_FF, 1, C.c_void_p(ws_h.data_ptr()), queue) == 0
    L.bestla_device_sync(queue)

    def capture(fn):
        assert L.ns_graph_begin(queue) == 0, ns.last_error()
        fn()
        g = L.ns_graph_end(queue)
        assert g, ns.last_error()
        return C.c_void_p(g)

    use_graph = not args.no_graph
    g_step = capture(step_calls) if use_graph else None
    g_gemv = capture(gemv_only_calls) if use_graph else None
    lc1 = L.ns_launch_count()

    def run_step():
        if use_graph:
            assert L.ns_graph_launch(g_step, queue) == 0, ns.last_error()
        else:
            step_calls()

    def timed(fn, steps, warmup, collective=True):
        """device time of `steps` calls; collective=True: every rank calls this (barrier before, max over ranks after)"""
        for _ in range(warmup):
            fn()
        L.bestla_device_sync(queue)
        if world > 1 and collective:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1 and collective:
            import torch.distributed as dist
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_perop = timed(run_step, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:  # before any other leg reuses these buffers
        dump_outputs(args.dump_outputs, {"last_layer_qkv": qkv.cpu().numpy(), "last_layer_o": o.cpu().numpy(),
                                         "last_layer_ffn": ffn.cpu().numpy(), "logits": logits.cpu().numpy()})
    # a leg of at least one second of back-to-back steps: sustained clocks / power rather than a 20 ms burst
    sus_steps = max(args.steps, int(1.05 / (ms_perop * 1e-3)))
    ms_sus = timed(run_step, sus_steps, 3)
    ms_step = ms_perop  # headline = the fastest complete path (one fused act-quant + GEMV launch per matmul node)
    # dominant kernel alone (graph of GEMV launches on pre-quantised activations)
    n_gemv = 4 * n_layers + 1
    if use_graph:
        ms_gemv = timed(lambda: L.ns_graph_launch(g_gemv, queue), args.steps, args.warmup)
    else:
        ms_gemv = timed(gemv_only_calls, args.steps, args.warmup)
    gemv_gbs = alg_bytes / (ms_gemv * 1e-3) / 1e9
    step_gbs = alg_bytes / (ms_step * 1e-3) / 1e9

    # ---- prefill: the same matmul nodes for a 2048-token prompt through the tcgen05 tensor-core GEMM (bf16 numerics)
    prefill = None
    if rank == 0 and not args.skip_prefill:
        MP = args.prefill_tokens
        xp = torch.randn(MP, N_EMBD, device="cuda")
        ap_ = torch.randn(MP, N_EMBD, device="cuda")
        qkvp = torch.zeros(3, MP, N_EMBD, device="cuda")
        op_ = torch.zeros(MP, N_EMBD, device="cuda")
        tmpp = torch.zeros(2, MP, N_FF, device="cuda")
        ffnp = torch.zeros(MP, N_EMBD, device="cuda")
        wsp_bytes = L.ns_device_workspace_bytes(MP, N_FF)
        wsp_t = torch.zeros(wsp_bytes, dtype=torch.uint8, device="cuda")
        wpp = C.c_void_p(wsp_t.data_ptr())
        torch.cuda.synchronize()

        def prefill_calls():
            for lay in layers:
                rc = L.ns_mul_qkv(lay["wq"].h, lay["wk"].h, lay["wv"].h, C.c_void_p(xp.data_ptr()), N_EMBD, C.c_void_p(qkvp.data_ptr()),
                                  N_EMBD, MP, wpp, queue)
                rc |= L.ns_mul_mat(lay["wo"].h, C.c_void_p(ap_.data_ptr()), N_EMBD, C.c_void_p(op_.data_ptr()), N_EMBD, MP, None, None, 0,
                                   wpp, queue)
                rc |= L.ns_ffn_silu(lay["w1"].h, lay["w2"].h, lay["w3"].h, C.c_void_p(xp.data_ptr()), N_EMBD, C.c_void_p(tmpp.data_ptr()),
                                    C.c_void_p(ffnp.data_ptr()), N_EMBD, MP, wpp, queue)
                assert rc == 0, ns.last_error()

        prefill_calls()
        L.bestla_device_sync(queue)
        psteps = max(2, min(5, args.steps))
        ms_pf = timed(prefill_calls, psteps, 1, collective=False)  # rank 0 only: no collectives in here
        flops = 2.0 * MP * sum(w.n * w.k for lay in layers for w in lay.values())
        tf = flops / (ms_pf * 1e-3) / 1e12
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        prefill = {"tokens": MP, "tokens_per_s": MP / (ms_pf * 1e-3), "ms": ms_pf, "tflops": tf,
                   "roofline": {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if "bf16_tflops_sustained" in peaks else "fallback 1400",
                                "kernel": "gemm_w4_tc_kernel<256> (tcgen05.mma kind::f16, in-smem int4->bf16 dequant)"},
                   "note": f"{7 * n_layers} GEMMs of the {n_layers} layers (lm_head excluded: only the last token needs logits), "
                           "fp32 activations converted to bf16 per GEMM, outputs fp32; includes silu*mul and conversion kernels"}
        del xp, ap_, qkvp, op_, tmpp, ffnp, wsp_t
        torch.cuda.empty_cache()

    # ---- whole decode step: ns_llama_* (embedding, RMSNorm, RoPE, fp16 KV cache, attention, residuals, argmax around the
    # same matmuls), greedy generation with the argmax fed back on the device; one host call for the whole run
    engine = None
    if not args.skip_engine and n_layers == N_LAYER:
        n_ctx, n_prompt, n_new = 2304, 32, args.gen_tokens
        eng = ns.Llama(N_VOCAB, N_EMBD, 32, 32, n_layers, N_FF, n_ctx, 1e-5, 10000.0, 1.0, queue)
        emb = (torch.randn(N_VOCAB, N_EMBD) * 1.0).numpy()
        eng.set_f32(ns.Llama.TOK_EMBD, 0, emb)
        del emb
        ones = np.ones(N_EMBD, np.float32)
        eng.set_f32(ns.Llama.OUT_NORM, 0, ones)
        eng.set_weight(ns.Llama.OUTPUT, 0, lm_head)
        ids = dict(wq=ns.Llama.WQ, wk=ns.Llama.WK, wv=ns.Llama.WV, wo=ns.Llama.WO, w1=ns.Llama.W1, w2=ns.Llama.W2, w3=ns.Llama.W3)
        for il, lay in enumerate(layers):
            eng.set_f32(ns.Llama.ATTN_NORM, il, ones)
            eng.set_f32(ns.Llama.FFN_NORM, il, ones)
            for name, w in lay.items():
                eng.set_weight(ids[name], il, w)
        prompt = np.random.default_rng(3).integers(3, N_VOCAB, n_prompt).astype(np.int32)
        prompt[0] = 1  # BOS
        t0 = time.perf_counter()
        _, nxt = eng.eval(prompt, 0, want_logits=False)
        t_prompt = time.perf_counter() - t0
        eng.generate(int(nxt), n_prompt, 8)  # warm-up: builds the decode graph
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        lcg = L.ns_launch_count()
        t0 = time.perf_counter()
        toks = eng.generate(int(nxt), n_prompt, n_new)
        dt_gen = time.perf_counter() - t0
        launches_tok = (L.ns_launch_count() - lcg)  # graph replays do not count; kept for reference
        t0 = time.perf_counter()
        eng.eval(prompt, 0, want_logits=False)
        t_prompt2 = time.perf_counter() - t0
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([dt_gen], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_gen = float(t.item())
        # long prompt + decode at a long context on the same engine (rank 0 only: wall clock, not a collective leg)
        long_ctx = None
        if rank == 0 and n_ctx >= 2048 + 80:
            lp = np.random.default_rng(4).integers(3, N_VOCAB, 2048).astype(np.int32)
            lp[0] = 1
            eng.eval(lp[:64], 0, want_logits=False)  # sizes the activation buffers of the prompt path outside the timed call
            t0 = time.perf_counter()
            _, nx2 = eng.eval(lp, 0, want_logits=False)
            t_lp = time.perf_counter() - t0
            t0 = time.perf_counter()
            _, nx2 = eng.eval(lp, 0, want_logits=False)
            t_lp2 = time.perf_counter() - t0
            eng.generate(int(nx2), 2048, 4)
            t0 = time.perf_counter()
            eng.generate(int(nx2), 2048, 64)
            t_ld = time.perf_counter() - t0
            long_ctx = {"prompt_tokens": 2048, "prompt_eval_ms": t_lp2 * 1e3, "first_prompt_eval_ms": t_lp * 1e3,
                        "prompt_tokens_per_s": 2048 / t_lp2, "decode_tokens_per_s_at_2048": 64 / t_ld, "decode_ms_per_token_at_2048": t_ld / 64 * 1e3,
                        "note": "ns_llama_eval of a 2048-token prompt (tcgen05 GEMMs + mma.sync causal attention + everything else), then "
                                "64 greedy tokens at positions 2048..2111 (split-context decode attention); host wall clock"}
        engine = {"tokens_per_s": world * n_new / dt_gen, "long_context": long_ctx, "ms_per_token": dt_gen / n_new * 1e3, "new_tokens": n_new,
                  "prompt_tokens": n_prompt, "n_ctx": n_ctx, "prompt_eval_ms": t_prompt2 * 1e3, "first_prompt_eval_ms": t_prompt * 1e3,
                  "kv_cache_bytes": eng.kv_bytes(), "distinct_tokens": int(len(set(int(v) for v in toks))),
                  "timer": "host wall clock around ns_llama_generate (H2D first token, one CUDA graph per token, D2H token ids)",
                  "roofline_frac": (alg_bytes * n_new / dt_gen / 1e9) / hbm_peak,
                  "path": "ns_llama_generate: greedy, argmax fed back on device"}
        eng.close()
        del eng
        torch.cuda.empty_cache()

    # ---- the other BASELINE.json configs, same protocol (one CUDA graph of a token's matmul nodes, CUDA events on the launching
    # stream, weights >> L2): synthetic weight images of the right geometry (ns_weight_random: values do not matter to a
    # bandwidth-bound path; parity of every format is covered by the tests).  Rank 0 only.
    configs = []
    if rank == 0 and not args.skip_configs and n_layers == N_LAYER:
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))

        def build(shape_layer, lm_shape, **kw):
            lays = [{nm: ns.Weight.random(n, k, seed=17 + 131 * li + i, queue=queue, **kw) for i, (nm, n, k) in enumerate(shape_layer)}
                    for li in range(N_LAYER)]
            head = ns.Weight.random(lm_shape[1], lm_shape[2], seed=7, queue=queue, **kw)
            L.bestla_device_sync(queue)
            return lays, head

        def token_calls(lays, head, M, E, FF, kvd, xb, ab, qb, ob, tb, fb, lb, wsb):
            cp = lambda t: C.c_void_p(t.data_ptr())
            for lay in lays:
                if kvd == E:
                    rc = L.ns_mul_qkv(lay["wq"].h, lay["wk"].h, lay["wv"].h, cp(xb), E, cp(qb), E, M, wsb, queue)
                else:  # grouped-query attention: k and v are narrower, three nodes (llama.cpp:223-231)
                    rc = L.ns_mul_mat(lay["wq"].h, cp(xb), E, cp(qb), E, M, None, None, 0, wsb, queue)
                    rc |= L.ns_mul_mat(lay["wk"].h, cp(xb), E, cp(ob), kvd, M, None, None, 0, wsb, queue)
                    rc |= L.ns_mul_mat(lay["wv"].h, cp(xb), E, cp(ob), kvd, M, None, None, 0, wsb, queue)
                rc |= L.ns_mul_mat(lay["wo"].h, cp(ab), E, cp(ob), E, M, None, None, 0, wsb, queue)
                rc |= L.ns_ffn_silu(lay["w1"].h, lay["w2"].h, lay["w3"].h, cp(xb), E, cp(tb), cp(fb), E, M, wsb, queue)
                assert rc == 0, ns.last_error()
            if head is not None:
                assert L.ns_mul_mat(head.h, cp(xb), E, cp(lb), N_VOCAB, M, None, None, 0, wsb, queue) == 0, ns.last_error()

        def leg(name, lays, head, M, E, FF, kvd, steps, with_head=True, graph=True):
            xb, ab = torch.randn(M, E, device="cuda"), torch.randn(M, E, device="cuda")
            qb, ob = torch.zeros(3, M, E, device="cuda"), torch.zeros(M, E, device="cuda")
            tb, fb = torch.zeros(2, M, FF, device="cuda"), torch.zeros(M, E, device="cuda")
            lb = torch.zeros(M, N_VOCAB, device="cuda")
            wsz = L.ns_device_workspace_bytes(M, FF)
            wst = torch.zeros(wsz, dtype=torch.uint8, device="cuda")
            wsb = C.c_void_p(wst.data_ptr())
            torch.cuda.synchronize()
            fn = lambda: token_calls(lays, head if with_head else None, M, E, FF, kvd, xb, ab, qb, ob, tb, fb, lb, wsb)
            lc = L.ns_launch_count()
            fn()
            L.bestla_device_sync(queue)
            nl = int(L.ns_launch_count() - lc)
            if graph:
                g = capture(fn)
                run = lambda: L.ns_graph_launch(g, queue)
            else:
                run = fn
            ms = timed(run, steps, 3, collective=False)
            nbytes = sum(w.algorithmic_bytes for lay in lays for w in lay.values()) + (head.algorithmic_bytes if with_head else 0)
            nweights = sum(w.n * w.k for lay in lays for w in lay.values()) + (head.n * head.k if with_head else 0)
            out = {"name": name, "batch": M, "ms_per_step": ms, "tokens_per_s": M * 1000.0 / ms, "launches_per_step": nl}
            if M <= 32:   # weight streaming bound: the packed weights are read once per step whatever the batch
                gbs = nbytes / (ms * 1e-3) / 1e9
                out["roofline"] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                   "algorithmic_bytes_per_step": int(nbytes)}
            else:
                tf = 2.0 * M * nweights / (ms * 1e-3) / 1e12
                out["roofline"] = {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak}
            del xb, ab, qb, ob, tb, fb, lb, wst
            return out

        csteps = max(5, min(20, args.steps))
        per7b = per_layer
        lm7b = lm
        # config 2: Llama-2-7B INT4 group 128 symmetric (RTN geometry: f32 scales, int8 compute), decode + 2048-token prefill
        lays, head = build(per7b, lm7b, group=128, wfmt=ns.W_S4, stype=ns.S_F32, comp=ns.COMP_INT8, asym=False)
        configs.append(dict(leg("llama2-7b int4 g128 sym (RTN), decode", lays, head, 1, N_EMBD, N_FF, N_EMBD, csteps), config=2))
        configs.append(dict(leg("llama2-7b int4 g128 sym (RTN), prefill 2048", lays, head, args.prefill_tokens, N_EMBD, N_FF, N_EMBD, 3,
                                with_head=False, graph=False), config=2))
        del lays, head
        torch.cuda.empty_cache()
        # config 3: GPTQ / AWQ INT4 g128 (asymmetric zero points, bf16 scales as the reference's qpack emits), batch 1 / 8 / 32
        lays, head = build(per7b, lm7b, group=128, wfmt=ns.W_S4, stype=ns.S_BF16, comp=ns.COMP_INT8, asym=True)
        for M in (1, 8, 32):
            configs.append(dict(leg(f"llama2-7b GPTQ/AWQ int4 g128 asym, batch {M}", lays, head, M, N_EMBD, N_FF, N_EMBD, csteps), config=3))
        del lays, head
        torch.cuda.empty_cache()
        # config 4: Mistral-7B shapes (n_ff 14336, 8 KV heads), NF4 and INT8 weights, bf16 compute
        MFF, MKV = 14336, 1024
        mis = [("wq", N_EMBD, N_EMBD), ("wk", MKV, N_EMBD), ("wv", MKV, N_EMBD), ("wo", N_EMBD, N_EMBD), ("w1", MFF, N_EMBD),
               ("w3", MFF, N_EMBD), ("w2", N_EMBD, MFF)]
        for nm, kw in (("nf4 g32", dict(group=32, wfmt=ns.W_NF4, stype=ns.S_F32, comp=ns.COMP_BF16, asym=False)),
                       ("int8 g32", dict(group=32, wfmt=ns.W_S8, stype=ns.S_F32, comp=ns.COMP_BF16, asym=False))):
            lays, head = build(mis, lm7b, **kw)
            configs.append(dict(leg(f"mistral-7b {nm}, bf16 compute, decode", lays, head, 1, N_EMBD, MFF, MKV, csteps), config=4))
            del lays, head
            torch.cuda.empty_cache()

    # ---- e2e (headline): the token through the device-backend C-ABI of INTEGRATION.md B -- what ne_device_sync does in the
    # reference's NS_SYCL slot: the token's fp32 hidden state comes from pinned HOST memory (bestla_device_memcpy H2D), the
    # matmul nodes run device-resident (one ns_graph_launch), the fp32 logits go back to pinned HOST memory (D2H), then
    # bestla_device_sync.  Wall clock around the steps, every rank, max over ranks.
    e2e = None
    cpu = None
    if not args.skip_e2e:
        hx_pin = torch.randn(1, N_EMBD).pin_memory()
        hlogits_pin = torch.empty(1, N_VOCAB).pin_memory()
        nbx, nbl = N_EMBD * 4, N_VOCAB * 4

        def e2e_token():
            L.bestla_device_memcpy(C.c_void_p(x.data_ptr()), C.c_void_p(hx_pin.data_ptr()), nbx, queue)
            run_step()
            L.bestla_device_memcpy(C.c_void_p(hlogits_pin.data_ptr()), C.c_void_p(logits.data_ptr()), nbl, queue)
            L.bestla_device_sync(queue)

        for _ in range(max(3, args.warmup)):
            e2e_token()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_token()
        torch.cuda.synchronize()
        dt_e2e = (time.perf_counter() - t0) / args.steps
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([dt_e2e], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_e2e = float(t.item())
        assert bool(torch.isfinite(hlogits_pin).all())
        e2e = {"value": world / dt_e2e, "unit": "tokens/s", "h2d_bytes_per_step": nbx, "d2h_bytes_per_step": nbl,
               "ms_per_step": dt_e2e * 1e3, "steps": args.steps, "timer": "host wall clock, sync after every token",
               "path": "bestla_device_memcpy(H2D hidden state, pinned) -> ns_graph_launch (129 matmul nodes, device-resident "
                       "weights) -> bestla_device_memcpy(D2H logits, pinned) -> bestla_device_sync, per token"}
    if rank == 0 and not args.skip_e2e:
        host_rows = {}
        per = per_layer + [lm]
        # host copies of the Q4_0 rows of the first layer + lm_head; the host ABI uploads/caches them by address
        rng = np.random.default_rng(7)
        hx = rng.standard_normal((1, N_EMBD), dtype=np.float32)
        hh = rng.standard_normal((1, N_FF), dtype=np.float32)
        hw = {}
        for name, n, k in per:
            wt = torch.randn(n, k, device="cuda") * 0.02
            rows = torch.empty(n * (k // 32) * 18, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            assert L.ns_device_quantize_q4_0(C.c_void_p(wt.data_ptr()), C.c_void_p(rows.data_ptr()), n, k, None) == 0
            L.bestla_device_sync(None)
            hw[name] = (rows.cpu().numpy().reshape(n, -1), n, k)
        outs = {name: np.zeros((1, n), np.float32) for name, n, k in per}

        def host_token():
            h2d = d2h = 0
            for _ in range(n_layers):
                for name, n, k in per_layer:
                    rws, nn, kk = hw[name]
                    a = hh if kk == N_FF else hx
                    rc = L.ns_mul_mat_q4_0_f32_host(rws.ctypes.data_as(C.c_void_p), rws.shape[1], a.ctypes.data_as(C.c_void_p),
                                                    outs[name].ctypes.data_as(C.c_void_p), kk, nn, 1)
                    assert rc == 0, ns.last_error()
                    h2d += kk * 4
                    d2h += nn * 4
            rws, nn, kk = hw["lm_head"]
            rc = L.ns_mul_mat_q4_0_f32_host(rws.ctypes.data_as(C.c_void_p), rws.shape[1], hx.ctypes.data_as(C.c_void_p),
                                            outs["lm_head"].ctypes.data_as(C.c_void_p), kk, nn, 1)
            assert rc == 0, ns.last_error()
            return h2d + kk * 4, d2h + nn * 4

        for _ in range(2):
            h2d, d2h = host_token()
        es = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(es):
            host_token()
        dt = (time.perf_counter() - t0) / es
        e2e["host_nodes"] = {"value": 1.0 / dt, "unit": "tokens/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                             "ms_per_step": dt * 1e3, "steps": es,
                             "path": "INTEGRATION.md A: ns_mul_mat_q4_0_f32_host x 225 per token, every node H2D + D2H + sync "
                                     "(host fp32 in/out, pageable), weights device-resident"}
    if rank == 0 and not args.skip_cpu:
        ref = CpuReference(distinct=2)
        tps, spt = ref.time_tokens(2, 1)
        cpu = {"value": tps, "unit": "tokens/s", "cores": ref.threads, "kind": ref.kind,
               "sample": f"2 full tokens (32 layers x 7 matmuls + lm_head) after 1 warm-up, {ref.threads} OpenMP threads"}

    tp_res = None
    if world > 1 and not args.skip_tp:
        # free the 7B replicas first: the TP leg builds its own shards
        try:
            tp_res = run_tp(world, rank, hbm_peak, max(5, min(20, args.steps)))
        except Exception as e:  # the replica numbers stay valid
            import traceback
            tp_res = {"error": repr(e)[:300], "where": traceback.format_exc()[-600:]}
    if rank == 0:
        scale = n_layers / N_LAYER
        traffic, traffic_src = (ncu_traffic("gemv_ring_kernel") if (args.fmt == "q4_0" and n_layers == N_LAYER) else (None, None))
        line = {
            "metric": METRIC if args.fmt == "q4_0" else METRIC.replace("Q4_0", "int4 g128 sym"),
            "value_is": "decode tokens/s (first component of the metric); prefill tok/s is prefill.tokens_per_s",
            "value": world * 1000.0 / ms_step, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8xint4->f32 (q8_0 x q4_0)" if args.fmt == "q4_0" else "u8xint4->f32",
            "data": "synthetic: W~N(0,0.02^2) seed 1234, quantised on device; activations N(0,1)",
            "config": {"workload": f"llama2-7b {args.fmt} decode matmul path, batch 1: {n_gemv} fused weight-only matmuls/token "
                                   f"({n_layers} layers x [QKV, o, gate/up+SiLU*mul, down] + lm_head), Q8_0 activation "
                                   f"quantisation fused into each GEMV, one CUDA graph per token (graph={use_graph})",
                       "weights": int(n_weights), "packed_bytes_per_step": int(alg_bytes),
                       "l2_policy": "inputs (3.7 GB of weights per step) exceed the 126 MB L2; no flush needed",
                       "parallelism": "replicas" if world > 1 else "single"},
            "roofline": {"bound": "hbm", "achieved": step_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": step_gbs / hbm_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, parsed at run time from the
                         # committed ncu launch list of this same command (profiles/r02_launches_bench.csv); null when that
                         # file is absent or the workload differs (other formats / layer counts)
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "gemv_ring_kernel<S8,M=1,sym,f16,NC=14> (one CTA per SM: 14 consumer + 2 producer warps, fused Q8_0 activation quantisation)",
                         "launches_per_step": launches_per_step, "avg_launch_us": ms_step * 1e3 / max(1, launches_per_step),
                         "peak_source": peak_kind, "algorithmic_bytes_per_launch": int(alg_bytes // max(1, launches_per_step)),
                         "note": "the timed region contains only this kernel (129 launches per token, one CUDA graph, PDL)",
                         "per_op_gemv_only": {"kernel": "gemv_ring_kernel<S8,M=1,sym,f16,NC=7> (two CTAs per SM, pre-quantised activation image)", "achieved": gemv_gbs,
                                              "frac": gemv_gbs / hbm_peak, "avg_launch_us": ms_gemv * 1e3 / n_gemv,
                                              "launches": n_gemv}},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "launches_per_step": launches_per_step, "clocks": clocks, "setup_s": setup_s,
            "sustained": {"steps": sus_steps, "ms_per_step": ms_sus, "tokens_per_s": world * 1000.0 / ms_sus,
                          "frac": (alg_bytes / (ms_sus * 1e-3) / 1e9) / hbm_peak, "note": "the same step repeated for >= 1 s"},
            "prefill": prefill, "decode_engine": engine, "configs": configs, "tp": tp_res,
        }
        if n_layers != N_LAYER:
            line["config"]["note"] = f"REDUCED run: {n_layers} of 32 layers (debug only, not a valid bench value)"
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 500; 20 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--fmt", default="q4_0", choices=["q4_0", "int4g128"])
    ap.add_argument("--layers", type=int, default=N_LAYER, help="debug: fewer layers (invalid as a bench value)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-prefill", action="store_true")
    ap.add_argument("--skip-engine", action="store_true")
    ap.add_argument("--gen-tokens", type=int, default=128)
    ap.add_argument("--prefill-tokens", type=int, default=2048)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="skip the BASELINE configs 2-4 legs")
    ap.add_argument("--skip-tp", action="store_true", help="N > 1: skip the Llama-2-70B tensor-parallel leg (config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 500
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
