#!/usr/bin/env python
"""bench.py -- Llama-2-7B int4 g128 greedy decode, batch 1 (BASELINE.json configs[1]); one step = one generated token.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

ours:       synthetic GPTQ-style weights (random nibbles, seed 1234, SURVEY.md section 8d), every op a kernel of
            libqbits_b200.so; one decode step = ONE launch of the persistent kernel k_decode_mega (csrc/mega.cu).
            value  = tokens/s with the token fed back on the device (CUDA events on the launching stream)
            e2e    = tokens/s through the host-buffer runtime call (pinned h2d token id + step + d2h token id per step)
            roofline = k_decode_mega: algorithmic bytes of one token (SURVEY.md 8d, KV at the mean context of the timed
                       steps) / the average launch duration inside the timed region; roofline_gemv = the stand-alone WOQ
                       GEMV family (4 launches x 32 layers per pass) that the multi-kernel fallback path uses
            cpu_baseline = the oracle's C port of the reference CPU path on the box's host cores, bounded sample
reference:  the same C port (oracle/woq_cpu.c: the reference's own kernels cannot be built offline) on all host threads.
N > 1:      replicas only in this round (one engine per rank, no collective); value = sum over ranks.
--dump-outputs DIR (ours, rank 0): after the timed steps, what each timed path handed back in its last step, as
            DIR/<name>.npy (float32 / float64).  Weights, prompt and first token are seeded, so two builds run with the
            same arguments can be compared output for output:
            decode_resident_logits [1, vocab]  logits of the last device-resident step
            decode_host_logits     [1, vocab]  logits of the last host-buffer step
            decode_host_token      [1]         the token id that step returned
            prefill_logits         [8, vocab]  last-position logits of the end-to-end prefill (absent without prefill)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "llama2-7b int4(sym) g128 bf16-scales greedy decode, batch=1, ctx 1..steps"
PREFILL_B, PREFILL_S = 8, 2048   # BASELINE.json configs[2]: the other half of the metric (prefill TFLOPS vs roofline)


def common_config():
    """The keys both arms print (the driver compares the two `config` objects)."""
    return {"workload": WORKLOAD, "model": "llama2-7b (synthetic weights)", "weights": "int4 sym g128, bf16 scales", "batch": 1,
            "bytes_per_token_algorithmic": algorithmic_bytes_per_token(0)}


def prefill_flops():
    """SURVEY.md section 8d: WOQ linears 2*M*6476005376 + causal attention + lm_head on the last position only."""
    H, L, V = GEOM["hidden"], GEOM["n_layers"], GEOM["vocab"]
    M = PREFILL_B * PREFILL_S
    lin = 2.0 * M * 6476005376
    attn = L * 2.0 * (2.0 * PREFILL_B * GEOM["n_heads"] * PREFILL_S * PREFILL_S * GEOM["head_dim"]) / 2.0
    lm = 2.0 * PREFILL_B * V * H
    return lin, attn, lm
GEOM = dict(hidden=4096, inter=11008, n_layers=32, n_heads=32, n_kv_heads=32, head_dim=128, vocab=32000)
GROUP = 128


def algorithmic_bytes_per_token(ctx=0):
    """SURVEY.md section 8d: packed int4 + bf16 scales + bf16 lm_head (+ bf16 KV at context ctx)."""
    H, I, L, V = GEOM["hidden"], GEOM["inter"], GEOM["n_layers"], GEOM["vocab"]
    params = L * (4 * H * H + 3 * H * I)
    return params // 2 + (params // GROUP) * 2 + V * H * 2 + 2 * L * H * ctx * 2


class ClockSampler:
    def __init__(self, idx=0):
        self.samples, self.reasons, self._stop, self.idx = [], set(), threading.Event(), idx
        self.stamps = []   # perf_counter of every NVML sample: lets a block report the clocks of its own window
        self.max_mhz = None

    def _run(self):
        # NVML in-process (nvidia_ml_py): a query costs ~0.1 ms and takes no global driver lock; spawning nvidia-smi every
        # 200 ms was measured to add ~35 us per token to the end-to-end loop it is supposed to observe
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            while not self._stop.is_set():
                self.samples.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                self.stamps.append(time.perf_counter())
                r = int(get_reasons(h))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                self._stop.wait(0.05)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.5)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=3)

    def window(self, t0, t1):
        """median SM clock of the samples taken between two perf_counter stamps (None without NVML)"""
        w = sorted(c for c, t in zip(self.samples, self.stamps) if t0 <= t <= t1)
        return w[len(w) // 2] if w else None

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------- CPU baseline
def cpu_tokens_per_s(budget_s=15.0, n_distinct_layers=4, ctx0=8):
    """Reference CPU path (C port, oracle/woq_cpu.c) on the host cores: full-depth single-token decode steps INCLUDING the
    attention over a growing context (RoPE, KV append, softmax over pos + 1 keys).  Weights: 4 distinct synthetic decoder
    layers cycled 8x (404 MB > any LLC) + the bf16 lm_head.  The thread count is calibrated first (one layer timed at
    all / half / quarter ... of the usable CPUs, fastest kept): an all-CPUs spinning pool collapses on a host whose
    cgroup quota or other tenants leave fewer CPUs than sched_getaffinity shows.  >= 3 warm-up tokens, then as many whole
    tokens as fit in ~budget_s.  Returns (tokens/s, threads used, sample description, GB/s of algorithmic bytes)."""
    import ctypes as C
    import numpy as np
    from oracle import cpu_port
    lib = cpu_port.lib()
    H, I, L, V, D = GEOM["hidden"], GEOM["inter"], GEOM["n_layers"], GEOM["vocab"], GEOM["head_dim"]
    NH, NKV = GEOM["n_heads"], GEOM["n_kv_heads"]
    rng = np.random.default_rng(1234)

    def lin(K, N):
        qw = rng.integers(-2**31, 2**31 - 1, size=(K // 8, N), dtype=np.int64).astype(np.int32)
        sc = ((0.5 + rng.random((K // GROUP, N), dtype=np.float32)) * (2.0 / 15.0) * 0.02).astype(np.float32)
        return qw, sc

    layers = [dict(qkv=lin(H, 3 * H), o=lin(H, H), gu=lin(H, 2 * I), d=lin(I, H)) for _ in range(n_distinct_layers)]
    lm = rng.integers(0, 2**16, size=(V, H), dtype=np.uint16) & 0xBFFF  # finite bf16 bit patterns
    lm = np.ascontiguousarray((lm & 0x807F) | 0x3C00).astype(np.uint16)  # |w| ~ 0.01
    ones = np.ones(H, np.float32)
    h = (rng.standard_normal(H) * 0.1).astype(np.float32)
    tmax = 128
    scratch = np.zeros(H + 3 * H + 2 * I + I + H + tmax + 64, np.float32)
    kc = (rng.standard_normal((L, NKV, tmax, D)) * 0.1).astype(np.float32)   # pre-filled context of ctx0 tokens
    vc = (rng.standard_normal((L, NKV, tmax, D)) * 0.1).astype(np.float32)
    logits = np.zeros(V, np.float32)
    fp = C.POINTER(C.c_float)
    i32 = C.POINTER(C.c_int32)

    def layer(hh, l, pos):
        w = layers[l % n_distinct_layers]
        lib.llama_layer_decode_f32(hh.ctypes.data_as(fp), H, I, NH, NKV, D, GROUP,
                                   w["qkv"][0].ctypes.data_as(i32), w["qkv"][1].ctypes.data_as(fp),
                                   w["o"][0].ctypes.data_as(i32), w["o"][1].ctypes.data_as(fp),
                                   w["gu"][0].ctypes.data_as(i32), w["gu"][1].ctypes.data_as(fp),
                                   w["d"][0].ctypes.data_as(i32), w["d"][1].ctypes.data_as(fp),
                                   ones.ctypes.data_as(fp), ones.ctypes.data_as(fp), 1e-5,
                                   kc[l].ctypes.data_as(fp), vc[l].ctypes.data_as(fp), int(pos), tmax, 10000.0, scratch.ctypes.data_as(fp))

    def token(pos):
        hh = h.copy()
        for l in range(L):
            layer(hh, l, pos)
        lib.dense_bf16_f32(hh.ctypes.data_as(fp), 1, H, lm.ctypes.data_as(C.POINTER(C.c_uint16)), V, logits.ctypes.data_as(fp))
        return int(logits.argmax())

    nt = cpu_port.threads()
    cands = sorted({max(1, nt >> k) for k in range(0, 5)} | {min(nt, 16), min(nt, 32)}, reverse=True)
    best_n, best_t = nt, None
    hh = h.copy()
    for n in cands:
        lib.woq_cpu_set_active(n)
        for l in range(n_distinct_layers):
            layer(hh, l, ctx0)                      # warm this count (pool start, page faults)
        t0 = time.perf_counter()
        for rep in range(2):
            for l in range(n_distinct_layers):
                layer(hh, l, ctx0)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_n, best_t = n, dt
    lib.woq_cpu_set_active(best_n)
    pos = ctx0
    for _ in range(3):                               # warm-up tokens
        token(pos)
        pos += 1
    n, t0 = 0, time.perf_counter()
    while True:
        token(min(pos, tmax - 1))
        pos += 1
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 64:
            break
    gbs = algorithmic_bytes_per_token(ctx0) * n / dt / 1e9
    sample = (f"{n} full-depth tokens incl. attention (ctx {ctx0}+, {n_distinct_layers} distinct synthetic layers cycled x{L // n_distinct_layers} "
              f"+ lm_head), {dt:.1f} s, {best_n} of {nt} threads (calibrated, {'pinned' if cpu_port.pinned() else 'unpinned'}), {gbs:.1f} GB/s")
    return n / dt, best_n, sample, gbs


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps = max(1, args.steps)
    # each "step" is a bounded sample: one whole token; K steps + W warm-ups must end within minutes
    per_step_budget = max(1.0, min(20.0, 120.0 / (steps + args.warmup)))
    # one measurement covers warm-up + timed tokens (the port is deterministic work per token)
    v, cores, sample, gbs = cpu_tokens_per_s(budget_s=min(60.0, per_step_budget * steps))
    print(json.dumps({
        "impl": "reference", "metric": "decode tokens/sec (Llama-2-7B int4 g128, batch 1)", "value": v, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32 accumulate over int4 weights (CPU)", "data": "synthetic",
        "config": common_config(),
        "note": "reference CPU path restated in C (oracle/woq_cpu.c); BesTLA itself cannot be built offline",
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample, "gb_per_s": gbs},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def write_outputs(out_dir, outputs):
    """Each tensor as out_dir/<name>.npy: float64 stays float64, every other dtype is stored as float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t if t.dtype == torch.float64 else t.float()).numpy())


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from intel_extension_for_transformers_b200 import _capi
    from intel_extension_for_transformers_b200.runtime.engine import LlamaEngine, LlamaGeometry
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    lib = _capi.lib()
    geom = LlamaGeometry(**GEOM)
    max_seq = args.warmup + 2 * args.steps + 64
    do_prefill = not os.environ.get("QB_BENCH_SKIP_PREFILL")
    eng = LlamaEngine.synthetic(geom, group=GROUP, weight_dtype="int4_clip", scale_dtype="bf16", asym=False, seed=1234 + rank,
                                max_seq=max(256, max_seq, PREFILL_S + 8 if do_prefill else 0),
                                max_batch=PREFILL_B if do_prefill else 1, device=dev)
    torch.cuda.synchronize()
    eng.reset()
    launches0 = lib.qb_launch_count()
    tok, pos = [1], 0
    for _ in range(max(3, args.warmup)):        # warm-up through the host path (also builds the graph)
        tok = eng.decode_host(tok, pos)
        pos += 1
    eng.decode_resident(1, pos, 3)               # builds + warms the resident graph
    pos += 3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with ClockSampler(local_rank) as clk:
        # ---- device-resident: K steps, CUDA events on the launching stream
        barrier()
        ctx_first = pos
        ms_dev = eng.decode_resident(1, pos, args.steps)
        pos += args.steps
        barrier()
        outputs = {}
        if args.dump_outputs:
            outputs["decode_resident_logits"] = eng.last_logits(1)
        # ---- end to end: host token in, host token out, every step
        tok = eng.decode_host(tok, pos)
        pos += 1
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tok = eng.decode_host(tok, pos)
            pos += 1
        torch.cuda.synchronize()
        ms_e2e = (time.perf_counter() - t0) * 1e3
        barrier()
        if args.dump_outputs:
            outputs["decode_host_logits"] = eng.last_logits(1)
            outputs["decode_host_token"] = torch.tensor(tok, dtype=torch.float64)
        # ---- dominant kernel family alone
        ms_lin, bytes_lin, n_lin = eng.time_linears(1, reps=5)
        # ---- prefill, B=8 x S=2048 (configs[2]): device time per op class by CUDA events, then end to end from host ids
        pre = None
        if do_prefill:
            ptok = torch.randint(0, GEOM["vocab"], (PREFILL_B, PREFILL_S), generator=torch.Generator().manual_seed(99), dtype=torch.int32)
            ptok_pin = ptok.pin_memory()
            eng.reset(); eng.prefill(ptok); torch.cuda.synchronize()          # warm-up (scratch allocation, tensor maps)
            eng.reset(); eng.prefill(ptok); torch.cuda.synchronize()
            best = None
            t_pre0 = time.perf_counter()
            for _ in range(3):
                barrier()
                eng.reset()
                _, pr = eng.prefill_profile(ptok)
                if best is None or pr["total_ms"] < best["total_ms"]:
                    best = pr
            barrier()
            eng.reset()
            t0 = time.perf_counter()
            lg = eng.prefill(ptok_pin.to(dev, non_blocking=True))              # h2d of the ids inside the timed region
            first = torch.argmax(lg, dim=-1).cpu()                              # d2h of the first generated ids
            pre_e2e_ms = (time.perf_counter() - t0) * 1e3
            pre = (best, pre_e2e_ms, int(first[0]))
            if args.dump_outputs:
                outputs["prefill_logits"] = lg
            pre_clock = clk.window(t_pre0, time.perf_counter())
    launches = lib.qb_launch_count() - launches0
    # ---- N > 1 only: ONE model sharded over the N GPUs (Megatron column/row split, partial sums exchanged through NVLink peer
    # memory inside the GEMV epilogue; runtime/tp.py + csrc/comm.cu).  Reported beside the replica number, never instead of it.
    tp_ms = None
    if world > 1 and not os.environ.get("QB_BENCH_SKIP_TP") and geom.n_kv_heads % world == 0:
        tpe = LlamaEngine.synthetic(geom, group=GROUP, weight_dtype="int4_clip", scale_dtype="bf16", asym=False, seed=4321,
                                    max_seq=max(256, args.steps + 64), max_batch=1, device=dev, tp_rank=rank, tp_size=world)
        tpe.connect_tp()
        tpe.reset()
        tpe.prefill(torch.ones((1, 8), dtype=torch.int32))
        tpe.decode_resident(1, 8, 8)
        barrier()
        tp_ms = tpe.decode_resident(1, 16, args.steps)
        tp_mode = tpe.step_mode(1)
        barrier()
    if world > 1:
        t = torch.tensor([ms_dev, ms_e2e, pre[0]["total_ms"] if pre else 0.0, pre[1] if pre else 0.0, tp_ms or 0.0], device=dev,
                         dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e, pre_total, pre_e2e, tp_max = t.tolist()
        if tp_ms is not None:
            tp_ms = tp_max
        if pre:
            pre[0]["total_ms"], pre = pre_total, (pre[0], pre_e2e, pre[2])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    value = world * args.steps / (ms_dev / 1e3)
    e2e = world * args.steps / (ms_e2e / 1e3)
    achieved_gemv = bytes_lin / (ms_lin / 1e3) / 1e9
    mega = "megakernel" in eng.step_mode(1)
    ctx_mean = ctx_first + (args.steps - 1) / 2.0
    bytes_step = algorithmic_bytes_per_token(ctx_mean)
    us_launch = ms_dev * 1e3 / args.steps           # the timed region is exactly K launches of the step kernel
    achieved = bytes_step / (us_launch * 1e-6) / 1e9
    if os.environ.get("QB_BENCH_SKIP_CPU"):
        cpu_v, cpu_cores, cpu_sample, cpu_gbs = None, None, "skipped (QB_BENCH_SKIP_CPU)", None
    else:
        cpu_v, cpu_cores, cpu_sample, cpu_gbs = cpu_tokens_per_s(budget_s=15.0)
    prefill = None
    if pre:
        pr, pre_e2e_ms, _ = pre
        lin_f, attn_f, lm_f = prefill_flops()
        tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
        tot_f = lin_f + attn_f + lm_f
        prefill = {
            "workload": f"llama2-7b int4 g128 prefill, batch {PREFILL_B} x seq {PREFILL_S} (M = {PREFILL_B * PREFILL_S}), per GPU",
            "ms": pr["total_ms"], "prompt_tokens_per_s": world * PREFILL_B * PREFILL_S / (pr["total_ms"] / 1e3),
            "tflops": tot_f / (pr["total_ms"] / 1e3) / 1e12, "flop": tot_f,
            "peak_tflops": tf_peak, "peak_kind": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if "bf16_tflops_sustained" in peaks else "fallback 1400",
            "frac": tot_f / (pr["total_ms"] / 1e3) / 1e12 / tf_peak,
            "split_ms": {"woq_gemm": pr["gemm_ms"], "attention": pr["attention_ms"], "other": pr["other_ms"]},
            "woq_gemm_tflops": lin_f / (pr["gemm_ms"] / 1e3) / 1e12, "attention_tflops": attn_f / (pr["attention_ms"] / 1e3) / 1e12,
            "e2e_ms": pre_e2e_ms, "e2e_prompt_tokens_per_s": world * PREFILL_B * PREFILL_S / (pre_e2e_ms / 1e3),
            "h2d_bytes": PREFILL_B * PREFILL_S * 4, "d2h_bytes": PREFILL_B * 8,
            "sm_mhz_during_prefill": pre_clock,
        }
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "mega_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        pass
    print(json.dumps({
        "metric": "decode tokens/sec (Llama-2-7B int4 g128, batch 1)", "value": value, "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16 activations x int4 weights, fp32 accumulate", "data": "synthetic",
        "config": common_config(),
        "run": {"parallelism": f"replicas x{world}" if world > 1 else "single GPU", "step_kernel": eng.step_mode(1),
                "l2": "weights 3.34 GB/token >> 126 MB L2 (inputs larger than L2)",
                "hbm_roofline_tokens_per_s": peak * 1e9 / algorithmic_bytes_per_token(0),
                "whole_step_frac_of_hbm_roofline": (args.steps / (ms_dev / 1e3)) * algorithmic_bytes_per_token(0) / (peak * 1e9)},
        "prefill": prefill,
        "tensor_parallel": None if tp_ms is None else {
            "parallelism": f"tp{world}", "scaling": "strong", "workload": "the same batch-1 decode, ONE model sharded over the GPUs",
            "tokens_per_s": args.steps / (tp_ms / 1e3), "ms_per_token": tp_ms / args.steps, "step_kernel": tp_mode,
            "vs_one_gpu": (args.steps / (tp_ms / 1e3)) / (value / world)},
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": 4, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "k_decode_mega (one launch = one token)" if mega else "decode step (CUDA graph of 5L+3 kernels)",
                     "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak,
                     "bytes_per_launch": bytes_step, "us_per_launch": us_launch, "ctx_mean": ctx_mean, "traffic": traffic},
        "roofline_gemv": {"kernel": "k_woq_gemv (all WOQ linears of a step, stand-alone launches)", "achieved": achieved_gemv,
                          "unit": "GB/s", "frac": achieved_gemv / peak, "bytes_per_launch_avg": bytes_lin / n_lin,
                          "us_per_launch_avg": ms_lin * 1e3 / n_lin},
        "cpu_baseline": {"value": cpu_v, "unit": "tokens/s", "cores": cpu_cores, "kind": "port", "sample": cpu_sample, "gb_per_s": cpu_gbs},
        "clocks": clk.summary(),
    }))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed steps to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
