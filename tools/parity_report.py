"""Achieved parity of the decode step per test case, written to profiles/r2_parity.md.

Default: the persistent decode kernel's cases (tests/test_gpu_mega.CASES): normwise error of its fp32 logits against the
oracle decoder (tests/test_gpu_engine._ref_forward) and against the multi-kernel form, for every generated token.
--long: the cases of tests/test_gpu_engine_long.py (split attention, batch > 2, batch 8 x 2048 prefill, Llama-2-7B geometry
after a long prompt, the last KV slot): worst per-sequence error against the oracle, the bound the test uses, the oracle's
own fp32-vs-fp64 difference at the same rows, and split-vs-unsplit differences.
Each mode rewrites its own section of the file and keeps the other.  --out PATH writes the result to PATH instead."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from test_gpu_mega import CASES, _build
from test_gpu_engine import _ref_forward
from intel_extension_for_transformers_b200.runtime.engine import LlamaGeometry

OUT = os.path.join(ROOT, "profiles", "r2_parity.md")
LONG_HEAD = "## Long contexts, batch > 2, KV-cache end (tests/test_gpu_engine_long.py)"


def persistent_section():
    rows = []
    for case in CASES:
        H, I, L, nh, nkv, V, group, asym, stype, B, T, NEW = case
        geom = LlamaGeometry(hidden=H, inter=I, n_layers=L, n_heads=nh, n_kv_heads=nkv, head_dim=128, vocab=V)
        rng = np.random.default_rng(11)
        eng, layers, embed, fnorm, lm_head = _build(geom, group, asym, stype, rng, max_seq=T + NEW + 8, max_batch=B)
        tokens = rng.integers(0, V, size=(B, T))
        ref = _ref_forward(geom, layers, embed, fnorm, lm_head, tokens, group, stype)
        nxt = ref[:, -1].argmax(-1)
        seq = tokens.copy()
        eng.reset(); eng.prefill(torch.from_numpy(tokens))
        e1, e2, fl = [], [], []
        for step in range(NEW):
            seq = np.concatenate([seq, nxt[:, None]], axis=1)
            pos = seq.shape[1] - 1
            ref_full = _ref_forward(geom, layers, embed, fnorm, lm_head, seq, group, stype)[:, -1]
            eng.decode_host([int(x) for x in nxt], pos)
            lg = eng.last_logits(B).cpu().numpy()
            e1.append(float(np.linalg.norm(lg - ref_full) / np.linalg.norm(ref_full)))
            _, lg2 = eng.decode(torch.from_numpy(nxt.astype(np.int32)), pos, want_logits=True)
            lg2 = lg2.cpu().numpy()
            e2.append(float(np.linalg.norm(lg - lg2) / np.linalg.norm(lg2)))
            if H <= 1024:   # the oracle's own noise floor: fp32 (BLAS) vs fp64 accumulation, same rounding points
                ref64 = _ref_forward(geom, layers, embed, fnorm, lm_head, seq, group, stype, f64=True)[:, -1]
                fl.append(float(np.linalg.norm(ref_full - ref64) / np.linalg.norm(ref64)))
            nxt = ref_full.argmax(-1)
        rows.append((case, max(e1), max(e2), max(fl) if fl else None))
        print(case, "vs oracle %.2e  vs multi-kernel %.2e  oracle fp32-vs-fp64 %s" % (max(e1), max(e2), ("%.2e" % max(fl)) if fl else "-"), flush=True)
        del eng
    out = ["# Persistent decode kernel: achieved parity (normwise error of fp32 logits, worst generated token per case)", "",
           "| hidden | inter | layers | heads/kv | vocab | group | asym | scales | batch | context | vs oracle decoder | vs multi-kernel form | oracle fp32 vs fp64 accumulation (noise floor) |", "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for (H, I, L, nh, nkv, V, group, asym, stype, B, T, NEW), a, b, f in rows:
        out.append(f"| {H} | {I} | {L} | {nh}/{nkv} | {V} | {group} | {asym} | {stype} | {B} | {T}+{NEW} | {a:.2e} | {b:.2e} | {('%.2e' % f) if f is not None else 'not computed (fp64 dequantised weights too large)'} |")
    out += ["", "Both sides round to bf16 at the same points; the residual error is bf16 roundings that flip under a different accumulation order",
            "(the last column shows how much the oracle itself moves between fp32 and fp64 accumulation).  Integer unpack indices, dequantised",
            "weights and RTN codes are bit-exact (tests/test_gpu_qbits.py); a single WOQ linear is within 1e-5 normwise of the fp64 oracle."]
    return "\n".join(out) + "\n"


def long_section():
    import test_gpu_engine_long as T
    dev = torch.cuda.get_device_properties(0)
    try:   # read-only query: the power limit belongs beside the numbers
        import subprocess
        watts = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, check=True).stdout.strip()
        power = f", power limit {float(watts):.0f} W"
    except Exception:
        power = ", power limit not read"
    rows, srows = [], []

    def add(name, path, case, r, tol):
        H = case[0]
        pre = max(T._row_err(r["got"][0], r["ref"][0])) if path != "kv-end" else None
        steps = max(max(T._row_err(g, f)) for g, f in zip(r["got"][1:] if pre is not None else r["got"],
                                                          r["ref"][1:] if pre is not None else r["ref"]))
        floor = max(max(f) for f in r["floor"])
        rows.append((name, path, H, pre, steps, tol, floor))
        print(name, path, "prefill %s  steps %.2e  bound %.1e  floor %.2e" % ("-" if pre is None else "%.2e" % pre, steps, tol, floor), flush=True)

    for c in T.SPLIT_CASES:
        add(T._case_id(c), "persistent", c, T.run_split_case(c, floor=True), c[-1])
    for c in T.BATCH_CASES:
        add(T._batch_id(c), "multi-kernel", c, T.run_batch_case(c, floor=True), c[-1])
    add("batch8_prefill_t2048", "multi-kernel", T.BENCH_PREFILL, T.run_batch_case(T.BENCH_PREFILL, floor=True), T.BENCH_PREFILL[-1])
    add("llama7b_" + T._case_id(T.LLAMA_LONG), "persistent", T.LLAMA_LONG, T.run_split_case(T.LLAMA_LONG, floor=True), T.LLAMA_LONG[-1])
    for p in sorted(T.KV_END):
        r = T.run_kv_end(p, floor=True)
        del r["eng"]
        add("kv_end_" + p, "kv-end", T.KV_END[p], r, T.KV_END[p][-1])

    def setenv(k, v):
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    for c, env in T.SPLIT_VS_UNSPLIT:
        d = T.run_split_vs_unsplit(c, env, setenv)
        worst = max(max(x) for x in d)
        srows.append((T._case_id(c), "default" if env is None else env, worst))
        print("split vs unsplit", c, env, "%.2e" % worst, flush=True)

    out = [LONG_HEAD, "",
           f"Measured on {dev.name} ({dev.multi_processor_count} SMs{power}).  Normwise error of the fp32 logits of each sequence; each column is",
           "the worst sequence over the case's prompt (prefill) or decode steps.  Bound: what the test asserts per sequence.  Noise floor:",
           "the oracle's own fp32-vs-fp64 accumulation difference at the same rows (same bf16 rounding points).", "",
           "| case | path | hidden | prefill vs oracle | decode steps vs oracle | bound | oracle fp32 vs fp64 (noise floor) |",
           "|---|---|---|---|---|---|---|"]
    for name, path, H, pre, steps, tol, floor in rows:
        out.append(f"| {name} | {path} | {H} | {'-' if pre is None else '%.2e' % pre} | {steps:.2e} | {tol:.1e} | {floor:.2e} |")
    out += ["", "Split against unsplit: the same persistent step run with the split attention (default threshold, or QB_MEGA_ATTN_SPLIT as",
            "given) and with it switched off; worst normwise difference of a sequence's logits over the case's steps.", "",
            f"| case | split from | split vs unsplit | bound |", "|---|---|---|---|"]
    for name, env, worst in srows:
        out.append(f"| {name} | {env} | {worst:.2e} | {T.SPLIT_VS_UNSPLIT_TOL:.1e} |")
    return "\n".join(out) + "\n"


if __name__ == "__main__":
    # --out PATH: write the updated report there instead of over profiles/r2_parity.md (which is still read as the base)
    args = sys.argv[1:]
    long_mode = "--long" in args
    dst = args[args.index("--out") + 1] if "--out" in args else OUT
    old = open(OUT).read() if os.path.exists(OUT) else ""
    head, sep, tail = old.partition(LONG_HEAD)
    text = (head.rstrip("\n") + "\n\n" + long_section()) if long_mode else (persistent_section() + ("\n" + sep + tail if sep else ""))
    open(dst, "w").write(text)
