"""GPU: the decode step at long contexts, batch sizes above 2 and the ends of the KV cache, against the oracle decoder.

The other engine tests stay at short contexts and batch <= 2.  Here:
  - the persistent kernel's split attention (csrc/mega.cu: past `attn_split_min` cached tokens, the tokens of each
    (sequence, head) pair are split over ns = min(4, grid / pairs) CTAs and merged by part 0), for ns = 1, 2, 3 and 4,
    at contexts around the threshold, not a multiple of ns x 16 warps, and near 2048;
  - the same step with the split and without it: both round at the same points and differ only in the fp32 merge order,
    so this comparison resolves far finer than the oracle's own fp32-vs-fp64 noise;
  - the multi-kernel form at batch 3, 5, 8 and 16 (k_lm_head<4> partial and repeated passes, a KV cache laid out for more
    sequences than run), eager and CUDA graph;
  - the benchmark's prefill shape (batch 8 x 2048) and a decode step after it;
  - a Llama-2-7B-geometry step after a ~1000-token prompt;
  - the last KV slot, and the refusal of the step after it.
Every comparison is per sequence: a whole-batch norm would let one bad row hide.  The oracle runs one sequence at a time
(O.attention's fp64 score matrix stays [heads, T, T]) and computes the logits of every checked position in one pass: the
fed tokens are drawn up front (teacher forcing), so prefill and each decode step read their rows out of the same forward.
Prefill positions that ran through the tensor-core GEMM (64 rows or more) are computed by the oracle with bf16-rounded
dequantised weights, as that GEMM does.  The normwise bounds are ~3x the errors measured on a B200; profiles/r2_parity.md
lists them with the oracle's noise floor (tools/parity_report.py --long)."""
import numpy as np
import pytest
import torch

from test_gpu_engine import _ref_forward  # tests/ is on sys.path (rootdir conftest)
from test_gpu_mega import _build

pytestmark = pytest.mark.gpu

# csrc/mega.h MG_PS (CTAs that may share one 16-row strip), csrc/blob.h QB_TILE_K (k per weight tile), and the default
# of QB_MEGA_ATTN_SPLIT in csrc/engine.cu mega_launch (cached tokens from which the persistent kernel splits attention)
MG_PS, TILE_K, SPLIT_MIN = 8, 256, 160


def _geom(H, I, nh, nkv, V, L=2):
    from intel_extension_for_transformers_b200.runtime.engine import LlamaGeometry
    return LlamaGeometry(hidden=H, inter=I, n_layers=L, n_heads=nh, n_kv_heads=nkv, head_dim=128, vocab=V)


def _mega_grid(geom):
    """CTAs of the persistent kernel, as engine.cu mega_prepare sizes it: one per SM, but no more than keeps every 16-row
    strip of every linear shared by at most MG_PS CTAs."""
    D = geom.head_dim
    grid = torch.cuda.get_device_properties(0).multi_processor_count
    for K, N in [(geom.hidden, (geom.n_heads + 2 * geom.n_kv_heads) * D), (geom.n_heads * D, geom.hidden),
                 (geom.hidden, 2 * geom.inter), (geom.inter, geom.hidden)]:
        T, S = -(-K // TILE_K), -(-N // 16)
        grid = min(grid, max(1, S * T // -(-T // (MG_PS - 2))))
    return grid


def _split(geom, batch, pos, split_min=SPLIT_MIN):
    """Parts the persistent kernel cuts each (sequence, head) pair's cached tokens into at this position (mega.cu)."""
    return max(1, min(4, _mega_grid(geom) // (batch * geom.n_heads))) if pos >= split_min else 1


def _ref_rows(model, group, stype, tokens, last, prompt, f64=False):
    """Oracle logits [B, last, V] of the last `last` positions of every sequence of tokens [B, T], one sequence at a time.
    `prompt`: positions the engine prefilled; a prefill of 64 rows or more (batch x prompt) runs the tensor-core GEMM, whose
    dequantised weights are bf16 (engine.cu linear, gemm_tc.cu), and the oracle rounds them the same way for those positions."""
    geom, layers, embed, fnorm, lm_head = model
    wround = prompt if tokens.shape[0] * prompt >= 64 else 0
    return np.concatenate([_ref_forward(geom, layers, embed, fnorm, lm_head, tokens[b:b + 1], group, stype, f64=f64, last=last,
                                        wround=wround) for b in range(tokens.shape[0])])


def _row_err(got, ref):
    return np.linalg.norm(got - ref, axis=-1) / np.linalg.norm(ref, axis=-1)


def _check_rows(got, ref, tol, what):
    """Per sequence: normwise error, and the argmax wherever the oracle's top-2 margin is clear (test_gpu_engine's rule)."""
    err = _row_err(got, ref)
    assert (err < tol).all(), (what, err)
    top2 = np.sort(ref, axis=-1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 0.05 * np.abs(top2[:, 1])
    assert (got.argmax(-1)[clear] == ref.argmax(-1)[clear]).all(), (what, got.argmax(-1), ref.argmax(-1))
    return err


# The last field of every case below is its normwise bound against the oracle decoder: ~3x the worst per-sequence error
# measured on a B200 over the prompt and the decode steps (profiles/r2_parity.md).  What is left is bf16 roundings that
# flip under a different accumulation order; the oracle's own fp32-vs-fp64 difference at the same rows is of the same size
# (up to ~2e-2 at the toy widths, where one flipped rounding of an activation moves a logit by ~2^-9 of it).


def _case_id(c):
    return "h%d_%dx%d_b%d_t%d_ns%d" % (c[0], c[2], c[3], c[8], c[9], c[11])


# ---------------------------------------------------------------------------------------------------------------------
# 1. persistent kernel, split attention, against the oracle
SPLIT_CASES = [
    # hidden, inter, heads, kv heads, vocab, group, asym, scale type, batch, prompt, new tokens, ns past the threshold, bound
    # (on a 148-SM B200: grid 16 for hidden 256 / inter 512, 128 for hidden 512 / inter 1024, 148 for Llama-2-7B)
    (256, 512, 2, 1, 1000, 128, False, "bf16", 1, 159, 3, 4, 3e-2),      # steps at 159 | 160 | 161: unsplit, then split
    (256, 512, 2, 1, 1000, 128, True, "fp32", 2, 1021, 2, 4, 2.5e-2),    # 1021 cached tokens: not a multiple of ns x 16 warps
    (512, 1024, 32, 8, 1000, 128, False, "bf16", 2, 1021, 2, 2, 1.5e-2), # 64 pairs on 128 CTAs, GQA 4:1
    (512, 1024, 40, 8, 1000, 64, False, "bf16", 1, 1021, 2, 3, 1e-2),    # 40 pairs
    (512, 1024, 40, 8, 1000, 128, True, "bf16", 2, 1021, 2, 1, 5.5e-2),  # 80 pairs: past the threshold, but one CTA per pair
    (256, 512, 2, 2, 1000, 32, False, "bf16", 1, 2045, 2, 4, 3e-2),      # near 2048
]


def run_split_case(case, floor=False):
    """Prefill, then the case's decode steps as the persistent kernel (max_seq = prompt + new: the last step writes the
    last KV slot).  Returns per-row errors: prefill and every step against the oracle (and, with floor=True, the oracle's
    fp32-vs-fp64 difference at the same rows)."""
    H, I, nh, nkv, V, group, asym, stype, B, T, NEW, ns, _ = case
    geom = _geom(H, I, nh, nkv, V)
    rng = np.random.default_rng(23)
    eng, *model = _build(geom, group, asym, stype, rng, max_seq=T + NEW, max_batch=B)
    model = (geom, *model)
    assert "persistent" in eng.step_mode(B), "this geometry must be eligible for the persistent kernel"
    seq = rng.integers(0, V, size=(B, T + NEW))
    ref = _ref_rows(model, group, stype, seq, NEW + 1, T)
    eng.reset()
    got = [eng.prefill(torch.from_numpy(seq[:, :T])).cpu().numpy()]
    for pos in range(T, T + NEW):
        assert _split(geom, B, pos) == (ns if pos >= SPLIT_MIN else 1), (pos, _mega_grid(geom))
        tok = eng.decode_host(seq[:, pos].tolist(), pos)
        got.append(eng.last_logits(B).cpu().numpy())
        assert tok == got[-1].argmax(-1).tolist(), "argmax inside the kernel disagrees with its own logits"
    out = dict(got=got, ref=[ref[:, j] for j in range(NEW + 1)])
    if floor:
        ref64 = _ref_rows(model, group, stype, seq, NEW + 1, T, f64=True)
        out["floor"] = [_row_err(ref[:, j], ref64[:, j]) for j in range(NEW + 1)]
    del eng
    return out


@pytest.mark.timeout(600)
@pytest.mark.parametrize("case", SPLIT_CASES, ids=_case_id)
def test_persistent_split_attention_matches_oracle(case):
    r = run_split_case(case)
    for j, (got, ref) in enumerate(zip(r["got"], r["ref"])):
        _check_rows(got, ref, case[-1], "prefill" if j == 0 else "step %d" % j)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the same step with and without the split.  Not at the benchmark geometry with batch 2: its steps are not bit-
# reproducible (test_gpu_mega.test_batch2_benchmark_geometry_is_bit_reproducible), which would blur this comparison.
UNSPLIT = "1000000"
SPLIT_VS_UNSPLIT = [
    # case as above (without a bound) + the QB_MEGA_ATTN_SPLIT value of the split run (None: the default threshold)
    ((256, 512, 2, 1, 1000, 128, False, "bf16", 1, 1021, 2, 4), None),
    ((512, 1024, 32, 8, 1000, 128, False, "bf16", 2, 1021, 2, 2), None),
    ((512, 1024, 40, 8, 1000, 64, True, "fp32", 1, 1021, 2, 3), None),
    ((256, 512, 2, 1, 1000, 128, False, "bf16", 2, 1, 3, 4), "1"),   # forced at contexts 1..3: parts without any token
]
# Normwise bound of split against unsplit logits.  Measured on a B200: 0 in three cases (no bf16 rounding of an attention
# output flips under the other merge order) and 2.7e-3 in one (one flip, cascaded through the later layers); ~3x that.
SPLIT_VS_UNSPLIT_TOL = 8e-3


def run_split_vs_unsplit(case, split_env, setenv):
    """Per decode step: the persistent step with the split (default threshold or `split_env`) and then the same step
    (same position, same cached tokens) with the split switched off.  Returns the per-row differences."""
    H, I, nh, nkv, V, group, asym, stype, B, T, NEW, ns = case
    geom = _geom(H, I, nh, nkv, V)
    rng = np.random.default_rng(29)
    eng, *_ = _build(geom, group, asym, stype, rng, max_seq=T + NEW, max_batch=B)
    assert "persistent" in eng.step_mode(B)
    split_min = int(split_env) if split_env else SPLIT_MIN
    seq = rng.integers(0, V, size=(B, T + NEW))
    eng.reset()
    eng.prefill(torch.from_numpy(seq[:, :T]))
    diffs = []
    for pos in range(T, T + NEW):
        assert _split(geom, B, pos, split_min) == ns, (pos, _mega_grid(geom))
        assert _split(geom, B, pos, int(UNSPLIT)) == 1
        setenv("QB_MEGA_ATTN_SPLIT", split_env)
        eng.decode_host(seq[:, pos].tolist(), pos)
        la = eng.last_logits(B).cpu().numpy()
        setenv("QB_MEGA_ATTN_SPLIT", UNSPLIT)
        eng.decode_host(seq[:, pos].tolist(), pos)   # re-writes the same KV slot
        lb = eng.last_logits(B).cpu().numpy()
        setenv("QB_MEGA_ATTN_SPLIT", None)
        diffs.append(_row_err(la, lb))
    del eng
    return diffs


@pytest.mark.parametrize("case,split_env", SPLIT_VS_UNSPLIT,
                         ids=lambda c: _case_id(c) if isinstance(c, tuple) else ("split_default" if c is None else "split_from_" + c))
def test_split_attention_matches_unsplit_step(case, split_env, monkeypatch):
    def setenv(k, v):
        monkeypatch.setenv(k, v) if v is not None else monkeypatch.delenv(k, raising=False)
    for step, err in enumerate(run_split_vs_unsplit(case, split_env, setenv)):
        assert (err < SPLIT_VS_UNSPLIT_TOL).all(), (step, err)


# ---------------------------------------------------------------------------------------------------------------------
# 3. multi-kernel form at batch > 2
BATCH_CASES = [
    # hidden, inter, heads, kv heads, vocab, group, asym, scale type, batch, max_batch, prompt, new tokens, bound
    (256, 512, 2, 1, 1000, 128, False, "bf16", 3, 16, 40, 3, 3e-2),     # KV cache laid out for 16; lm_head: one pass, 1 padding row
    (256, 512, 2, 2, 1000, 64, True, "fp32", 5, 5, 33, 3, 8.5e-2),      # lm_head: a second pass with one row
    (256, 768, 4, 2, 777, 128, False, "bf16", 8, 8, 24, 3, 5.5e-2),     # two full passes; GQA 2:1
    (256, 512, 2, 1, 1000, 128, False, "bf16", 16, 16, 20, 2, 3.5e-2),  # four passes
]


def _batch_id(c):
    return "h%d_%dx%d_b%d_maxb%d_t%d" % (c[0], c[2], c[3], c[8], c[9], c[10])


def run_batch_case(case, floor=False):
    """Prefill a different prompt per sequence, then the decode steps eagerly (decode) and, after a fresh prefill, through
    the CUDA graph (decode_host).  Returns the eager logits, the oracle's rows and both token streams."""
    H, I, nh, nkv, V, group, asym, stype, B, MB, T, NEW, _ = case
    geom = _geom(H, I, nh, nkv, V)
    rng = np.random.default_rng(31)
    eng, *model = _build(geom, group, asym, stype, rng, max_seq=T + NEW, max_batch=MB)
    model = (geom, *model)
    assert "persistent" not in eng.step_mode(B)
    seq = rng.integers(0, V, size=(B, T + NEW))
    ref = _ref_rows(model, group, stype, seq, NEW + 1, T)
    eng.reset()
    got = [eng.prefill(torch.from_numpy(seq[:, :T])).cpu().numpy()]
    eager = []
    for pos in range(T, T + NEW):
        tok, lg = eng.decode(torch.from_numpy(seq[:, pos].astype(np.int32)), pos, want_logits=True)
        got.append(lg.cpu().numpy())
        eager.append(tok.cpu().tolist())
    eng.reset()
    eng.prefill(torch.from_numpy(seq[:, :T]))
    graph = [eng.decode_host(seq[:, pos].tolist(), pos) for pos in range(T, T + NEW)]
    out = dict(got=got, ref=[ref[:, j] for j in range(NEW + 1)], eager=eager, graph=graph)
    if floor:
        ref64 = _ref_rows(model, group, stype, seq, NEW + 1, T, f64=True)
        out["floor"] = [_row_err(ref[:, j], ref64[:, j]) for j in range(NEW + 1)]
    del eng
    return out


@pytest.mark.timeout(300)
@pytest.mark.parametrize("case", BATCH_CASES, ids=_batch_id)
def test_multikernel_batch_matches_oracle(case):
    r = run_batch_case(case)
    for j, (got, ref) in enumerate(zip(r["got"], r["ref"])):
        _check_rows(got, ref, case[-1], "prefill" if j == 0 else "step %d" % j)
    for j, (tok, got) in enumerate(zip(r["eager"], r["got"][1:])):
        assert tok == got.argmax(-1).tolist(), j
    assert r["graph"] == r["eager"]


# ---------------------------------------------------------------------------------------------------------------------
# 4. the benchmark's prefill shape on a toy-width model, then one multi-kernel decode step at position 2048
BENCH_PREFILL = (256, 512, 2, 1, 1000, 128, False, "bf16", 8, 8, 2048, 1, 4.5e-2)


@pytest.mark.timeout(900)
def test_batch8_prefill_2048_and_next_step_match_oracle():
    """tcgen05 GEMM at M = 16384 with the fused epilogues, tcgen05 attention at 2048 x batch 8, k_gather_rows, lm_head at
    batch 8; then k_attn_decode over 2048 cached tokens per sequence."""
    r = run_batch_case(BENCH_PREFILL)
    _check_rows(r["got"][0], r["ref"][0], BENCH_PREFILL[-1], "prefill")
    _check_rows(r["got"][1], r["ref"][1], BENCH_PREFILL[-1], "step at 2048")
    assert r["graph"] == r["eager"]


# ---------------------------------------------------------------------------------------------------------------------
# 5. Llama-2-7B geometry (2 layers), batch 1, after a ~1000-token prompt: 32 pairs on 148 CTAs, ns = 4
LLAMA_LONG = (4096, 11008, 32, 32, 32000, 128, False, "bf16", 1, 999, 2, 4, 6.5e-3)


@pytest.mark.timeout(900)
def test_llama7b_geometry_long_context_persistent_step():
    r = run_split_case(LLAMA_LONG)
    for j, (got, ref) in enumerate(zip(r["got"], r["ref"])):
        _check_rows(got, ref, LLAMA_LONG[-1], "prefill" if j == 0 else "step %d" % j)


# ---------------------------------------------------------------------------------------------------------------------
# 6. the end of the KV cache
KV_END = {
    # hidden, inter, heads, kv heads, vocab, group, asym, scale type, batch, max_batch, prompt, new tokens, bound
    "persistent": (256, 512, 2, 1, 1000, 128, False, "bf16", 1, 2, 29, 3, 1.7e-2),
    "multikernel": (256, 512, 2, 1, 1000, 128, True, "fp32", 3, 4, 29, 3, 4e-2),
}


def run_kv_end(path, floor=False):
    """max_seq = prompt + new: every step through decode_host, the last one writing KV slot max_seq - 1.  Returns the logits,
    the oracle's rows and the engine with the token that would come next."""
    H, I, nh, nkv, V, group, asym, stype, B, MB, T, NEW, _ = KV_END[path]
    geom = _geom(H, I, nh, nkv, V)
    rng = np.random.default_rng(37)
    max_seq = T + NEW
    eng, *model = _build(geom, group, asym, stype, rng, max_seq=max_seq, max_batch=MB)
    model = (geom, *model)
    assert ("persistent" in eng.step_mode(B)) == (path == "persistent")
    seq = rng.integers(0, V, size=(B, max_seq + 1))
    ref = _ref_rows(model, group, stype, seq[:, :max_seq], NEW, T)
    eng.reset()
    eng.prefill(torch.from_numpy(seq[:, :T]))
    got = []
    for pos in range(T, max_seq):
        eng.decode_host(seq[:, pos].tolist(), pos)
        got.append(eng.last_logits(B).cpu().numpy())
    out = dict(got=got, ref=[ref[:, j] for j in range(NEW)], eng=eng, next=seq[:, max_seq], max_seq=max_seq)
    if floor:
        ref64 = _ref_rows(model, group, stype, seq[:, :max_seq], NEW, T, f64=True)
        out["floor"] = [_row_err(ref[:, j], ref64[:, j]) for j in range(NEW)]
    return out


@pytest.mark.parametrize("path", sorted(KV_END))
def test_last_kv_slot_matches_oracle_then_full_cache_is_refused(path):
    """The last step writes slot max_seq - 1 and is checked; the step after it is refused on the host by decode_host and by
    decode, and nothing runs (the logits buffer keeps the last step's values)."""
    from intel_extension_for_transformers_b200._capi import QbitsError
    r = run_kv_end(path)
    B = len(r["next"])
    for j, (got, ref) in enumerate(zip(r["got"], r["ref"])):
        _check_rows(got, ref, KV_END[path][-1], "step %d" % j)
    eng, nxt, max_seq = r["eng"], r["next"], r["max_seq"]
    last = eng.last_logits(B)
    with pytest.raises(QbitsError, match="KV cache"):
        eng.decode_host(nxt.tolist(), max_seq)
    with pytest.raises(QbitsError, match="KV cache"):
        eng.decode(torch.from_numpy(nxt.astype(np.int32)), max_seq)
    assert torch.equal(eng.last_logits(B), last)
