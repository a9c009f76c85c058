"""GPU: the native decode runtime against a CPU restatement of the decoder built from oracle pieces
(oracle.rmsnorm / apply_rope / attention / dequantize; HF Llama semantics, modeling_llama.py:72-96,208-301)."""
import numpy as np
import pytest
import torch

from oracle import qbits_oracle as O

pytestmark = pytest.mark.gpu


def _mk_lin(rng, K, N, group, asym):
    q = rng.integers(-8, 8, size=(K, N)).astype(np.int8)
    s = ((0.5 + rng.random((K // group, N), dtype=np.float32)) * 0.02).astype(np.float32)
    z = rng.integers(-3, 4, size=(K // group, N)).astype(np.int8) if asym else None
    return dict(q=q, scale=s, zp=z)


def _ref_forward(geom, layers, embed, fnorm, lm_head, tokens, group, stype, f64=False, last=None, wround=0):
    """tokens [B, T] -> logits [B, T, V] in numpy with bf16 rounding at the points where the reference's bf16 modules round
    (module outputs, residual adds, RMSNorm, RoPE, attention output, SiLU, the gate * up product).  Matrix products
    accumulate in fp32 (BLAS) or, with f64=True, in fp64: the difference between the two is the test's own noise floor
    (a bf16 rounding that flips on one side moves a logit by ~2^-9 of an activation; tools/parity_report.py records it).
    last=n: logits [B, n, V] of the last n positions only; the last layer's attention queries, MLP and the lm_head then run
    on those n rows (earlier layers still need every position for the keys and values).
    wround=n: positions 0..n-1 multiply by the dequantised weights rounded to bf16, as the tensor-core GEMM that runs a
    prefill of 64 rows or more does (gemm_tc.cu); later positions (decode steps: exact integer math, fp32 scaling) do not."""
    r = O.bf16_round
    if f64:
        class _M:  # matmul in fp64, result back in fp32
            def __init__(self, a): self.a = a
            def __matmul__(self, b): return (self.a.astype(np.float64) @ np.asarray(b, np.float64)).astype(np.float32)
        wrap = _M
    else:
        wrap = lambda a: a
    B, T = tokens.shape
    D, Hq, Hkv = geom.head_dim, geom.n_heads, geom.n_kv_heads
    h = embed[tokens]  # [B,T,H]
    cos, sin = O.rope_cos_sin(np.arange(T), D, geom.rope_theta)
    cos, sin = r(cos), r(sin)
    deq = lambda l: O.dequantize(l["q"], l["scale"], l["zp"], group, "int4_clip", stype)

    def mm(x, l):   # x [B, rows, K]: the last `rows` positions
        w = deq(l)
        n = min(max(wround - (T - x.shape[1]), 0), x.shape[1])
        if n == 0:
            return wrap(x) @ w
        return np.concatenate([wrap(x[:, :n]) @ r(w), wrap(x[:, n:]) @ w], axis=1)

    for li, L in enumerate(layers):
        x = r(r(O.rmsnorm(h, np.ones_like(L["an"]), geom.rms_eps)) * L["an"])
        q = r(mm(x, L["q"])).reshape(B, T, Hq, D).transpose(0, 2, 1, 3)
        k = r(mm(x, L["k"])).reshape(B, T, Hkv, D).transpose(0, 2, 1, 3)
        v = r(mm(x, L["v"])).reshape(B, T, Hkv, D).transpose(0, 2, 1, 3)
        rope = lambda t: r(r(t * cos[None, None]) + r(O.rotate_half(t) * sin[None, None]))
        q, k = rope(q), rope(k)
        if last is not None and li == len(layers) - 1:   # queries at positions T - last .. T - 1 (O.attention's default offset)
            q, h = q[:, :, T - last:], h[:, T - last:]
        a = r(O.attention(q, k, v, causal=True)).transpose(0, 2, 1, 3).reshape(B, q.shape[2], Hq * D)
        h = r(h + r(mm(a, L["o"])))          # the module output is bf16 before `residual + hidden` (HF LlamaDecoderLayer)
        x = r(r(O.rmsnorm(h, np.ones_like(L["mn"]), geom.rms_eps)) * L["mn"])
        g, u = r(mm(x, L["gate"])), r(mm(x, L["up"]))
        m = r(r(O.silu(g)) * u)                 # act_fn(gate_proj(x)) * up_proj(x): every op rounds to bf16 (HF LlamaMLP)
        h = r(h + r(mm(m, L["down"])))
    x = r(r(O.rmsnorm(h, np.ones_like(fnorm), geom.rms_eps)) * fnorm)
    return wrap(x) @ lm_head.T


@pytest.mark.parametrize("asym,stype", [(False, "bf16"), (True, "fp32")])
def test_engine_prefill_and_decode_match_oracle(asym, stype):
    from intel_extension_for_transformers_b200.runtime.engine import LlamaEngine, LlamaGeometry
    geom = LlamaGeometry(hidden=256, inter=512, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=128, vocab=1000)
    group = 128
    rng = np.random.default_rng(0)
    H, I, D = geom.hidden, geom.inter, geom.head_dim
    layers = []
    eng = LlamaEngine(geom, max_seq=64, max_batch=2)
    dev = "cuda"
    t = lambda d: {k: (torch.from_numpy(v).to(dev) if v is not None else None) for k, v in d.items()}
    for l in range(geom.n_layers):
        L = dict(q=_mk_lin(rng, H, geom.n_heads * D, group, asym), k=_mk_lin(rng, H, geom.n_kv_heads * D, group, asym),
                 v=_mk_lin(rng, H, geom.n_kv_heads * D, group, asym), o=_mk_lin(rng, geom.n_heads * D, H, group, asym),
                 gate=_mk_lin(rng, H, I, group, asym), up=_mk_lin(rng, H, I, group, asym), down=_mk_lin(rng, I, H, group, asym),
                 an=O.bf16_round(1.0 + 0.1 * rng.standard_normal(H).astype(np.float32)),
                 mn=O.bf16_round(1.0 + 0.1 * rng.standard_normal(H).astype(np.float32)))
        layers.append(L)
        blobs = LlamaEngine.pack_layer(t(L["q"]), t(L["k"]), t(L["v"]), t(L["o"]), t(L["gate"]), t(L["up"]), t(L["down"]),
                                       "int4_clip", stype, "bf16", asym, group)
        eng.set_layer(l, *blobs, torch.from_numpy(L["an"]).to(dev), torch.from_numpy(L["mn"]).to(dev))
    embed = O.bf16_round(rng.standard_normal((geom.vocab, H)).astype(np.float32) * 0.5)
    lm_head = O.bf16_round(rng.standard_normal((geom.vocab, H)).astype(np.float32) * 0.05)
    fnorm = O.bf16_round(1.0 + 0.1 * rng.standard_normal(H).astype(np.float32))
    eng.set_globals(torch.from_numpy(embed).to(dev), torch.from_numpy(fnorm).to(dev), torch.from_numpy(lm_head).to(dev))

    B, T, NEW = 2, 9, 6
    tokens = rng.integers(0, geom.vocab, size=(B, T))
    eng.reset()
    logits = eng.prefill(torch.from_numpy(tokens)).cpu().numpy()
    ref = _ref_forward(geom, layers, embed, fnorm, lm_head, tokens, group, stype)
    err = np.linalg.norm(logits - ref[:, -1]) / np.linalg.norm(ref[:, -1])
    assert err < 2e-2, err  # bf16 activations between ops on both sides; kernels are exact to ~1e-5 (test_gpu_qbits)
    assert (logits.argmax(-1) == ref[:, -1].argmax(-1)).all()

    # a longer prompt (2 x 40 = 80 rows >= 64) takes the tcgen05 GEMM with the fused residual / SiLU*mul epilogues
    tokens_l = rng.integers(0, geom.vocab, size=(B, 40))
    eng.reset()
    logits_l = eng.prefill(torch.from_numpy(tokens_l)).cpu().numpy()
    ref_l = _ref_forward(geom, layers, embed, fnorm, lm_head, tokens_l, group, stype)
    err_l = np.linalg.norm(logits_l - ref_l[:, -1]) / np.linalg.norm(ref_l[:, -1])
    assert err_l < 3e-2, err_l   # + one bf16 rounding of every dequantised weight (gemm_tc.cu)
    eng.reset()
    eng.prefill(torch.from_numpy(tokens))

    # decode: feed tokens one at a time (teacher forcing with the oracle's greedy choices) through graph replay
    seq = tokens.copy()
    nxt = ref[:, -1].argmax(-1)
    for step in range(NEW):
        seq = np.concatenate([seq, nxt[:, None]], axis=1)
        ref_full = _ref_forward(geom, layers, embed, fnorm, lm_head, seq, group, stype)
        pos = seq.shape[1] - 1
        out, lg = eng.decode(torch.from_numpy(nxt.astype(np.int32)), pos, want_logits=True)
        lg = lg.cpu().numpy()
        err = np.linalg.norm(lg - ref_full[:, -1]) / np.linalg.norm(ref_full[:, -1])
        assert err < 2e-2, (step, err)
        nxt = ref_full[:, -1].argmax(-1)
        top2 = np.sort(ref_full[:, -1], axis=-1)[:, -2:]
        clear = (top2[:, 1] - top2[:, 0]) > 0.05 * np.abs(top2[:, 1])
        assert (out.cpu().numpy()[clear] == nxt[clear]).all()

    # host-buffer path (CUDA graph) reproduces the eager device path bit for bit
    eng.reset()
    eng.prefill(torch.from_numpy(tokens))
    first = ref[:, -1].argmax(-1).tolist()
    a = eng.decode_host(first, T)
    eng.reset()
    eng.prefill(torch.from_numpy(tokens))
    b = eng.decode(torch.tensor(first, dtype=torch.int32), T).cpu().tolist()
    assert a == b
    a2 = eng.decode_host(a, T + 1)
    b2 = eng.decode(torch.tensor(b, dtype=torch.int32), T + 1).cpu().tolist()
    assert a2 == b2


def test_attention_op_matches_oracle():
    """qb_attention (prefill flash kernel) vs the oracle, GQA 4:1, ragged lengths, causal with a KV prefix."""
    import ctypes as C
    from intel_extension_for_transformers_b200._capi import check, lib, stream_ptr
    torch.manual_seed(0)
    for (B, Hq, Hkv, Tq, Tk) in [(2, 4, 1, 70, 70), (1, 8, 8, 33, 97), (1, 4, 2, 1, 50), (2, 2, 1, 128, 128)]:
        D = 128
        q = torch.randn(B, Hq, Tq, D).to(torch.bfloat16)
        k = torch.randn(B, Hkv, Tk, D).to(torch.bfloat16)
        v = torch.randn(B, Hkv, Tk, D).to(torch.bfloat16)
        out = torch.empty(B, Hq, Tq, D, dtype=torch.bfloat16, device="cuda")
        qd, kd, vd = q.cuda(), k.cuda(), v.cuda()
        check(lib().qb_attention(qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), out.data_ptr(), B, Hq, Hkv, Tq, Tk, Tk, D,
                                 1.0 / np.sqrt(D), 1, 1.0, stream_ptr()))
        ref = O.attention(q.float().numpy(), k.float().numpy(), v.float().numpy(), causal=True)
        got = out.float().cpu().numpy()
        assert np.abs(got - ref).max() < 2e-2, (B, Hq, Hkv, Tq, Tk, np.abs(got - ref).max())
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 6e-3


@pytest.mark.timeout(300)
def test_attention_tcgen05_kernel_matches_oracle():
    """The tcgen05 / TMEM prefill attention (attn_tc.cu, taken for >= 64 queries): ragged query blocks, a KV prefix that is
    not a multiple of the key tile, GQA, several key tiles (running max / lazy rescale of O in tensor memory)."""
    from intel_extension_for_transformers_b200._capi import check, lib, stream_ptr
    torch.manual_seed(1)
    for (B, Hq, Hkv, Tq, Tk, scale) in [(1, 4, 2, 300, 300, 1.0), (1, 2, 1, 200, 333, 1.0), (2, 8, 2, 512, 512, 1.0), (1, 2, 2, 64, 1000, 1.0),
                                        (1, 2, 1, 384, 384, 4.0)]:
        D = 128
        q = (torch.randn(B, Hq, Tq, D) * scale).to(torch.bfloat16)   # scale 4: peaked softmax, the running max moves a lot
        k = torch.randn(B, Hkv, Tk, D).to(torch.bfloat16)
        v = torch.randn(B, Hkv, Tk, D).to(torch.bfloat16)
        out = torch.full((B, Hq, Tq, D), float("nan"), dtype=torch.bfloat16, device="cuda")
        qd, kd, vd = q.cuda(), k.cuda(), v.cuda()
        check(lib().qb_attention(qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), out.data_ptr(), B, Hq, Hkv, Tq, Tk, Tk, D,
                                 1.0 / np.sqrt(D), 1, 1.0, stream_ptr()))
        torch.cuda.synchronize()
        ref = O.attention(q.float().numpy(), k.float().numpy(), v.float().numpy(), causal=True)
        got = out.float().cpu().numpy()
        assert np.isfinite(got).all(), (B, Hq, Hkv, Tq, Tk)
        assert np.abs(got - ref).max() < 3e-2, (B, Hq, Hkv, Tq, Tk, np.abs(got - ref).max())
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 6e-3, (B, Hq, Hkv, Tq, Tk)
