"""CPU-only: host logic, config surface, C-ABI exports, oracle C port, bench accounting.  No GPU compute."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import qbits_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from intel_extension_for_transformers_b200 import _capi
    lib = _capi.lib()
    hdr = open(os.path.join(ROOT, "include", "qbits_b200.h")).read()
    declared = set(re.findall(r"\b(qb_[a-z0-9_]+)\s*\(", hdr)) - {"qb_engine", "qb_llama_config", "qb_llama_layer"}
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/qbits_b200.h but not exported"
    assert set(_capi.EXPORTS) <= declared
    assert lib.qb_version() >= 100


def test_no_cpu_fallback():
    import intel_extension_for_transformers_b200.qbits as qbits
    q = torch.zeros(256, 32, dtype=torch.int8)
    with pytest.raises(RuntimeError, match="Qbits"):
        qbits.repack_quantized_weight(q, torch.ones(2, 32), torch.empty(0), torch.empty(0), "int4_clip", "fp32", "fp32", False, 128)
    with pytest.raises(RuntimeError, match="Qbits"):
        qbits.woq_linear(torch.zeros(1, 256), torch.zeros(8, dtype=torch.int8), torch.empty(0), torch.zeros(1, 32), "fp32",
                         "int4_clip", "fp32", False)
    if not torch.cuda.is_available():
        from intel_extension_for_transformers_b200 import _capi
        assert _capi.lib().qb_device_ok() == 0
        assert not qbits.check_isa_supported("SM100")
    assert not qbits.check_isa_supported("AMX")


def test_packed_size_is_host_computable_and_layout_consistent():
    import intel_extension_for_transformers_b200.qbits as qbits
    n, k = 4096, 11008
    sz = qbits.get_packed_weight_size(k, n, "int4_clip", "bf16", "bf16", False, 128, False)
    kp = (k + 255) // 256 * 256
    assert sz >= n * kp // 2 + n * (kp // 128) * 2 + 256
    assert sz < 1.02 * (n * kp // 2 + n * (kp // 128) * 2) + 4096
    with pytest.raises(RuntimeError, match="unsupported weight_type"):
        qbits.get_packed_weight_size(k, n, "fp8_e4m3", "fp32", "fp32", False, 128, False)
    with pytest.raises(RuntimeError, match="unsupported blocksize"):
        qbits.get_packed_weight_size(k, n, "int4_clip", "fp32", "fp32", False, 48, False)
    with pytest.raises(RuntimeError, match="float-weight unsupports asym"):
        qbits.get_packed_weight_size(k, n, "nf4", "fp32", "fp32", True, 128, False)


def test_config_defaults_match_reference(golden_dir):
    """RtnConfig / GPTQConfig against the reference file's own behaviour (tests/golden/config_defaults.json) and the
    assertions of tests/CI/test_weight_only.py:93-115."""
    from intel_extension_for_transformers_b200.transformers.utils.config import GPTQConfig, RtnConfig, WeightOnlyQuantConfig
    d = json.load(open(os.path.join(golden_dir, "config_defaults.json")))
    for tag, v in d.items():
        if tag.startswith("_"):
            continue
        cls = {"RtnConfig": RtnConfig, "GPTQConfig": GPTQConfig}[v["cls"]]
        c = cls(**v["kwargs"])
        assert json.loads(json.dumps(c.to_diff_dict(), default=str)) == v["to_diff_dict"], tag
        c.post_init_cpu()
        for k, x in v["post_init_cpu"].items():
            got = getattr(c, k) if k != "quant_method" else c.quant_method.value
            assert got == x, (tag, k, got, x)
    for tag, kw in {"default": {}, "int4_g32": dict(bits=4, weight_dtype="int4", group_size=32)}.items():
        c = RtnConfig(**kw)
        c.post_init_runtime()
        for k, x in d["_post_init_runtime"][tag].items():
            got = getattr(c, k) if k != "quant_method" else c.quant_method.value
            assert got == x, (tag, k, got, x)
    assert WeightOnlyQuantConfig is RtnConfig
    c = RtnConfig(bits=4, weight_dtype="int4", group_size=32)
    assert c.to_diff_dict() == {"weight_dtype": "int4"}          # test_weight_only.py:96-97
    c = RtnConfig(bits=4, compute_dtype="bf16", scale_dtype="bf16", group_size=128)
    c.post_init_cuda()
    assert (c.weight_dtype, c.compute_dtype, c.scale_dtype, c.use_neural_speed) == ("int4_clip", "bf16", "bf16", False)
    with pytest.raises(ValueError):
        RtnConfig(bits=4, weight_dtype="nf4", sym=False).post_init_cuda()


def test_torch_unpack_weight_matches_reference(golden_dir):
    from types import SimpleNamespace
    from intel_extension_for_transformers_b200.transformers.llm.quantization.utils import pack_weight, unpack_weight
    z = np.load(os.path.join(golden_dir, "unpack_weight.npz"))
    for tag in ("b4_sym", "b4_asym", "b8_sym", "b8_asym"):
        bits, sym, K, N, group = z[f"{tag}_meta"]
        w, s, zeros = unpack_weight(torch.from_numpy(z[f"{tag}_qweight"]), torch.from_numpy(z[f"{tag}_scales"]),
                                    torch.from_numpy(z[f"{tag}_qzeros"]), SimpleNamespace(bits=int(bits), sym=bool(sym)))
        w = w.view(-1, w.shape[-1])
        assert np.array_equal(w.numpy().astype(np.int64), z[f"{tag}_w"].astype(np.int64)), tag
        assert np.array_equal(zeros.numpy().astype(np.int64), z[f"{tag}_z"].astype(np.int64)), tag
    # pack_weight (save_low_bit) inverts it
    g = torch.Generator().manual_seed(0)
    q = torch.randint(0, 16, (64, 16), generator=g)
    zu = torch.randint(1, 17, (2, 16), generator=g)
    qw, qz = pack_weight(q, zu, 4)
    w, _, zz = unpack_weight(qw, torch.ones(2, 16), qz, SimpleNamespace(bits=4, sym=False))
    assert torch.equal(w.view(-1, 16).long(), q) and torch.equal(zz.long(), zu)


def test_c_port_matches_numpy_oracle():
    from oracle import cpu_port
    rng = np.random.default_rng(0)
    for sym in (True, False):
        K, N, g = 512, 384, 128
        d = O.synth_gptq_linear(K, N, g, sym=sym, seed=3)
        w, s, z = O.unpack_weight(d["qweight"], d["scales"].astype(np.float32), d["qzeros"], 4, sym)
        q, zs = O.recenter_int4(w, z)
        W = O.dequantize(q, s, None if sym else zs, g)
        x = rng.standard_normal((2, K)).astype(np.float32)
        ref = O.woq_linear(x, W)
        got = cpu_port.woq_linear_int4(x, d["qweight"], d["scales"].astype(np.float32), None if sym else z, g)
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-5
    assert cpu_port.threads() >= 1


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_bench_accounting_matches_survey():
    b = _load_bench()
    assert b.algorithmic_bytes_per_token(0) == 3_238_002_688 + 101_187_584 + 262_144_000   # SURVEY.md section 8d
    assert b.algorithmic_bytes_per_token(10) - b.algorithmic_bytes_per_token(0) == 524_288 * 10


def test_bench_dump_outputs_are_float32_or_float64(tmp_path):
    b = _load_bench()
    logits = torch.randn(2, 5).to(torch.bfloat16)
    b.write_outputs(str(tmp_path / "out"), {"logits": logits, "token": torch.tensor([31999], dtype=torch.float64)})
    assert sorted(os.listdir(tmp_path / "out")) == ["logits.npy", "token.npy"]
    got = np.load(tmp_path / "out" / "logits.npy")
    assert got.dtype == np.float32 and np.array_equal(got, logits.float().numpy())
    tok = np.load(tmp_path / "out" / "token.npy")
    assert tok.dtype == np.float64 and tok.tolist() == [31999.0]


def test_interleave_gate_up_layout():
    from intel_extension_for_transformers_b200.runtime.engine import interleave_gate_up
    g = torch.arange(32).view(1, 32)
    u = 100 + torch.arange(32).view(1, 32)
    m = interleave_gate_up(g, u)
    assert m.shape == (1, 64)
    assert m[0, :8].tolist() == list(range(8)) and m[0, 8:16].tolist() == list(range(100, 108))
    assert m[0, 16:24].tolist() == list(range(8, 16))


def test_gptq_checkpoint_directory_is_recognised_and_split(tmp_path):
    """Host side of the GPTQ directory loader (modeling/gptq_checkpoint.py): detection from config.json and the split of a
    safetensors shard set into the floating-point state dict and the per-linear optimum-layout tensors."""
    import json
    import torch
    from safetensors.torch import save_file
    from oracle import qbits_oracle as O
    from intel_extension_for_transformers_b200.transformers.modeling import gptq_checkpoint as G
    assert not G.is_gptq_checkpoint(str(tmp_path))                      # no config.json
    json.dump({"model_type": "llama"}, open(tmp_path / "config.json", "w"))
    assert not G.is_gptq_checkpoint(str(tmp_path))                      # not quantised
    json.dump({"model_type": "llama", "quantization_config": {"quant_method": "GPTQ", "bits": 4, "group_size": 128}},
              open(tmp_path / "config.json", "w"))
    assert G.is_gptq_checkpoint(str(tmp_path))
    d = O.synth_gptq_linear(256, 128, 128, sym=False, seed=3)
    shard1 = {"model.layers.0.mlp.down_proj.qweight": torch.from_numpy(d["qweight"]),
              "model.layers.0.mlp.down_proj.qzeros": torch.from_numpy(d["qzeros"]),
              "model.embed_tokens.weight": torch.ones(4, 8, dtype=torch.float16)}
    shard2 = {"model.layers.0.mlp.down_proj.scales": torch.from_numpy(d["scales"]),
              "model.layers.0.mlp.down_proj.g_idx": torch.from_numpy(d["g_idx"]),
              "model.norm.weight": torch.ones(8, dtype=torch.float16)}
    save_file(shard1, str(tmp_path / "model-00001-of-00002.safetensors"))
    save_file(shard2, str(tmp_path / "model-00002-of-00002.safetensors"))
    sd, packed = G.read_tensors(str(tmp_path))
    assert sorted(sd) == ["model.embed_tokens.weight", "model.norm.weight"] and all(v.dtype == torch.bfloat16 for v in sd.values())
    assert list(packed) == ["model.layers.0.mlp.down_proj"]
    t = packed["model.layers.0.mlp.down_proj"]
    assert sorted(t) == ["g_idx", "qweight", "qzeros", "scales"] and t["qweight"].dtype == torch.int32
    # the packed tensors round-trip through the oracle's unpack exactly
    w, s, z = O.unpack_weight(t["qweight"].numpy(), t["scales"].float().numpy(), t["qzeros"].numpy(), 4, False)
    assert (w == d["q_u"]).all() and (z == d["zp_nibble"].astype(z.dtype) + 1).all()


def test_ctypes_signatures_have_the_arity_the_header_declares():
    """ABI drift guard: every entry of _capi._SIGS must list as many arguments as the prototype in include/qbits_b200.h."""
    from intel_extension_for_transformers_b200 import _capi
    hdr = open(os.path.join(ROOT, "include", "qbits_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)          # drop comments (some sit inside parameter lists)
    protos = {}
    for m in re.finditer(r"\b(qb_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    checked = 0
    for name, (_res, args) in _capi._SIGS.items():
        assert name in protos, f"{name} bound in _capi.py but not declared in the header"
        assert len(args) == protos[name], f"{name}: ctypes lists {len(args)} arguments, the header declares {protos[name]}"
        checked += 1
    assert checked >= 25


def test_generate_routing_and_engine_gating():
    """Host logic behind model.generate(): the native greedy loop only takes requests it reproduces exactly (EOS / pad
    handled in the loop, greedy_search.py:163-167), everything else goes to HF generate; checkpoints whose attention /
    RoPE / MLP differ from plain Llama-2 never get the native runtime."""
    from types import SimpleNamespace as NS
    from intel_extension_for_transformers_b200.transformers.modeling import modeling_auto as ma
    eng = NS(max_batch=2, max_seq=64)
    ids = torch.ones(1, 5, dtype=torch.long)
    plan = ma._native_generate_plan(None, dict(max_new_tokens=7), ids, eng)
    assert plan == (7, [], None)
    gc = NS(max_new_tokens=None, max_length=20, eos_token_id=[2, 9], pad_token_id=None, num_beams=1, do_sample=False,
            repetition_penalty=1.0, temperature=0.6, top_p=0.9)
    assert ma._native_generate_plan(gc, {}, ids, eng) == (15, [2, 9], 2)   # max_length - prompt, pad defaults to the first EOS
    assert ma._native_generate_plan(gc, dict(eos_token_id=3, pad_token_id=0, max_new_tokens=4), ids, eng) == (4, [3], 0)
    # anything the loop does not implement -> HF generate
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, repetition_penalty=1.3), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, stopping_criteria=[object()]), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, logits_processor=[object()]), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, min_length=3), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, do_sample=True), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, num_beams=4), ids, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, some_future_flag=1), ids, eng) is None
    assert ma._native_generate_plan(NS(repetition_penalty=1.2), dict(max_new_tokens=4), ids, eng) is None
    # the installed transformers' default GenerationConfig (every field None in 5.x) must stay on the native loop
    import transformers
    assert ma._native_generate_plan(transformers.GenerationConfig(), dict(max_new_tokens=5), ids, eng) == (5, [], None)
    assert ma._native_generate_plan(transformers.GenerationConfig(num_beams=4), dict(max_new_tokens=5), ids, eng) is None
    two = torch.ones(2, 5, dtype=torch.long)
    left_padded = torch.tensor([[0, 0, 1, 1, 1], [1, 1, 1, 1, 1]])
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, attention_mask=left_padded), two, eng) is None
    assert ma._native_generate_plan(None, dict(max_new_tokens=4, attention_mask=torch.ones(2, 5)), two, eng) == (4, [], None)
    assert ma._native_generate_plan(None, dict(max_new_tokens=60), ids, eng) is None           # beyond max_seq
    assert ma._native_generate_plan(None, dict(max_new_tokens=4), torch.ones(3, 5, dtype=torch.long), eng) is None
    # engine gating
    base = dict(rope_scaling=None, sliding_window=None, attention_bias=False, mlp_bias=False, hidden_act="silu")
    assert ma._engine_unsupported(NS(**base), 4096) is None
    assert "rope" in ma._engine_unsupported(NS(**{**base, "rope_scaling": {"rope_type": "llama3", "factor": 8.0}}), 4096)
    assert "rope" in ma._engine_unsupported(NS(**{**base, "rope_scaling": {"type": "linear", "factor": 2.0}}), 4096)
    assert "rope" in ma._engine_unsupported(NS(**{**base, "rope_parameters": {"rope_type": "yarn", "rope_theta": 1e4}}), 4096)
    assert ma._engine_unsupported(NS(**{**base, "rope_parameters": {"rope_type": "default", "rope_theta": 1e4}}), 4096) is None
    assert "sliding_window" in ma._engine_unsupported(NS(**{**base, "sliding_window": 1024}), 4096)
    assert ma._engine_unsupported(NS(**{**base, "sliding_window": 4096}), 4096) is None
    assert ma._engine_unsupported(NS(**{**base, "attention_bias": True}), 4096) == "attention_bias"
    assert ma._engine_unsupported(NS(**{**base, "mlp_bias": True}), 4096) == "mlp_bias"
    assert "hidden_act" in ma._engine_unsupported(NS(**{**base, "hidden_act": "gelu"}), 4096)
