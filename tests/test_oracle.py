"""CPU suite: pins the oracle restatement against golden vectors committed from the unmodified reference; checks host logic
and that libdsk.so exports the declared C-ABI."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

import oracle as O
from conftest import rel_l2

P = O.Ops("port")


@pytest.fixture(scope="module")
def kat(golden_dir):
    return json.load(open(os.path.join(golden_dir, "kat.json")))


@pytest.fixture(scope="module")
def ops(golden_dir):
    return np.load(os.path.join(golden_dir, "ops.npz"))


# ---- known answers carried by the reference's own tests (src/test.cpp:128-186) --------------------
def test_testcpp_matmul_kat(kat):
    x = np.array(kat["testcpp_x"], np.float32)
    w = np.array(kat["testcpp_w"], np.float32)
    exp = np.array(kat["testcpp_expect_f32_f16"])
    assert np.allclose(P.matmul(x, w, "fp32", 2, 16), exp, atol=1e-4)                       # test.cpp:150-153
    assert np.allclose(P.matmul(x, w.astype(np.float16), "fp16", 2, 16), exp, atol=1e-3)    # test.cpp:156-160
    w8 = (w.astype(np.float16).view(np.uint16) >> 8).astype(np.uint8)
    got = P.matmul(x, w8, "f8e5m2", 2, 16)
    assert np.allclose(got, exp, atol=3.78e-1)                                               # test.cpp:163-166
    assert np.allclose(got, kat["testcpp_ref_f8"], rtol=1e-6)
    L = O.port_lib()
    for v in (1.0, -1.5, 0.109375):                                                          # test.cpp:129-131
        h = L.ork_float_to_half(v)
        assert L.ork_f8e5m2_to_float(h >> 8) == v


def test_survey_kats(kat):
    assert np.allclose(P.rmsnorm(kat["rmsnorm_in"], kat["rmsnorm_w"], kat["rmsnorm_eps"]), kat["rmsnorm_out"], rtol=1e-6)
    assert np.allclose(P.rope(kat["rope_in"], 8, kat["rope_pos"], kat["rope_theta"], False), kat["rope_v2_out"], rtol=1e-5, atol=1e-6)
    assert np.allclose(P.rope(kat["rope_in"], 8, kat["rope_pos"], kat["rope_theta"], True), kat["rope_v3_out"], rtol=1e-5, atol=1e-6)
    i, w, _ = P.moe_gate(kat["gate_logits"], None, 3, False, 2.0, False, 0, 1, 1)
    assert i.tolist() == kat["gate_softmax_greedy"]["idx"] and np.allclose(w, kat["gate_softmax_greedy"]["w"], rtol=1e-6)
    i, w, _ = P.moe_gate(kat["gate_logits"], None, 3, True, 1.0, True, 1, 4, 1)
    assert i.tolist() == kat["gate_sigmoid_group"]["idx"] and np.allclose(w, kat["gate_sigmoid_group"]["w"], rtol=1e-6)
    assert abs(P.silu(1.5) - kat["silu_1p5"]) < 1e-6


# ---- golden op vectors (generated from the unmodified reference, tests/golden/make_golden.py) -----
def test_q8k_golden_bit_exact(ops):
    got = P.quantize_q8k(ops["q8k_x"]).reshape(-1, 292)
    exp = ops["q8k_blocks"].reshape(-1, 292)
    for b in range(exp.shape[0]):
        nz = ops["q8k_x"][b * 256:(b + 1) * 256].any()
        # the reference leaves bsums of an all-zero block uninitialised (src/quant.cpp:630-635)
        assert np.array_equal(got[b, :260], exp[b, :260]) and (not nz or np.array_equal(got[b], exp[b]))


@pytest.mark.parametrize("quant", ["q2_k", "q3_k"])
def test_kquant_gemv_and_dequant_golden(ops, quant):
    w, x = ops[f"{quant}_w"], ops[f"{quant}_x"]
    got = P.matmul(x, w, quant, w.shape[0], x.size)
    assert rel_l2(got, ops[f"{quant}_out"]) < 2e-6
    assert np.array_equal(P.dequantize(w[0], quant, x.size), ops[f"{quant}_deq_row0"]) or \
        np.allclose(P.dequantize(w[0], quant, x.size), ops[f"{quant}_deq_row0"], rtol=1e-6, atol=1e-8)


def test_dense_gemv_golden(ops):
    assert rel_l2(P.matmul(ops["f8_x"], ops["f8_w"], "f8e5m2", 200, 384, ops["f8_scale"]), ops["f8_out"]) < 1e-6
    assert rel_l2(P.matmul(ops["f16_x"], ops["f16_w"], "fp16", 40, 256), ops["f16_out"]) < 1e-6
    assert rel_l2(P.matmul(ops["f16_x"], ops["f32_w"], "fp32", 40, 256), ops["f32_out"]) < 1e-5


@pytest.mark.parametrize("name,cfg", [("v2lite", (6, 0, 1.0, 0, 0, 1, 1)), ("v2", (6, 0, 16.0, 0, 1, 8, 3)),
                                      ("v3", (8, 1, 2.5, 1, 1, 8, 4))])
def test_gate_golden(ops, name, cfg):
    K, norm, scale, sig, method, ng, tg = cfg
    bias = ops[f"gate_{name}_bias"] if f"gate_{name}_bias" in ops else None
    idx, w, sc = P.moe_gate(ops[f"gate_{name}_logits"], bias, K, norm, scale, sig, method, ng, tg)
    assert idx.tolist() == ops[f"gate_{name}_idx"].tolist()
    assert np.allclose(w, ops[f"gate_{name}_w"], rtol=2e-6)
    assert np.allclose(sc, ops[f"gate_{name}_scores"], rtol=2e-6, atol=1e-9)


def test_rope_attn_golden(ops):
    assert np.allclose(P.rope(ops["rope_x"], 64, 1234, 1e4, False), ops["rope_v2_p1234"], rtol=1e-4, atol=2e-5)
    assert np.allclose(P.rope(ops["rope_x"], 64, 1234, 1e4, True), ops["rope_v3_p1234"], rtol=1e-4, atol=2e-5)
    for v3, key in ((False, "rope16_v2_p1"), (True, "rope16_v3_p1")):
        got = P.rope_f16(ops["rope16_x"], 64, 1, 1e4, v3).view(np.float16).astype(np.float32)
        exp = ops[key].view(np.float16).astype(np.float32)
        assert np.max(np.abs(got - exp)) <= 2e-3  # at most one fp16 ulp
    nh, hd, vh, T = 3, 48, 32, 37
    got = np.concatenate([P.attn(ops["attn_q"][h * hd:(h + 1) * hd], ops["attn_k"][h * hd:], ops["attn_v"][h * vh:], hd, vh, nh, T)
                          for h in range(nh)])
    assert rel_l2(got, ops["attn_out"]) < 1e-6


def test_e2e_golden_port(golden_dir, tmp_path):
    """End-to-end teacher-forced logits of the port vs the reference's (committed), on checkpoints that can be
    minted without the reference (random valid Q2_K blocks / torch f8 cast)."""
    import mint
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    for preset, quant, tol in (("tiny_v3", "q2_k", 5e-2), ("tiny_v2lite", "f8e5m2", 1e-3)):
        d = str(tmp_path / f"{preset}_{quant}")
        mint.mint(d, preset, quant, fast=True, seed=77)
        s = O.PortSession(d)
        for p, t in enumerate(g[f"{preset}_{quant}_tokens"]):
            s.forward(int(t), p)
            exp = g[f"{preset}_{quant}_logits"][p]
            assert rel_l2(s.buffer("logits"), exp) < tol, (preset, quant, p)


def test_e2e_mla_golden_port(golden_dir, tmp_path):
    """True-MLA blocks (BlockMLA::_attention_impl src/infer.cpp:1051-1141, attn_mla 766-804) of the port vs the reference's
    committed outputs (tests/golden/e2e_mla.npz, make_golden_mla.py): logits, the latent / rope cache rows of layer 0 and the
    last token's q_c / value up-projection.  The fp32 case runs past original_max_position (sink re-rotation)."""
    import mint
    from golden.make_golden_mla import CASES
    g = np.load(os.path.join(golden_dir, "e2e_mla.npz"))
    tols = {"q2_k": 5e-2, "f8e5m2": 1e-3, "fp32": 1e-3}
    for preset, quant, kw in CASES:
        key = f"{preset}_{quant}"
        d = str(tmp_path / key)
        mint.mint(d, preset, quant, fast=True, seed=78, use_mla=True, **kw)
        s = O.PortSession(d)
        assert s.c["use_mla"] == 1
        for p, t in enumerate(g[key + "_tokens"]):
            s.forward(int(t), p)
            assert rel_l2(s.buffer("logits"), g[key + "_logits"][p]) < tols[quant], (key, p)
        n, c = len(g[key + "_tokens"]), s.c
        nh, vh = c["n_heads"], c["v_head_dim"]
        if quant != "q2_k":   # (a Q8_K rounding flip upstream moves these by more than a cache ulp)
            assert rel_l2(s.buffer("q_c"), g[key + "_q_c_last"]) < 1e-3
            assert rel_l2(s.buffer("kv_b")[:nh * vh], g[key + "_kv_b_last"][:nh * vh]) < 1e-3
            if "original_max_position" not in kw:   # (sink rows are re-rounded every step past the limit)
                for which, name, w in ((0, "_latent_cache_l0", c["kv_lora_rank"]), (1, "_rope_cache_l0", c["qk_rope_head_dim"])):
                    a = s.kv_cache(0, which)[:n * w].view(np.float16).astype(np.float32)
                    b = g[key + name].view(np.float16).astype(np.float32)
                    assert np.allclose(a, b, rtol=2e-3, atol=1e-4), (key, name)


# ---- port vs the unmodified reference (its outputs committed: tests/golden/make_golden_port.py) ----------
@pytest.fixture(scope="module")
def pvr(golden_dir):
    return np.load(os.path.join(golden_dir, "port_vs_ref.npz"))


def _logits(s, pvr):
    return s.buffer("logits")[pvr["logit_idx"]]


def test_q8k_bit_exact_vs_ref(pvr):
    from golden.make_golden_port import digest, q8k_inputs
    for t, x in enumerate(q8k_inputs()):
        assert np.array_equal(digest(P.quantize_q8k(x)), pvr["q8k_sha256"][t]), t


@pytest.mark.parametrize("quant,tol", [("fp32", 1e-5), ("fp16", 1e-6), ("f8e5m2", 1e-6), ("q2_k", 2e-6), ("q3_k", 2e-6)])
def test_gemv_vs_ref(pvr, quant, tol):
    from golden.make_golden_port import gemv_inputs
    assert rel_l2(P.matmul(*gemv_inputs(quant)), pvr[f"gemv_{quant}"]) < tol


@pytest.mark.parametrize("preset", ["tiny_v2lite", "tiny_v2", "tiny_v3"])
@pytest.mark.parametrize("quant,tol", [("fp32", 1e-3), ("f8e5m2", 1e-3), ("q3_k", 5e-2)])
def test_forward_port_vs_ref(ckpt, pvr, preset, quant, tol):
    from golden.make_golden_port import FORWARD_MINT_KW, FORWARD_TOKENS
    p = O.PortSession(ckpt(preset, quant, **FORWARD_MINT_KW))
    exp = pvr[f"forward_{preset}_{quant}_logits"]
    for pos, tok in enumerate(FORWARD_TOKENS):
        p.forward(tok, pos)
        assert rel_l2(_logits(p, pvr), exp[pos]) < tol


@pytest.mark.parametrize("preset", ["tiny_v2", "tiny_v3"])
@pytest.mark.parametrize("quant,tol", [("fp32", 1e-3), ("fp16", 1e-3), ("f8e5m2", 1e-3), ("q2_k", 1.5e-1)])   # (q2_k T3: sanity
# ceiling only — one Q8_K rounding flip between the two builds moves random-block logits by several 1e-2, see
# profiles/r02_reference_self_sensitivity.txt; the T2 part below is the proof)
def test_mla_block_port_vs_ref(ckpt, pvr, preset, quant, tol):
    """BlockMLA, layer by layer on the reference's cache rows, each layer against the reference's output for the same input
    (tier T2), then teacher-forced logits (T3)."""
    from golden.make_golden_port import FORWARD_TOKENS, MLA_T2_TOKENS, mla_mint_kw
    d = ckpt(preset, quant, **mla_mint_kw(quant))
    key = f"mla_{preset}_{quant}"
    p = O.PortSession(d)
    xi, n_layers, errs = pvr["x_idx"], p.c["n_layers"], []
    for pos, tok in enumerate(MLA_T2_TOKENS):
        p.copy_embedding(tok)
        for l in range(n_layers):
            for which, name in ((0, "_t2_latent"), (1, "_t2_rope")):
                rows = pvr[key + name][l]
                p.kv_cache(l, which)[:rows.size] = rows
            p.block(l, pos, 0, pos, pos + 1)
            errs.append(rel_l2(p.buffer("x")[xi], pvr[key + "_t2_x"][pos * n_layers + l]))
    errs = np.array(errs)
    if quant == "q2_k":   # Q8_K rounding flips between the two builds (-O3 -ffast-math vs -O2): most pairs clean, flips bounded
        assert np.median(errs) < 1e-5 and errs.max() < 5e-2, errs
    else:
        assert errs.max() < 1e-4, errs
    p = O.PortSession(d)
    for pos, tok in enumerate(FORWARD_TOKENS):
        p.forward(tok, pos)
        assert rel_l2(_logits(p, pvr), pvr[key + "_logits"][pos]) < tol, (preset, quant, pos)


def _sink_ring(ckpt, pvr, name):
    from golden.make_golden_port import SINK_STEPS, sink_mint_kw
    preset, kw = sink_mint_kw(name)
    p = O.PortSession(ckpt(preset, "fp32", **kw))
    for pos in range(SINK_STEPS):
        p.forward(pos * 7 % 1024, pos)
        assert rel_l2(_logits(p, pvr), pvr[f"{name}_logits"][pos]) < 1e-3, pos


def test_mla_sink_ring_port_vs_ref(ckpt, pvr):
    """MLA past original_max_position: 2 sink rows, ring overwrite, sink rope keys re-rotated (src/infer.cpp:1099-1111)."""
    _sink_ring(ckpt, pvr, "mla_sink")


def test_sink_ring_port_vs_ref(ckpt, pvr):
    """pos >= original_max_position: 2 sinks kept, ring overwrite, sink keys re-rotated (src/infer.cpp:1271-1277, 1008-1020)."""
    _sink_ring(ckpt, pvr, "sink")


# ---- host logic -------------------------------------------------------------------------------------
def test_dseek_roundtrip_and_config(ckpt):
    import dseek
    import dsk
    d = ckpt("tiny_v3", "q2_k")
    md, T = dseek.read_dir(d)
    c = dsk.Config.from_metadata(md)
    assert (c.dim, c.n_layers, c.is_v3, c.scoring_sigmoid, c.topk_method, c.quant) == (512, 3, 1, 1, 1, 3)
    assert T["model.layers.1.mlp.w1.weight"].shape == (16, 256, 512 // 256 * 84)
    assert T["model.layers.1.moegate.bias"].shape == (16,)
    c2 = dsk.Config.from_metadata(md, context=64)
    assert c2.max_seq_len == 64
    oc = O.config_from_metadata(md)
    for k in ("dim", "n_heads", "kv_lora_rank", "q_lora_rank", "n_group", "topk_group", "original_max_position"):
        assert getattr(c, k) == oc[k]


def test_cabi_header_is_plain_c_and_config_layout(repo):
    """include/dsk.h is the drop-in boundary: it must compile as C99 (no C++ or torch types in the signatures) and the ctypes
    mirror of dsk_config must have the compiler's layout (field order and size are part of the ABI; use_mla was appended in
    ABI 3)."""
    import ctypes
    import subprocess
    import dsk
    hdr = os.path.join(repo, "include", "dsk.h")
    subprocess.check_call(["gcc", "-std=c99", "-fsyntax-only", "-Wall", "-Wextra", "-pedantic", "-x", "c", hdr])
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "dsk.h"\nint main(void){printf("%zu %zu %zu %zu %d\\n", sizeof(dsk_config), '
            'offsetof(dsk_config, rope_theta), offsetof(dsk_config, routed_scaling_factor), offsetof(dsk_config, use_mla), DSK_ABI_VERSION);return 0;}')
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "l.c"), os.path.join(td, "l")
        open(src, "w").write(prog)
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(repo, "include"), src, "-o", exe])
        size, o_theta, o_rsf, o_mla, abi = map(int, subprocess.check_output([exe]).split())
    C = dsk.Config
    assert (ctypes.sizeof(C), C.rope_theta.offset, C.routed_scaling_factor.offset, C.use_mla.offset) == (size, o_theta, o_rsf, o_mla)
    assert abi == dsk.ABI_VERSION
    md = {"arch": "DeepseekV2ForCausalLM", "dim": "8", "hidden_dim": "8", "n_layers": "1", "n_heads": "1", "vocab_size": "8",
          "max_seq_len": "8", "rope_theta": "1e4", "quant": "fp32", "use_mla": "1", "q_lora_rank": "4",
          "rope_scaling_original_max_position_embeddings": "4096"}
    assert dsk.Config.from_metadata(md).use_mla == 1 and dsk.Config.from_metadata(dict(md, use_mla="0")).use_mla == 0


def test_cabi_exports_every_declared_symbol(repo):
    """libdsk.so must load on a GPU-less machine and export exactly what include/dsk.h declares."""
    import dsk
    hdr = open(os.path.join(repo, "include", "dsk.h")).read()
    names = sorted(set(re.findall(r"\b(dsk_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 25
    L = ctypes.CDLL(dsk.build())
    for n in names:
        assert hasattr(L, n), n
    assert L.dsk_abi_version() == 3


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device every compute entry point must fail loudly (no silent CPU path)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import dsk
    with pytest.raises(dsk.DskError):
        dsk.init(0)
    L = dsk.lib()
    out = np.zeros(4, np.float32)
    assert L.dsk_rmsnorm(out.ctypes.data_as(dsk.f32p), out.ctypes.data_as(dsk.f32p), 4, ctypes.c_float(1e-5),
                         out.ctypes.data_as(dsk.f32p)) != 0
    assert b"no CPU fallback" in L.dsk_last_error()
