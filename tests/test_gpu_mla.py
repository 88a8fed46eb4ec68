"""GPU parity of the true-MLA blocks (checkpoints converted with --mla: BlockMLA::_attention_impl src/infer.cpp:1051-1141,
attn_mla 766-804) against the UNMODIFIED reference (oracle/_ref) or, where that is absent, the C restatement: latent + rope
KV caches bit-compared after teacher-forced tokens, tier T2 (every layer re-synchronised on the checker's input and caches) and tier T3 (teacher-forced logits), the
in-kernel token loop, and the sink re-rotation past rope_scaling_original_max_position_embeddings."""
import os
import shutil
import sys
import tempfile

import numpy as np
import pytest

import oracle as O
from conftest import rel_l2

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
import mint  # noqa: E402

pytestmark = pytest.mark.gpu

TOKENS = [0, 17, 300, 5, 911, 42, 7, 650]
T2_TOL = {"fp32": 2e-5, "fp16": 2e-5, "f8e5m2": 5e-5, "q2_k": 5e-5, "q3_k": 5e-5}
T3_TOL = {"fp32": 1e-4, "fp16": 1e-4, "f8e5m2": 5e-4, "q2_k": 8e-2, "q3_k": 8e-2}


@pytest.fixture(scope="module")
def dsk():
    import dsk as d
    d.init(0)
    return d


def _mint(preset, quant, **kw):
    d = tempfile.mkdtemp(prefix=f"dsk_mla_{preset}_{quant}_")
    if quant == "f8e5m2":
        kw.setdefault("v_head_dim", 128)      # matmul_expert's per-head scale offset needs v_head_dim % block_size[0] == 0
    mint.mint(d, preset, quant, use_mla=True, fast=True, **kw)
    return d


CASES = [("tiny_v2", "fp32"), ("tiny_v3", "fp32"), ("tiny_v2", "fp16"), ("tiny_v2", "f8e5m2"), ("tiny_v3", "f8e5m2"),
         ("tiny_v2", "q2_k"), ("tiny_v3", "q3_k")]


@pytest.mark.parametrize("preset,quant", CASES)
def test_mla_layers_caches_and_logits(dsk, preset, quant):
    d = _mint(preset, quant)
    try:
        m = dsk.Model.from_dir(d)
        assert m.cfg.use_mla == 1
        o = O.open_session(d)
        kq = quant in ("q2_k", "q3_k")
        errs = []
        for pos, tok in enumerate(TOKENS[:5]):
            o.copy_embedding(tok)
            m.copy_embedding(tok)
            for l in range(m.cfg.n_layers):
                m.set_buffer("x", o.buffer("x").copy())
                for which in (0, 1):
                    m.set_kv_cache(l, which, o.kv_cache(l, which))
                o.block(l, pos, 0, pos, pos + 1)
                m.block(l, pos, 0, pos, pos + 1)
                e = rel_l2(m.buffer("x"), o.buffer("x"))
                errs.append(e)
                if not kq or e < 1e-5:
                    # the new cache rows: fp16 of fp32 values that agree to ~1e-6 -> at most the odd 1-ulp rounding flip
                    for which, w in ((0, m.cfg.kv_lora_rank), (1, m.cfg.qk_rope_head_dim)):
                        a = m.kv_cache(l, which)[pos * w:(pos + 1) * w].view(np.float16).astype(np.float32)
                        b = o.kv_cache(l, which)[pos * w:(pos + 1) * w].view(np.float16).astype(np.float32)
                        assert np.allclose(a, b, rtol=2e-3, atol=1e-4), (preset, quant, pos, l, which, np.abs(a - b).max())
        errs = np.array(errs)
        print(f"mla {preset}/{quant} T2: median {np.median(errs):.2e} max {errs.max():.2e}")
        if kq:
            assert errs.max() < 5e-2 and (errs < 1e-5).sum() >= errs.size // 2, errs
        else:
            # one fp16 rounding flip in the new latent cache row (2^-11 of one element) moves a layer's output by a few 1e-5
            assert np.median(errs) < T2_TOL[quant] and errs.max() < 3e-4, errs
        m.close(); o.close()
        # ---- T3: teacher-forced logits -----------------------------------------------------------------------------
        m = dsk.Model.from_dir(d)
        o = O.open_session(d)
        t3 = []
        for pos, tok in enumerate(TOKENS):
            logits, am = m.forward(tok, pos)
            o.forward(tok, pos)
            exp = o.buffer("logits")
            assert np.all(np.isfinite(logits))
            t3.append(rel_l2(logits, exp))
            assert am == int(np.argmax(logits))
        print(f"mla {preset}/{quant} T3: logits rel-L2 median {np.median(t3):.2e} max {max(t3):.2e}")
        assert max(t3) < T3_TOL[quant], t3
        # ---- in-kernel token loop == host-driven loop ------------------------------------------------------------------
        m2 = dsk.Model.from_dir(d)
        for p, t in enumerate(TOKENS):
            _, am2 = m2.forward(t, p, want_logits=False)
        host, pos = [], len(TOKENS)
        for _ in range(5):
            host.append(am)
            _, am = m.forward(am, pos, want_logits=False)
            pos += 1
        dev, _ = m2.decode_greedy(len(TOKENS), 5)
        assert dev.tolist() == host
        m.close(); m2.close(); o.close()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_mla_e2e_golden(dsk, golden_dir, tmp_path):
    """Committed reference outputs (tests/golden/e2e_mla.npz, make_golden_mla.py) on MLA checkpoints mintable without the
    reference: logits, layer-0 cache rows, the last token's q_c and value up-projection."""
    from golden.make_golden_mla import CASES
    g = np.load(os.path.join(golden_dir, "e2e_mla.npz"))
    tols = {"q2_k": 8e-2, "f8e5m2": 5e-4, "fp32": 2e-3}     # (fp32 case runs past original_max_position: fp16 sink re-rounding)
    for preset, quant, kw in CASES:
        key = f"{preset}_{quant}"
        d = str(tmp_path / key)
        mint.mint(d, preset, quant, fast=True, seed=78, use_mla=True, **kw)
        m = dsk.Model.from_dir(d)
        for p, t in enumerate(g[key + "_tokens"]):
            logits, _ = m.forward(int(t), p)
            assert rel_l2(logits, g[key + "_logits"][p]) < tols[quant], (key, p)
        c, n = m.cfg, len(g[key + "_tokens"])
        if quant != "q2_k":
            assert rel_l2(m.buffer("q_c"), g[key + "_q_c_last"]) < 1e-3
            assert rel_l2(m.buffer("kv_b")[:c.n_heads * c.v_head_dim], g[key + "_kv_b_last"][:c.n_heads * c.v_head_dim]) < 1e-3
            if "original_max_position" not in kw:
                for which, name, w in ((0, "_latent_cache_l0", c.kv_lora_rank), (1, "_rope_cache_l0", c.qk_rope_head_dim)):
                    a = m.kv_cache(0, which)[:n * w].view(np.float16).astype(np.float32)
                    b = g[key + name].view(np.float16).astype(np.float32)
                    assert np.allclose(a, b, rtol=2e-3, atol=1e-4), (key, name)
        m.close()


def test_mla_sinks_past_original_max(dsk):
    """pos >= rope_scaling_original_max_position_embeddings: 2 sink rows, ring positions, sink rope keys re-rotated by one
    position per step (src/infer.cpp:1099-1111) — teacher-forced against the reference through 8 steps past the limit."""
    d = tempfile.mkdtemp(prefix="dsk_mla_sink_")
    try:
        mint.mint(d, "tiny_v3", "fp32", use_mla=True, fast=True, original_max_position=12, max_seq_len=16)
        m = dsk.Model.from_dir(d)
        o = O.open_session(d)
        rng = np.random.default_rng(5)
        worst = 0.0
        for pos in range(20):
            tok = int(rng.integers(2, 1000))
            logits, _ = m.forward(tok, pos)
            o.forward(tok, pos)
            worst = max(worst, rel_l2(logits, o.buffer("logits")))
        print(f"mla sinks: worst logits rel-L2 {worst:.2e}")
        assert worst < 2e-3          # fp16 cache rows re-rotated 8 times: rounding flips accumulate (same bound as the MHA sink test)
        for which, w in ((0, m.cfg.kv_lora_rank), (1, m.cfg.qk_rope_head_dim)):
            a = m.kv_cache(0, which)[:12 * w].view(np.float16).astype(np.float32)
            b = o.kv_cache(0, which)[:12 * w].view(np.float16).astype(np.float32)
            assert np.allclose(a, b, rtol=1e-2, atol=2e-3), (which, np.abs(a - b).max())
        m.close(); o.close()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_mla_long_context(dsk):
    """700 cached positions (several passes of every loop of the attention stage: scores 8 positions per round, softmax and
    latent mix 256 per round), teacher-forced against the reference; logits compared every 100 tokens and on the last 10."""
    d = tempfile.mkdtemp(prefix="dsk_mla_long_")
    try:
        mint.mint(d, "tiny_v2", "fp16", use_mla=True, fast=True, max_seq_len=1024)
        m = dsk.Model.from_dir(d)
        o = O.open_session(d)
        rng = np.random.default_rng(11)
        worst, n = 0.0, 700
        for pos in range(n):
            tok = int(rng.integers(2, 1000))
            if pos % 100 == 99 or pos >= n - 10:
                logits, _ = m.forward(tok, pos)
                o.forward(tok, pos)
                worst = max(worst, rel_l2(logits, o.buffer("logits")))
            else:
                m.forward(tok, pos, dsk.HYDRATE_KV_CACHE, want_logits=False)
                o.forward(tok, pos, False)
        print(f"mla long context: worst logits rel-L2 {worst:.2e} over {n} positions")
        assert worst < 1e-3
        for which, w in ((0, m.cfg.kv_lora_rank), (1, m.cfg.qk_rope_head_dim)):   # the whole cache, row by row
            a = m.kv_cache(2, which)[:n * w].view(np.float16).astype(np.float32)
            b = o.kv_cache(2, which)[:n * w].view(np.float16).astype(np.float32)
            assert rel_l2(a, b) < 1e-3, which
        m.close(); o.close()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_mla_rejections(dsk):
    """Configurations the MLA path cannot serve fail at model creation with a message, never silently."""
    d = tempfile.mkdtemp(prefix="dsk_mla_rej_")
    try:
        mint.mint(d, "tiny_v2lite", "fp32", fast=True)
        m = dsk.Model.from_dir(d)
        cfg = m.cfg
        m.close()
        cfg.use_mla = 1                     # q_lora_rank == 0 (the reference asserts, src/infer.cpp:1057)
        with pytest.raises(dsk.DskError, match="q_lora_rank"):
            dsk.Model(cfg)
    finally:
        shutil.rmtree(d, ignore_errors=True)
