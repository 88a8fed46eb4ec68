"""GPU parity, tiers T2/T3 (SURVEY §8(c)): per-layer with re-synchronised inputs, and end-to-end teacher-forced,
through the reference-shaped call surface of the C-ABI (dsk_forward / dsk_block_forward / dsk_copy_embedding)."""
import os

import numpy as np
import pytest

import oracle as O
from conftest import rel_l2

pytestmark = pytest.mark.gpu

PRESETS = ["tiny_v2lite", "tiny_v2", "tiny_v3"]
# end-to-end tolerance on logits rel-L2: fp32 summation order for the dense quants; the K-quant bound is the
# reference-vs-reference floor (SURVEY §0.4: a single Q8_K rounding flip moves the residual stream by ~1e-2)
E2E_TOL = {"fp32": 2e-4, "fp16": 2e-4, "f8e5m2": 5e-4, "q2_k": 8e-2, "q3_k": 8e-2}
TOKENS = [0, 9, 400, 33, 1001, 77, 5, 640]


def _ckpt(ckpt, preset, quant):
    """K-quant checkpoints of random valid blocks (the seed of tests/golden/e2e.npz), so the weights do not depend on whether
    the reference's quantizer (oracle/_ref) is built on this machine."""
    return ckpt(preset, quant, fast=True, seed=77) if quant in ("q2_k", "q3_k") else ckpt(preset, quant)


@pytest.fixture(scope="module")
def dsk():
    import dsk as d
    d.init(0)
    return d


@pytest.mark.parametrize("preset", PRESETS)
@pytest.mark.parametrize("quant", ["fp32", "fp16", "f8e5m2", "q2_k", "q3_k"])
def test_forward_teacher_forced(dsk, ckpt, preset, quant):
    """T3: same token ids to both engines; logits rel-L2 under the stated bound, argmax equal whenever the
    checker's top-2 margin exceeds the observed max-abs error."""
    d = _ckpt(ckpt, preset, quant)
    m = dsk.Model.from_dir(d)
    o = O.open_session(d)
    for pos, tok in enumerate(TOKENS):
        logits, am = m.forward(tok, pos)
        o.forward(tok, pos)
        exp = o.buffer("logits")
        err = rel_l2(logits, exp)
        assert err < E2E_TOL[quant], (preset, quant, pos, err)
        top2 = np.sort(exp)[-2:]
        if top2[1] - top2[0] > 2 * np.max(np.abs(logits - exp)):
            assert am == o.argmax() == int(np.argmax(logits))
        if quant in ("fp32", "fp16", "f8e5m2") and m.cfg.n_routed_experts > 0:
            assert sorted(m.active_experts().tolist()) == sorted(o.active_experts().tolist())
    m.close()
    o.close()


@pytest.mark.parametrize("preset", PRESETS)
# fp32: the reference's scalar F32 GEMV is re-associated by -ffast-math vectorisation, so its own noise is ~4e-5
@pytest.mark.parametrize("quant,tol", [("fp32", 2e-4), ("f8e5m2", 5e-5), ("q2_k", 5e-5), ("q3_k", 5e-5)])
def test_layers_resynchronised(dsk, ckpt, preset, quant, tol):
    """T2: each layer is fed the checker's layer input AND the checker's KV cache, so a rounding flip upstream
    cannot leak in; K-quant outputs then agree to fp32 re-association unless a Q8_K rounding flips inside the
    layer itself (reported as a spike; at most a small fraction may exceed the tight bound)."""
    d = _ckpt(ckpt, preset, quant)
    m = dsk.Model.from_dir(d)
    o = O.open_session(d)
    n_layers, spikes, total = m.cfg.n_layers, 0, 0
    for pos, tok in enumerate(TOKENS[:6]):
        o.copy_embedding(tok)
        m.copy_embedding(tok)
        assert np.allclose(m.buffer("x"), o.buffer("x"), rtol=1e-6, atol=1e-7)   # embedding dequant row
        for l in range(n_layers):
            x_in = o.buffer("x").copy()
            m.set_buffer("x", x_in)
            for which in (0, 1):                                     # re-sync this layer's fp16 cache
                m.set_kv_cache(l, which, o.kv_cache(l, which))
            o.block(l, pos, 0, pos, pos + 1)
            m.block(l, pos, 0, pos, pos + 1)
            err = rel_l2(m.buffer("x"), o.buffer("x"))
            total += 1
            if err >= tol:
                spikes += 1
                assert quant in ("q2_k", "q3_k") and err < 5e-2, (preset, quant, pos, l, err)
            # the cache row written this step must match to one fp16 ulp
            for which in (0, 1):
                a = m.kv_cache(l, which).view(np.float16).astype(np.float32)
                b = np.asarray(o.kv_cache(l, which)).view(np.float16).astype(np.float32)
                assert np.allclose(a, b, rtol=2e-3, atol=1e-4) or quant in ("q2_k", "q3_k")
    assert spikes <= max(1, total // 6), (spikes, total)
    m.close()
    o.close()


@pytest.mark.parametrize("quant", ["fp32", "f8e5m2"])
def test_greedy_tokens_identical(dsk, ckpt, quant):
    """Free-running greedy decode (run_completion, -t 0): token-for-token identical for the dense quants,
    via the host loop (dsk_forward + argmax) and via the device-resident loop (dsk_decode_greedy)."""
    d = ckpt("tiny_v2lite", quant)
    o = O.open_session(d)
    prompt = [0, 104, 101, 108, 108, 111]
    for p, t in enumerate(prompt):
        o.forward(t, p, p + 1 == len(prompt))
    ref_tokens, pos = [], len(prompt)
    for _ in range(24):
        t = o.argmax()
        ref_tokens.append(t)
        o.forward(t, pos)
        pos += 1
    m = dsk.Model.from_dir(d)
    for p, t in enumerate(prompt):
        _, am = m.forward(t, p, dsk.OUTPUT_LOGITS if p + 1 == len(prompt) else dsk.HYDRATE_KV_CACHE, want_logits=False)
    host_tokens, pos = [], len(prompt)
    for _ in range(24):
        host_tokens.append(am)
        _, am = m.forward(am, pos, want_logits=False)
        pos += 1
    assert host_tokens == ref_tokens
    m2 = dsk.Model.from_dir(d)
    for p, t in enumerate(prompt):
        m2.forward(t, p, dsk.OUTPUT_LOGITS if p + 1 == len(prompt) else dsk.HYDRATE_KV_CACHE, want_logits=False)
    dev_tokens, ms = m2.decode_greedy(len(prompt), 24)
    assert dev_tokens.tolist() == ref_tokens and ms > 0
    m.close(); m2.close(); o.close()


def test_sink_ring(dsk, ckpt):
    """pos >= original_max_position: attention sinks + ring overwrite + fp16 sink re-rotation (src/infer.cpp:1271-1277,
    1008-1020), V2 (de-interleaving) and V3 (interleaved) layouts."""
    for preset in ("tiny_v2lite", "tiny_v3"):
        d = ckpt(preset, "fp32", original_max_position=8)
        m = dsk.Model.from_dir(d)
        o = O.open_session(d)
        for pos in range(15):
            tok = pos * 7 % 1024
            logits, _ = m.forward(tok, pos)
            o.forward(tok, pos)
            assert rel_l2(logits, o.buffer("logits")) < 2e-3, (preset, pos)  # fp16 re-rounding of sink keys each step
        m.close(); o.close()


def test_e2e_golden(dsk, golden_dir, tmp_path):
    """Committed reference logits (tests/golden/e2e.npz) on checkpoints mintable without the reference."""
    import mint
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    for preset, quant, tol in (("tiny_v3", "q2_k", 8e-2), ("tiny_v2lite", "f8e5m2", 5e-4)):
        d = str(tmp_path / f"{preset}_{quant}")
        mint.mint(d, preset, quant, fast=True, seed=77)
        m = dsk.Model.from_dir(d)
        for p, t in enumerate(g[f"{preset}_{quant}_tokens"]):
            logits, _ = m.forward(int(t), p)
            assert rel_l2(logits, g[f"{preset}_{quant}_logits"][p]) < tol, (preset, quant, p)
        m.close()


def _sample_restated(logits, temperature, top_p, coin):
    """Sampler::sample (src/sampler.cpp:41-75) restated: fp32 sequential sums, the UNSORTED walk, r = coin * top_p."""
    if temperature == 0.0:
        return int(np.argmax(logits))
    l = logits.astype(np.float32)
    e = np.exp(((l - l.max()) / np.float32(temperature)).astype(np.float32)).astype(np.float32)
    s = np.float32(0)
    for v in e:
        s = np.float32(s + v)
    p = (e / s).astype(np.float32)
    cum = np.cumsum(p, dtype=np.float32)          # sequential fp32 accumulation, like the reference's loop
    r = np.float32(np.float32(coin) * np.float32(top_p))
    hit = np.nonzero(cum >= r)[0]
    return int(hit[0]) if hit.size else l.size - 1, cum


def test_device_sampling(dsk, ckpt):
    """dsk_sample / dsk_sample_prob (Sampler::sample / sample_prob on the device, src/sampler.cpp:12-75) against the
    restated host algorithm on the model's own logits; the picked index may differ only when r falls within fp32
    summation error of a bucket edge (then it must be the neighbour)."""
    d = ckpt("tiny_v2lite", "fp32")
    m = dsk.Model.from_dir(d)
    rng = np.random.default_rng(8)
    logits, am = m.forward(7, 0)
    logits = logits.copy()
    assert m.sample(0.0, 0.95, 0.3) == am == int(np.argmax(logits))
    mx = logits.max()
    pr = np.exp(logits - mx) / np.exp(logits - mx).sum()
    for idx in (0, 5, int(np.argmax(logits)), logits.size - 1):
        assert abs(m.sample_prob(idx) - pr[idx]) <= 2e-6 * max(pr[idx], 1e-3)
    mism = 0
    for t in range(60):
        T, top_p, coin = float(rng.choice([0.5, 1.0, 1.7])), float(rng.choice([0.95, 1.0, 0.5])), float(rng.uniform(0, 1))
        exp, cum = _sample_restated(logits, T, top_p, coin)
        got = m.sample(T, top_p, coin)
        if got != exp:
            mism += 1
            r = coin * top_p
            assert abs(got - exp) <= 2 and min(abs(cum[got] - r), abs(cum[exp] - r)) < 1e-4, (t, got, exp)
    assert mism <= 3
    assert m.sample(1.0, 1.0, 0.0) == 0                       # r = 0: the first index already satisfies cumsum >= r
    m.forward(3, 1, dsk.HYDRATE_KV_CACHE)
    with pytest.raises(dsk.DskError):
        m.sample(1.0, 0.95, 0.5)                              # a hydrate-only forward leaves no logits to sample from
    m.close()


def test_errors_are_loud(dsk, ckpt):
    d = ckpt("tiny_v2lite", "fp32")
    m = dsk.Model.from_dir(d)
    with pytest.raises(dsk.DskError):
        m.forward(10 ** 6, 0)          # token out of range
    with pytest.raises(dsk.DskError):
        m.forward(1, 10 ** 6)          # past the KV cache (the reference would overrun it)
    with pytest.raises(dsk.DskError):
        m.decode_greedy(5, 4)          # must follow a forward
    m.forward(1, 0, dsk.OUTPUT_LOGITS)
    m.forward(2, 1, dsk.HYDRATE_KV_CACHE)
    with pytest.raises(dsk.DskError):
        m.decode_greedy(2, 4)          # hydrate-only forward: no LM-head stage ran, there is no arg-max to feed the loop
    m.forward(3, 2, dsk.OUTPUT_LOGITS)
    toks, _ = m.decode_greedy(3, 2)    # and after a logits forward it works
    assert toks.size == 2
    m.close()
    import dseek
    md, T = dseek.read_dir(d)
    m2 = dsk.Model(dsk.Config.from_metadata(md))
    with pytest.raises(dsk.DskError):
        m2.finalize()                  # missing tensors (check_tensor, src/model.cpp:129-136)
    with pytest.raises(dsk.DskError):
        m2.upload("model.norm.weight", "F32", (3,), np.zeros(3, np.float32))   # wrong size
    # dtype / shape validation of check_tensor / QTensor::from_codec_tensor (src/codec.cpp:166-234)
    dim = m2.cfg.dim
    with pytest.raises(dsk.DskError):
        m2.upload("model.norm.weight", "F16", (dim,), np.zeros(dim, np.float16))            # wrong dtype
    with pytest.raises(dsk.DskError):
        m2.upload("model.norm.weight", "F32", (dim // 2, 2), np.zeros(dim, np.float32))      # right bytes, wrong shape
    with pytest.raises(dsk.DskError):
        m2.upload("model.layers.0.attn.wo.weight", "F32", (m2.cfg.n_heads * m2.cfg.v_head_dim, dim),
                  np.zeros((m2.cfg.n_heads * m2.cfg.v_head_dim, dim), np.float32))           # transposed shape
    m2.upload("model.norm.weight", "F32", (dim,), np.ones(dim, np.float32))
    with pytest.raises(dsk.DskError):
        m2.upload("model.norm.weight", "F32", (dim,), np.ones(dim, np.float32))              # uploaded twice
    m2.close()
    bad = dsk.Config.from_metadata(md)
    bad.qk_rope_head_dim = 192
    with pytest.raises(dsk.DskError):
        dsk.Model(bad)                 # limits of the kernels are checked at model creation, not discovered as garbage
