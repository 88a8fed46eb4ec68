"""Generates tests/golden/port_vs_ref.npz from the UNMODIFIED reference (oracle/_ref/libdsref.so): the outputs that the
port-vs-reference tests of tests/test_oracle.py compare against, on inputs that are seeded and mintable without the reference
(K-quant checkpoints and matrices use random valid blocks, oracle/mint.py fast=True; the checkpoints use the seed of e2e.npz).

To stay small, logits are stored as float16 at a fixed sample of LOGIT_SAMPLE vocabulary indices (the float16 rounding adds
~3e-4 in quadrature to a relative L2 error, well under the 1e-3 bounds), BlockMLA layer outputs as float32 at X_SAMPLE
indices of the residual stream, and Q8_K blocks as SHA-256 digests (that comparison is bit-exact).

Run where oracle/_ref is built (`make -C oracle ref` with the reference sources present):
    python tests/golden/make_golden_port.py
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(REPO, "oracle"))
import oracle as O  # noqa: E402
import mint  # noqa: E402

LOGIT_SAMPLE, X_SAMPLE = 256, 128
GEMV_CASES = ("fp32", "fp16", "f8e5m2", "q2_k", "q3_k")
FORWARD_CASES = [(p, q) for p in ("tiny_v2lite", "tiny_v2", "tiny_v3") for q in ("fp32", "f8e5m2", "q3_k")]
FORWARD_TOKENS = [0, 9, 400, 33, 1001]
MLA_CASES = [(p, q) for p in ("tiny_v2", "tiny_v3") for q in ("fp32", "fp16", "f8e5m2", "q2_k")]
MLA_T2_TOKENS = [0, 9, 400, 33]
SINK_CASES = {"mla_sink": ("tiny_v3", dict(use_mla=True)), "sink": ("tiny_v2lite", {})}
SINK_STEPS = 14


def q8k_inputs():
    rng = np.random.default_rng(5)
    for _ in range(100):
        yield (rng.standard_normal(1024) * 10 ** rng.uniform(-4, 4)).astype(np.float32)


def gemv_inputs(quant):
    rng = np.random.default_rng(6)
    d, n = 96, 1024
    w = (rng.standard_normal((d, n)) * n ** -0.5).astype(np.float32)
    x = rng.standard_normal(n).astype(np.float32)
    scale = None
    if quant == "fp16":
        wq = w.astype(np.float16)
    elif quant == "f8e5m2":
        wq, scale = mint.f8e5m2_blockwise(w)
    elif quant in ("q2_k", "q3_k"):
        wq = mint.kquant_rows(w, quant, True, rng)
    else:
        wq = w
    return x, wq, quant, d, n, scale


FORWARD_MINT_KW = dict(fast=True, seed=77)


def mla_mint_kw(quant):
    return dict(use_mla=True, fast=True, **({"v_head_dim": 128} if quant == "f8e5m2" else {}))


def sink_mint_kw(name):
    preset, kw = SINK_CASES[name]
    return preset, dict(kw, fast=True, original_max_position=8)


def digest(a: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


if __name__ == "__main__":
    out = {}
    li = np.sort(np.random.default_rng(0).choice(1024, LOGIT_SAMPLE, replace=False)).astype(np.int32)
    xi = np.sort(np.random.default_rng(1).choice(512, X_SAMPLE, replace=False)).astype(np.int32)
    out["logit_idx"], out["x_idx"] = li, xi
    R = O.Ops("ref")
    out["q8k_sha256"] = np.stack([digest(R.quantize_q8k(x)) for x in q8k_inputs()])
    for quant in GEMV_CASES:
        x, wq, q, d, n, scale = gemv_inputs(quant)
        out[f"gemv_{quant}"] = R.matmul(x, wq, q, d, n, scale)

    def logits16(s):
        return s.buffer("logits")[li].astype(np.float16)

    with tempfile.TemporaryDirectory() as td:
        for preset, quant in FORWARD_CASES:
            d = os.path.join(td, f"fw_{preset}_{quant}")
            mint.mint(d, preset, quant, **FORWARD_MINT_KW)
            r = O.RefSession(d)
            lg = []
            for pos, tok in enumerate(FORWARD_TOKENS):
                r.forward(tok, pos)
                lg.append(logits16(r))
            out[f"forward_{preset}_{quant}_logits"] = np.stack(lg)
            r.close()
        for preset, quant in MLA_CASES:
            d = os.path.join(td, f"mla_{preset}_{quant}")
            mint.mint(d, preset, quant, **mla_mint_kw(quant))
            c = O.config_from_metadata(O.dseek.read_dir(d)[0])
            key = f"mla_{preset}_{quant}"
            # T2: every (position, layer) gets the port's input and the reference's cache rows; the port is deterministic
            # (no reductions across threads), so the test re-creates the same inputs.  The output is sampled.
            r, p, xs = O.RefSession(d), O.PortSession(d), []
            for pos, tok in enumerate(MLA_T2_TOKENS):
                p.copy_embedding(tok)
                for l in range(c["n_layers"]):
                    r.buffer("x")[:] = p.buffer("x")
                    for which in (0, 1):
                        p.kv_cache(l, which)[:] = r.kv_cache(l, which)
                    r.block(l, pos, 0, pos, pos + 1)
                    p.block(l, pos, 0, pos, pos + 1)
                    xs.append(r.buffer("x")[xi].copy())
            out[key + "_t2_x"] = np.stack(xs)
            # the cache rows of the positions before the last one: what each later block reads
            n = len(MLA_T2_TOKENS) - 1
            out[key + "_t2_latent"] = np.stack([r.kv_cache(l, 0)[:n * c["kv_lora_rank"]].copy() for l in range(c["n_layers"])])
            out[key + "_t2_rope"] = np.stack([r.kv_cache(l, 1)[:n * c["qk_rope_head_dim"]].copy() for l in range(c["n_layers"])])
            r.close()
            r, lg = O.RefSession(d), []
            for pos, tok in enumerate(FORWARD_TOKENS):
                r.forward(tok, pos)
                lg.append(logits16(r))
            out[key + "_logits"] = np.stack(lg)
            r.close()
        for name in SINK_CASES:
            preset, kw = sink_mint_kw(name)
            d = os.path.join(td, name)
            mint.mint(d, preset, "fp32", **kw)
            r, lg = O.RefSession(d), []
            for pos in range(SINK_STEPS):
                r.forward(pos * 7 % 1024, pos)
                lg.append(logits16(r))
            out[f"{name}_logits"] = np.stack(lg)
            r.close()
    np.savez_compressed(os.path.join(HERE, "port_vs_ref.npz"), **out)
    print("golden written:", {k: v.shape for k, v in out.items()})
