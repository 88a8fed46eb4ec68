#!/usr/bin/env python
"""bench.py — single-batch DeepSeek decode throughput on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this engine (libdsk.so), one rank per GPU
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU path (oracle/_ref)

Workload (every N): DeepSeek-V2 236B shapes, Q2_K, all 60 layers (BASELINE.json configs[3]; 77 GB of weights — fits ONE
B200, so N = 1, 2, 4, 8 is a legitimate strong-scaling curve of the model north_star says to shard).  The V2-Lite
configs[1] / configs[2] numbers of round 1 are measured in the same run at N = 1 and reported under `secondary`.
`--workload v3 --quant q2_k --gpus 8` times the north-star target (220 GB, needs >= 2 GPUs).

A "step" is one fixed 128-token greedy completion (the reference's `-n 128 -t 0`, src/main.cpp:324-335) after a
16-token prompt has hydrated the KV cache.  `value` is decode-only tok/s with everything resident in HBM (the token loop
runs inside ONE persistent kernel launch per completion, device arg-max feeding the next token, CUDA-event timed); `e2e`
is the same completion driven through the reference-shaped host call `dsk_forward(token, pos, OUTPUT_LOGITS, host_logits)`
per token: control words go host->device, the vocab-sized logits come device->host, and the host samples (argmax) — copies
inside the timed region.  Weights are synthetic (no checkpoints exist offline): N(0,1)/sqrt(fan_in) quantised like
convert.py (f8e5m2) or random valid K-quant blocks, generated on the GPU and handed to dsk_upload_tensor(src_on_device=1).
The reference arm / cpu_baseline run the UNMODIFIED reference (oracle/_ref) on a full-depth checkpoint of the same shapes
minted in /dev/shm (bounded by decoding a handful of tokens, not by truncating layers) whenever it fits the host.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "deepseek.cpp_b200"))

GEN_TOKENS = 128
PROMPT_LEN = 16

# shapes: HF configs of the DeepSeek family (SURVEY §8 table); K-quants need 256-multiples (SURVEY §0.2)
WORKLOADS = {
    "v2lite": dict(arch="DeepseekV2ForCausalLM", dim=2048, hidden_dim=10944, n_layers=27, n_heads=16, vocab_size=102400,
                   qk_nope_head_dim=128, qk_rope_head_dim=64, v_head_dim=128, kv_lora_rank=512, q_lora_rank=0,
                   first_k_dense_replace=1, n_shared_experts=2, n_routed_experts=64, n_active_routed=6,
                   moe_intermediate_size=1408, routed_scaling_factor=1.0, n_group=1, topk_group=1, norm_topk_prob=0,
                   scoring_sigmoid=0, topk_method=0),
    "v2": dict(arch="DeepseekV2ForCausalLM", dim=5120, hidden_dim=12288, n_layers=60, n_heads=128, vocab_size=102400,
               qk_nope_head_dim=128, qk_rope_head_dim=64, v_head_dim=128, kv_lora_rank=512, q_lora_rank=1536,
               first_k_dense_replace=1, n_shared_experts=2, n_routed_experts=160, n_active_routed=6,
               moe_intermediate_size=1536, routed_scaling_factor=16.0, n_group=8, topk_group=3, norm_topk_prob=0,
               scoring_sigmoid=0, topk_method=1),
    "v3": dict(arch="DeepseekV3ForCausalLM", dim=7168, hidden_dim=18432, n_layers=61, n_heads=128, vocab_size=129280,
               qk_nope_head_dim=128, qk_rope_head_dim=64, v_head_dim=128, kv_lora_rank=512, q_lora_rank=1536,
               first_k_dense_replace=3, n_shared_experts=1, n_routed_experts=256, n_active_routed=8,
               moe_intermediate_size=2048, routed_scaling_factor=2.5, n_group=8, topk_group=4, norm_topk_prob=1,
               scoring_sigmoid=1, topk_method=1),
}
QUANT_IDS = {"fp32": 0, "fp16": 1, "f8e5m2": 2, "q2_k": 3, "q3_k": 4}
KBYTES = {"q2_k": 84, "q3_k": 110}


def workload_cfg(name: str, quant: str, n_layers=None, max_seq_len=1024):
    w = dict(WORKLOADS[name])
    if quant in KBYTES:
        up = lambda v: (v + 255) // 256 * 256
        w["moe_intermediate_size"] = up(w["moe_intermediate_size"])
        w["hidden_dim"] = up(w["hidden_dim"])
    if n_layers:
        w["n_layers"] = n_layers
    w["max_seq_len"] = max_seq_len
    w["quant"] = quant
    return w


def tensor_plan(w):
    """(name, rows, cols, n_experts) for every quantised tensor + F32 extras, in .dseek naming (src/model.cpp:766-871)."""
    dim, nh = w["dim"], w["n_heads"]
    hd = w["qk_nope_head_dim"] + w["qk_rope_head_dim"]
    mi, E, ns = w["moe_intermediate_size"], w["n_routed_experts"], w["n_shared_experts"]
    plan, f32 = [("model.embed", w["vocab_size"], dim, 0), ("model.output", w["vocab_size"], dim, 0)], [("model.norm.weight", dim)]
    for l in range(w["n_layers"]):
        p = f"model.layers.{l}."
        f32 += [(p + "attn.norm.weight", dim), (p + "mlp.norm.weight", dim), (p + "attn.kv_a_norm.weight", w["kv_lora_rank"])]
        if w.get("use_mla"):   # convert.py --mla (convert.py:384-440): absorbed wc, rope-only wq_rope_b, per-head wv_b
            f32.append((p + "attn.q_a_norm.weight", w["q_lora_rank"]))
            plan += [(p + "attn.wq_a", w["q_lora_rank"], dim, 0), (p + "attn.wc", nh * w["kv_lora_rank"], w["q_lora_rank"], 0),
                     (p + "attn.wq_rope_b", nh * w["qk_rope_head_dim"], w["q_lora_rank"], 0),
                     (p + "attn.wkv_a", w["kv_lora_rank"] + w["qk_rope_head_dim"], dim, 0),
                     (p + "attn.wv_b", nh * w["v_head_dim"], w["kv_lora_rank"], 0), (p + "attn.wo", dim, nh * w["v_head_dim"], 0)]
        else:
            if w["q_lora_rank"] > 0:
                f32.append((p + "attn.q_a_norm.weight", w["q_lora_rank"]))
                plan += [(p + "attn.wq_a", w["q_lora_rank"], dim, 0), (p + "attn.wq_b", nh * hd, w["q_lora_rank"], 0)]
            else:
                plan.append((p + "attn.wq", nh * hd, dim, 0))
            plan += [(p + "attn.wkv_a", w["kv_lora_rank"] + w["qk_rope_head_dim"], dim, 0),
                     (p + "attn.wkv_b", nh * (w["qk_nope_head_dim"] + w["v_head_dim"]), w["kv_lora_rank"], 0),
                     (p + "attn.wo", dim, nh * w["v_head_dim"], 0)]
        if E > 0 and l >= w["first_k_dense_replace"]:
            f32.append((p + "moegate.weight", E * dim))
            if w["arch"] == "DeepseekV3ForCausalLM":
                f32.append((p + "moegate.bias", E))
            plan += [(p + "mlp.w1", mi, dim, E), (p + "mlp.w2", dim, mi, E), (p + "mlp.w3", mi, dim, E)]
            if ns > 0:
                plan += [(p + "shared_mlp.w1", ns * mi, dim, 0), (p + "shared_mlp.w2", dim, ns * mi, 0),
                         (p + "shared_mlp.w3", ns * mi, dim, 0)]
        else:
            plan += [(p + "mlp.w1", w["hidden_dim"], dim, 0), (p + "mlp.w2", dim, w["hidden_dim"], 0),
                     (p + "mlp.w3", w["hidden_dim"], dim, 0)]
    return plan, f32


def make_config(dsk, w):
    c = dsk.Config()
    for k in ("dim", "hidden_dim", "n_layers", "n_heads", "vocab_size", "max_seq_len", "first_k_dense_replace",
              "n_shared_experts", "n_routed_experts", "n_active_routed", "moe_intermediate_size", "n_group", "topk_group",
              "norm_topk_prob", "scoring_sigmoid", "topk_method", "kv_lora_rank", "q_lora_rank", "qk_nope_head_dim",
              "qk_rope_head_dim", "v_head_dim"):
        setattr(c, k, int(w[k]))
    c.rope_theta, c.norm_eps, c.act_silu = 10000.0, 1e-6, 1
    c.routed_scaling_factor = float(w["routed_scaling_factor"])
    c.is_v3 = 1 if w["arch"] == "DeepseekV3ForCausalLM" else 0
    c.quant = QUANT_IDS[w["quant"]]
    c.bs0, c.bs1 = (128, 128) if w["quant"] == "f8e5m2" else (0, 0)
    c.original_max_position = 4096
    c.use_mla = 1 if w.get("use_mla") else 0
    return c


def mint_on_gpu(dsk, w, rank, n_ranks, device):
    """Random-init weights of the named architecture, generated on the GPU (SURVEY §8(d) / N1)."""
    import zlib

    import torch
    dev = torch.device("cuda", device)
    m = dsk.Model(make_config(dsk, w), rank, n_ranks, device)

    def seed(name):   # per-tensor seed: every rank mints identical tensors no matter which expert chunks it skips
        torch.manual_seed(1234 + zlib.crc32(name.encode()))
    quant = w["quant"]
    plan, f32 = tensor_plan(w)
    E = w["n_routed_experts"]
    per = -(-E // n_ranks) if E else 0
    for name, n in f32:
        seed(name)
        if name.endswith("moegate.weight"):
            t = torch.randn(n, device=dev) * (w["dim"] ** -0.5) * 4.0
        elif name.endswith("moegate.bias"):
            t = 0.01 * torch.randn(n, device=dev)
        else:
            t = 1.0 + 0.1 * torch.randn(n, device=dev)
        t = t.float().contiguous()
        shape = (w["n_routed_experts"], w["dim"]) if name.endswith("moegate.weight") else (n,)
        m.upload_device(name, "F32", shape, t.data_ptr(), t.numel() * 4)
    for name, rows, cols, ne in plan:
        lead = max(1, ne)
        seed(name)
        if quant == "f8e5m2":
            chunks_q, chunks_s = [], []
            for e0 in range(0, lead, 16):
                e1 = min(lead, e0 + 16)
                seed(f"{name}#{e0}")
                if ne and n_ranks > 1 and (e1 <= rank * per or e0 >= (rank + 1) * per):
                    # another rank's experts: the library drops them anyway; skip the randn, keep shapes
                    chunks_q.append(torch.zeros(e1 - e0, rows, cols, dtype=torch.uint8, device=dev))
                    chunks_s.append(torch.ones(e1 - e0, -(-rows // 128), -(-cols // 128), device=dev))
                    continue
                x = torch.randn(e1 - e0, rows, cols, device=dev) * (cols ** -0.5 if name != "model.embed" else 1.0)
                Rp, Cp = -(-rows // 128) * 128, -(-cols // 128) * 128
                xp = torch.zeros(e1 - e0, Rp, Cp, device=dev)
                xp[:, :rows, :cols] = x
                blk = xp.view(e1 - e0, Rp // 128, 128, Cp // 128, 128)
                amax = blk.abs().amax(dim=(2, 4))
                scale = 57344.0 / amax.clamp(min=1e-12)                       # convert.py:216-244
                q = (blk * scale[:, :, None, :, None]).clamp(-57344.0, 57344.0).to(torch.float8_e5m2)
                chunks_q.append(q.view(e1 - e0, Rp, Cp)[:, :rows, :cols].contiguous().view(torch.uint8))
                chunks_s.append(scale.float().reciprocal())
                del x, xp, blk, q
            q = torch.cat(chunks_q).contiguous()
            s = torch.cat(chunks_s).float().contiguous()
            shape = (ne, rows, cols) if ne else (rows, cols)
            sshape = tuple(s.shape) if ne else tuple(s.shape[1:])
            m.upload_device(name + ".weight", "F8_E5M2", shape, q.data_ptr(), q.numel())
            m.upload_device(name + ".scale", "F32", sshape, s.data_ptr(), s.numel() * 4)
            del q, s, chunks_q, chunks_s
        elif quant in KBYTES:
            bb, nb = KBYTES[quant], cols // 256
            q = torch.randint(0, 256, (lead, rows, nb, bb), dtype=torch.uint8, device=dev)
            d = np.float16(0.1 / np.sqrt(cols))
            if quant == "q2_k":
                q[..., 80:82] = torch.from_numpy(np.frombuffer(d.tobytes(), np.uint8).copy()).to(dev)
                q[..., 82:84] = torch.from_numpy(np.frombuffer(np.float16(d * 1.5).tobytes(), np.uint8).copy()).to(dev)
            else:
                q[..., 108:110] = torch.from_numpy(np.frombuffer(np.float16(d / 8).tobytes(), np.uint8).copy()).to(dev)
            shape = (ne, rows, nb * bb) if ne else (rows, nb * bb)
            m.upload_device(name + ".weight", "U8", shape, q.data_ptr(), q.numel())
            del q
        else:
            x = torch.randn(lead, rows, cols, device=dev) * (cols ** -0.5 if name != "model.embed" else 1.0)
            if quant == "fp16":
                x = x.half()
            x = x.contiguous()
            m.upload_device(name + ".weight", "F16" if quant == "fp16" else "F32", x.shape, x.data_ptr(),
                            x.numel() * x.element_size())
            del x
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    m.finalize()
    return m


T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries exactly one JSON line)"""
    print(f"[bench +{time.time() - T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def prompt_ids(vocab):
    return [(7919 * (i + 1)) % vocab for i in range(PROMPT_LEN)]


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
# CPU reference leg (oracle/_ref = the unmodified reference compiled in the build container)
# ----------------------------------------------------------------------------------------------------
def ckpt_metadata(w, n_layers):
    quant = w["quant"]
    md = {"arch": w["arch"], "use_mla": "1" if w.get("use_mla") else "0", "quant": quant, "dim": w["dim"], "hidden_dim": w["hidden_dim"], "n_layers": n_layers,
          "n_heads": w["n_heads"], "vocab_size": w["vocab_size"], "max_seq_len": w["max_seq_len"], "bos_token_id": 0,
          "eos_token_id": 1, "rope_theta": 10000.0, "norm_eps": 1e-6, "norm_type": "rmsnorm", "act_type": "silu",
          "first_k_dense_replace": w["first_k_dense_replace"], "kv_lora_rank": w["kv_lora_rank"], "q_lora_rank": w["q_lora_rank"],
          "qk_nope_head_dim": w["qk_nope_head_dim"], "qk_rope_head_dim": w["qk_rope_head_dim"], "v_head_dim": w["v_head_dim"],
          "n_shared_experts": w["n_shared_experts"], "n_routed_experts": w["n_routed_experts"],
          "n_active_routed": w["n_active_routed"], "moe_intermediate_size": w["moe_intermediate_size"],
          "routed_scaling_factor": w["routed_scaling_factor"], "n_group": w["n_group"],
          "norm_topk_prob": "True" if w["norm_topk_prob"] else "False",
          "scoring_func": "sigmoid" if w["scoring_sigmoid"] else "softmax", "topk_group": w["topk_group"],
          "topk_method": "group_limited_greedy" if w["topk_method"] else "greedy", "rope_scaling_beta_fast": 32,
          "rope_scaling_beta_slow": 1, "rope_scaling_factor": 40.0, "rope_scaling_mscale": 1.0,
          "rope_scaling_mscale_all_dim": 1.0, "rope_scaling_original_max_position_embeddings": 4096}
    if quant == "f8e5m2":
        md["quantization_block_size_0"] = 128
        md["quantization_block_size_1"] = 128
    return md


def ckpt_bytes(w, n_layers):
    """Payload bytes of a .dseek checkpoint of these shapes (weights only)."""
    wt = dict(w, n_layers=n_layers)
    plan, f32 = tensor_plan(wt)
    bpw = {"fp32": 4.0, "fp16": 2.0, "f8e5m2": 1.0 + 4.0 / 16384, "q2_k": 84 / 256, "q3_k": 110 / 256}[w["quant"]]
    return int(sum(max(1, ne) * rows * cols * bpw for _, rows, cols, ne in plan) + 4 * sum(n for _, n in f32))


def mint_cpu_truncated(w, dirname, n_layers):
    """Synthetic .dseek checkpoint of the workload's shapes with `n_layers` layers (all of them for the full-depth reference
    arm), written STRAIGHT into a memory-mapped shard: each tensor is tiled from a pool of N(0,1) values cast like
    convert.py (f8e5m2 / f16 / f32) or of random valid K-quant blocks, so a 77 GB file costs one memcpy pass, not a
    77 GB random-number run.  (Tiling repeats values across tensors; every page is still a distinct copy in /dev/shm.)"""
    import json as _json
    import struct as _struct
    rng = np.random.default_rng(1234)
    wt = dict(w, n_layers=n_layers)
    plan, f32 = tensor_plan(wt)
    quant = w["quant"]
    import torch
    pool = torch.randn(1 << 24)
    pools = {}

    def payload_pool(cols, embed):
        key = (cols, embed)
        if key in pools:
            return pools[key]
        if quant == "f8e5m2":
            a = (pool * (57344.0 / 6.0)).clamp(-57344, 57344).to(torch.float8_e5m2).view(torch.uint8).numpy()
        elif quant in KBYTES:
            bb = KBYTES[quant]
            a = rng.integers(0, 256, size=(1 << 18, bb), dtype=np.uint8)
            d = np.float16(0.1 / np.sqrt(cols))
            if quant == "q2_k":
                a[:, 80:82] = np.frombuffer(d.tobytes(), np.uint8)
                a[:, 82:84] = np.frombuffer(np.float16(d * 1.5).tobytes(), np.uint8)
            else:
                a[:, 108:110] = np.frombuffer(np.float16(d / 8).tobytes(), np.uint8)
            a = a.reshape(-1)
        else:
            sc = np.float32(1.0 if embed else cols ** -0.5)
            a = (pool.numpy() * sc).astype(np.float16 if quant == "fp16" else np.float32).view(np.uint8).reshape(-1)
        pools[key] = a
        return a

    T = []   # (name, dtype, shape, nbytes, filler) in file order
    tok = np.frombuffer(b"\0".join(b"t%d" % i for i in range(w["vocab_size"])) + b"\0", np.uint8).copy()
    T.append(("tokenizer.tokens", "U8", tok.shape, tok.nbytes, tok))
    for name, n in f32:
        if name.endswith("moegate.weight"):
            a = (rng.standard_normal(n, dtype=np.float32) * w["dim"] ** -0.5 * 4.0).reshape(w["n_routed_experts"], w["dim"])
        elif name.endswith("moegate.bias"):
            a = (0.01 * rng.standard_normal(n)).astype(np.float32)
        else:
            a = (1.0 + 0.1 * rng.standard_normal(n)).astype(np.float32)
        T.append((name, "F32", a.shape, a.nbytes, a))
    for name, rows, cols, ne in plan:
        lead = max(1, ne)
        embed = name == "model.embed"
        if quant == "f8e5m2":
            shape = ((ne,) if ne else ()) + (rows, cols)
            T.append((name + ".weight", "F8_E5M2", shape, lead * rows * cols, ("tile", payload_pool(cols, embed), 1)))
            sshape = ((ne,) if ne else ()) + (-(-rows // 128), -(-cols // 128))
            sc = 6.0 / 57344.0 * (1.0 if embed else cols ** -0.5)
            sa = np.full(sshape, sc, np.float32)
            T.append((name + ".scale", "F32", sshape, sa.nbytes, sa))
        elif quant in KBYTES:
            bb, nb = KBYTES[quant], cols // 256
            shape = ((ne,) if ne else ()) + (rows, nb * bb)
            T.append((name + ".weight", "U8", shape, lead * rows * nb * bb, ("tile", payload_pool(cols, embed), bb)))
        else:
            isz = 2 if quant == "fp16" else 4
            shape = ((ne,) if ne else ()) + (rows, cols)
            T.append((name + ".weight", "F16" if quant == "fp16" else "F32", shape, lead * rows * cols * isz,
                      ("tile", payload_pool(cols, embed), isz)))
    T.sort(key=lambda t: t[0])
    header = {"__metadata__": {str(k): str(v) for k, v in ckpt_metadata(w, n_layers).items()}}
    off = 0
    for name, dt, shape, nbytes, _ in T:
        header[name] = {"dtype": dt, "shape": [int(v) for v in shape], "data_offsets": [off, off + nbytes]}
        off += nbytes
    hjson = _json.dumps(header, separators=(",", ":")).encode("utf-8")
    hjson += b" " * ((-len(hjson)) % 8)
    os.makedirs(dirname, exist_ok=True)
    path = os.path.join(dirname, "shard_000.dseek")
    total = 8 + len(hjson) + off
    with open(path, "wb") as f:
        f.truncate(total)
    mm = np.memmap(path, dtype=np.uint8, mode="r+")
    mm[:8] = np.frombuffer(_struct.pack("<Q", len(hjson)), np.uint8)
    mm[8:8 + len(hjson)] = np.frombuffer(hjson, np.uint8)
    base = 8 + len(hjson)
    for name, dt, shape, nbytes, fill in T:
        b0 = base + header[name]["data_offsets"][0]
        if isinstance(fill, tuple):
            _, pl, unit = fill
            start = int(rng.integers(0, pl.size // unit)) * unit      # unit-aligned phase into the pool
            done = 0
            while done < nbytes:
                n = min(nbytes - done, pl.size - start)
                mm[b0 + done:b0 + done + n] = pl[start:start + n]
                done += n
                start = 0
        else:
            mm[b0:b0 + nbytes] = np.ascontiguousarray(fill).view(np.uint8).reshape(-1)
    mm.flush()
    del mm
    return total


def host_free_bytes(path):
    try:
        st = os.statvfs(path)
        return st.f_bavail * st.f_frsize
    except Exception:
        return 0


def cpu_reference_leg(w, steps, warmup, tokens_per_step=6):
    """Times the UNMODIFIED reference (oracle/_ref/libdsref.so) on this box's host cores.  The sample is bounded by the
    number of decoded tokens, not by the model: a FULL-DEPTH checkpoint of the workload's shapes is minted in /dev/shm
    whenever it fits (<= 120 GB and <= 40 % of the free space); otherwise (V3-size) a 3-layer truncation with per-block
    times extrapolated, labelled as such.  Returns (tok/s, seconds actually spent decoding, description dict)."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import oracle as O
    if O.ref_lib() is None:
        O.port_lib()
        raise RuntimeError("oracle/_ref/libdsref.so is not present")
    nl_full, fk = w["n_layers"], w["first_k_dense_replace"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else tempfile.gettempdir()
    full_bytes = ckpt_bytes(w, nl_full)
    full = full_bytes <= 120e9 and full_bytes <= 0.4 * host_free_bytes(base) and os.environ.get("DSK_REF_TRUNCATE", "0") != "1"
    n_ck = nl_full if full else min(nl_full, fk + 2)
    d = tempfile.mkdtemp(prefix="dsk_ref_", dir=base)
    try:
        t0 = time.time()
        log(f"cpu reference: minting {'full-depth ' if full else ''}{n_ck}-layer checkpoint ({ckpt_bytes(w, n_ck) / 1e9:.1f} GB) in {d}")
        mint_cpu_truncated(w, d, n_ck)
        log(f"cpu reference: minted in {time.time() - t0:.1f} s")
        cores = os.cpu_count() or 1
        best = None
        cands = sorted({min(cores, 32), max(1, cores // 2)}) if full and full_bytes > 30e9 else sorted({min(cores, 16), min(cores, 32), max(1, cores // 2)})
        n_tok = max(1, (warmup + steps)) * tokens_per_step
        for threads in cands:
            log(f"cpu reference: {threads} threads")
            O.ref_lib().ref_set_num_threads(threads)
            s = O.RefSession(d, 0)
            pr = prompt_ids(w["vocab_size"])[:4]
            if full:
                s.timed_decode(pr, 1)                                   # page-touch pass (weights are in tmpfs already)
                secs, _ = s.timed_decode(pr, n_tok)
                tps, spent = n_tok / secs, secs
            else:
                for p, t in enumerate(pr):
                    s.forward(t, p, True)
                pos, per_tok, spent = len(pr), [], 0.0
                for it in range(n_tok):
                    tok = s.argmax()
                    t0 = time.perf_counter(); s.forward(tok, pos, True); t_f = time.perf_counter() - t0
                    tb = []
                    for l in range(n_ck):
                        t0 = time.perf_counter(); s.block(l, pos, 0, pos, pos + 1); tb.append(time.perf_counter() - t0)
                    pos += 1
                    spent += t_f + sum(tb)
                    if it >= warmup * tokens_per_step:
                        t_dense = float(np.mean(tb[:fk])) if fk else 0.0
                        t_moe = float(np.mean(tb[fk:])) if n_ck > fk else 0.0
                        per_tok.append(max(0.0, t_f - sum(tb)) + fk * t_dense + (nl_full - fk) * t_moe)
                tps = 1.0 / float(np.mean(per_tok))
            s.close()
            if best is None or tps > best[0]:
                best = (tps, threads, spent)
        sample = (f"full-depth {nl_full}-layer checkpoint of the workload's shapes ({full_bytes / 1e9:.1f} GB in {base}), {n_tok} greedy tokens "
                  f"decoded after a 4-token prompt (ref_timed_decode = run_completion's loop), no extrapolation") if full else \
                 (f"{n_ck}-layer truncation ({fk} dense + {n_ck - fk} MoE + LM head) of the workload's shapes, {n_tok} decoded tokens, "
                  f"per-block times EXTRAPOLATED to {nl_full} layers (the full checkpoint, {full_bytes / 1e9:.0f} GB, is not minted on the host)")
        return best[0], best[2], {"kind": "reference", "cores": best[1], "host_cpus": cores, "extrapolated": not full,
                                  "sample": sample + f"; unmodified reference (-O3 -ffast-math -fopenmp -mavx2), best of OMP threads {cands}"}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


# ----------------------------------------------------------------------------------------------------
DTYPES = {"f8e5m2": "f8e5m2 weights x f32 activations", "q2_k": "u2 x i8 integer dot (Q2_K x Q8_K), f32 accumulate",
          "q3_k": "u3 x i8 integer dot (Q3_K x Q8_K), f32 accumulate", "fp16": "f16 weights x f32", "fp32": "f32"}
NAMES = {"v2lite": "DeepSeek-V2-Lite", "v2": "DeepSeek-V2 236B", "v3": "DeepSeek-V3 671B"}


def workload_name(workload, quant):
    return (f"{NAMES.get(workload, workload)}-shaped {quant} single-batch decode, {PROMPT_LEN}-token prompt + {GEN_TOKENS}-token "
            f"greedy completion")


# --dump-outputs: the e2e path returns GEN_TOKENS x vocab logits per completion; a fixed sample of vocabulary columns keeps the
# dump small (V3: 128 x 129280 fp32 would be 66 MB)
DUMP_VOCAB_SAMPLE = 8192


def measure(dsk, torch, dist, w, rank, world, local_rank, steps, warmup, want_e2e=True, profile=False, keep_outputs=False):
    """Mints the workload on this rank's GPU and times `steps` completions: returns a dict (rank-local; times are max over ranks).
    keep_outputs: also return what the last timed completion of each path handed back (res["outputs"], name -> array)."""
    m = mint_on_gpu(dsk, w, rank, world, local_rank)
    log(f"rank {rank}/{world}: minted {m.resident_bytes() / 1e9:.2f} GB resident, {m.active_bytes_per_token() / 1e9:.3f} GB/token algorithmic")
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.frombuffer(bytearray(dsk.Model.comm_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(uid, 0)
        m.comm_init(bytes(uid.cpu().numpy().tobytes()))
    vocab = w["vocab_size"]
    pr = prompt_ids(vocab)
    sharded_check = None
    if world > 1 and os.environ.get("DSK_CHECK_SHARDED", "1") == "1" and m.resident_bytes() * world < 60e9:
        # consistency of the expert-sharded path: same synthetic weights unsharded on rank 0, teacher-forced logits compared
        errs = []
        ref_m = mint_on_gpu(dsk, w, 0, 1, local_rank) if rank == 0 else None
        for p, t in enumerate(pr[:4]):
            lg, _ = m.forward(t, p)
            if rank == 0:
                lg = lg.copy()
                lr, _ = ref_m.forward(t, p)
                errs.append(float(np.linalg.norm(lg - lr) / np.linalg.norm(lr)))
        if rank == 0:
            sharded_check = {"rel_l2_vs_single_gpu": max(errs), "positions": len(errs)}
            ref_m.close()
            log(f"sharded vs single-GPU logits rel-L2 (max over {len(errs)} positions): {max(errs):.2e}")

    def hydrate():
        am = None
        for p, t in enumerate(pr):
            last = p + 1 == len(pr)
            _, am = m.forward(t, p, dsk.OUTPUT_LOGITS if last else dsk.HYDRATE_KV_CACHE, want_logits=False)
        return am

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    timeline = None
    if profile:   # every rank takes part (the forward is collective); rank 0 prints its CTA-0 timeline
        hydrate()
        m.profile_token(pr[0], PROMPT_LEN)
        timeline = m.profile_token(pr[1], PROMPT_LEN + 1)
        if rank == 0:
            print(timeline, file=sys.stderr, flush=True)

    # ---- value: device-resident decode, CUDA events inside dsk_decode_greedy (one persistent launch per completion) ----
    for _ in range(warmup):
        hydrate()
        m.decode_greedy(PROMPT_LEN, GEN_TOKENS)
    clocks = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    t_wall0 = time.perf_counter()
    dev_ms, toks = 0.0, None
    for _ in range(steps):
        hydrate()
        barrier()
        toks, ms = m.decode_greedy(PROMPT_LEN, GEN_TOKENS)
        dev_ms += ms
    barrier()
    wall = time.perf_counter() - t_wall0
    clk = clocks.stop() if clocks else None
    if dist is not None:
        t = torch.tensor([dev_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = steps * GEN_TOKENS / (dev_ms / 1e3)
    log(f"value {value:.1f} tok/s ({dev_ms / steps / GEN_TOKENS:.3f} ms/token)")

    # ---- e2e: reference-shaped host loop, host buffers, copies inside the timed region -------------
    e2e = None
    outputs = {"tokens": toks.astype(np.float64)} if keep_outputs else None
    if want_e2e:
        cols = np.sort(np.random.default_rng(0).choice(vocab, min(vocab, DUMP_VOCAB_SAMPLE), replace=False))

        def host_completion(keep=False):
            am = hydrate()
            t0 = time.perf_counter()
            pos = PROMPT_LEN
            kept_tokens, kept_logits = [], []
            for _ in range(GEN_TOKENS):
                logits, _ = m.forward(am, pos)            # H2D control words, D2H vocab logits, sync
                am = int(np.argmax(logits))               # host sampler (Sampler::sample_argmax)
                if keep:
                    kept_tokens.append(am)
                    kept_logits.append(logits[cols])
                pos += 1
            elapsed = time.perf_counter() - t0
            if keep:
                outputs.update(e2e_tokens=np.array(kept_tokens, np.float64), e2e_logits=np.stack(kept_logits),
                               e2e_logits_vocab_index=cols.astype(np.float64))
            return elapsed
        for _ in range(max(1, warmup // 2)):
            host_completion()
        barrier()
        e2e_s = sum(host_completion(keep=keep_outputs and i + 1 == steps) for i in range(steps))
        if dist is not None:
            t = torch.tensor([e2e_s], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        e2e = steps * GEN_TOKENS / e2e_s
        log(f"e2e {e2e:.1f} tok/s")
    res = {"value": value, "dev_ms": dev_ms, "wall": wall, "e2e": e2e, "clocks": clk, "sharded_check": sharded_check,
           "abytes": m.active_bytes_per_token(), "resident_gb": m.resident_bytes() / 1e9, "tokens": toks[:8].tolist(),
           "launches_per_forward": m.launches_per_forward(dsk.OUTPUT_LOGITS), "timeline": timeline, "outputs": outputs}
    m.close()
    torch.cuda.empty_cache()
    return res


def committed_traffic(workload, quant):
    """roofline.traffic: dram__bytes_read + dram__bytes_write of the decode kernel, per launch == per token, from the committed
    `ncu --set full` capture of this workload (profiles/r02_traffic.json).  A number taken under the profiler; it is reported
    only while the kernel sources still hash to what the capture ran (otherwise null: it would describe another build)."""
    try:
        import hashlib
        rec = json.load(open(os.path.join(REPO, "profiles", "r02_traffic.json")))
        h = hashlib.sha256()
        for f in ("dsk_mega.cuh", "dsk_kernels.cuh"):
            h.update(open(os.path.join(REPO, "deepseek.cpp_b200", "csrc", f), "rb").read())
        e = rec.get(f"{workload}/{quant}")
        if e and e.get("kernel_sources_sha256") == h.hexdigest():
            return float(e["dram_bytes_per_token"]), e.get("capture")
    except Exception:
        pass
    return None, None


def main():
    # stdout carries exactly ONE JSON line: libraries (NCCL banner, the reference's loader chatter) go to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DSK_WORKLOAD", "v2"))
    ap.add_argument("--quant", default=os.environ.get("DSK_QUANT", "q2_k"))
    ap.add_argument("--n-layers", type=int, default=int(os.environ.get("DSK_LAYERS", "0")))
    ap.add_argument("--mla", action="store_true", help="true-MLA blocks (convert.py --mla shapes: wc / wq_rope_b / wv_b, latent KV cache)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the V2-Lite configs[1]/[2] continuity numbers")
    ap.add_argument("--profile-token", action="store_true", help="print the per-stage timeline of one token to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed completion returned as DIR/<name>.npy: tokens (device loop), e2e_tokens and "
                         "e2e_logits (host loop, at the vocabulary columns in e2e_logits_vocab_index); inputs are seeded")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = workload_cfg(a.workload, a.quant, a.n_layers or None)
    if a.mla:
        w["use_mla"] = 1
    base = {"metric": "tok/s single-batch decode (128-tok gen)", "unit": "tok/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": DTYPES[a.quant],
            "data": "synthetic (random-init weights of the named architecture; no checkpoints offline)",
            "config": {"workload": workload_name(a.workload, a.quant) + (" (true-MLA blocks, use_mla=1)" if a.mla else ""), "baseline_config": {"v2lite": "configs[1]/[2]", "v2": "configs[3]", "v3": "configs[4]"}.get(a.workload),
                       "layers": w["n_layers"], "tokens_per_step": GEN_TOKENS,
                       "parallelism": (f"tensor parallel over {a.gpus} GPUs: attention heads, wo columns, shared-expert / dense-FFN hidden units, LM-head rows and routed experts sharded; two in-kernel peer-memory exchanges per layer" if os.environ.get("DSK_TP", "1") != "0" else f"routed experts sharded over {a.gpus} GPU(s), rest replicated; one in-kernel peer-memory exchange per MoE layer") if a.gpus > 1 else "1 GPU",
                       "l2": "weights streamed per token (GBs) exceed the 126 MB L2; no flush needed"}}

    if a.impl == "reference":
        if rank != 0:
            return 0
        try:
            t0 = time.time()
            tps, spent, desc = cpu_reference_leg(w, max(1, a.steps), max(1, a.warmup))
        except Exception as e:  # the oracle always exists in this tier; this only trips if _ref did not travel
            emit({"impl": "reference", "unavailable": str(e)[:200]})
            return 0
        out = dict(base)
        # a reference "step" is the bounded sample actually decoded (ms_per_step x steps = the CPU time really spent decoding);
        # `value` is its tok/s — measured on the full-depth model unless cpu_baseline.extrapolated says otherwise
        out.update({"impl": "reference", "value": tps, "ms_per_step": spent / max(1, a.steps) * 1e3, "n_gpus": a.gpus,
                    "step_note": "reference arm: one step = 1/steps of the bounded token sample described in cpu_baseline.sample",
                    "cpu_baseline": dict(desc, value=tps, unit="tok/s", seconds_decoding=spent, seconds_total=time.time() - t0),
                    "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    "gpu_launches": 0, "dtype": "reference CPU path (AVX2/F16C, OpenMP)"})
        emit(out)
        return 0

    import torch
    import dsk
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dsk.init(local_rank)
    log(f"rank {rank}/{world}: workload {a.workload}/{a.quant}")
    R = measure(dsk, torch, dist, w, rank, world, local_rank, a.steps, a.warmup, want_e2e=True, profile=a.profile_token,
                keep_outputs=bool(a.dump_outputs) and rank == 0)
    if R["outputs"]:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in R["outputs"].items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
        log(f"outputs of the last timed step written to {a.dump_outputs}: {sorted(R['outputs'])}")

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- roofline: whole-token algorithmic bytes vs measured HBM peak + the dominant stage kinds alone ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    abytes, value = R["abytes"], R["value"]
    achieved = abytes * value / 1e9 / a.gpus
    kern = {}
    try:
        hd = w["qk_nope_head_dim"] + w["qk_rope_head_dim"]
        shapes = {"lm_head": (w["vocab_size"], w["dim"]), "wo": (w["dim"], w["n_heads"] * w["v_head_dim"]),
                  "expert_w1": (w["moe_intermediate_size"], w["dim"])}
        if w["q_lora_rank"] > 0:
            shapes["wq_b"] = (w["n_heads"] * hd, w["q_lora_rank"])
        else:
            shapes["wq"] = (w["n_heads"] * hd, w["dim"])
        for label, (d_, n_) in shapes.items():
            n_mats = max(2, int(300e6 // (d_ * n_)) + 1)
            ms_k, b_k = dsk.bench_gemv(a.quant, d_, n_, n_mats=min(n_mats, 64), warmup=3, iters=20)
            kern[label] = {"rows": d_, "cols": n_, "us": ms_k * 1e3, "GB/s": b_k / (ms_k / 1e3) / 1e9, "frac": b_k / (ms_k / 1e3) / 1e9 / peak}
        kern["note"] = "ONE interpreter GEMV stage per launch (decode_kernel<Q>, production tile plan); launch overhead included"
    except Exception as e:
        kern = {"error": str(e)[:120]}
    traffic, capture = committed_traffic(a.workload, a.quant) if world == 1 and not a.n_layers and not a.mla else (None, None)
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_unit": "bytes per token (= per launch / tokens per launch), ncu capture in profiles/", "traffic_capture": capture,
            "kernel": "decode_kernel<Q> (a whole completion is one launch; achieved = algorithmic bytes/token x tok/s / N_gpus, i.e. every "
                      "barrier, staging phase and attention is charged to the GEMV stream)",
            "algorithmic_bytes_per_token": abytes, "peak_source": peak_src, "isolated_stages": kern}

    out = dict(base)
    vocab = w["vocab_size"]
    out.update({"value": value, "ms_per_step": R["dev_ms"] / a.steps, "wall_s": R["wall"],
                "e2e": {"value": R["e2e"], "unit": "tok/s", "h2d_bytes_per_step": GEN_TOKENS * 48, "d2h_bytes_per_step": GEN_TOKENS * vocab * 4},
                "gpu_launches": a.steps * R["launches_per_forward"],
                "gpu_launches_note": "decode_kernel launches inside the timed region of `value`: one persistent cooperative launch per 128-token "
                                     "completion (the e2e region launches it once per token: steps x 128)",
                "roofline": roof, "clocks": R["clocks"], "sharded_check": R["sharded_check"], "resident_gb": R["resident_gb"],
                "sample_tokens": R["tokens"]})
    # ---- secondary: the V2-Lite configs of BASELINE.json (round-1 headline), same run, N = 1 only ---------------------
    if world == 1 and not a.no_secondary and a.workload != "v2lite" and not a.n_layers:
        sec = {}
        for sq in ("f8e5m2", "q2_k"):
            try:
                ws = workload_cfg("v2lite", sq)
                r2 = measure(dsk, torch, None, ws, 0, 1, local_rank, max(2, a.steps // 2), max(3, a.warmup), want_e2e=True)
                sec[f"v2lite/{sq}"] = {"workload": workload_name("v2lite", sq), "value": r2["value"], "e2e": r2["e2e"], "unit": "tok/s",
                                       "algorithmic_bytes_per_token": r2["abytes"], "roofline_frac": r2["abytes"] * r2["value"] / 1e9 / peak}
            except Exception as e:
                sec[f"v2lite/{sq}"] = {"error": str(e)[:160]}
        if a.workload == "v2" and not a.mla:   # the same model converted with --mla (BlockMLA): absorbed projections, latent KV cache
            try:
                wm = dict(w, use_mla=1)
                r3 = measure(dsk, torch, None, wm, 0, 1, local_rank, max(2, a.steps // 2), max(3, a.warmup), want_e2e=False)
                sec[f"v2/{a.quant}+mla"] = {"workload": workload_name("v2", a.quant) + " (true-MLA blocks, use_mla=1)", "value": r3["value"],
                                            "unit": "tok/s", "algorithmic_bytes_per_token": r3["abytes"],
                                            "roofline_frac": r3["abytes"] * r3["value"] / 1e9 / peak, "resident_gb": r3["resident_gb"]}
            except Exception as e:
                sec[f"v2/{a.quant}+mla"] = {"error": str(e)[:160]}
        out["secondary"] = sec
    if a.gpus == 1 and not a.no_cpu_baseline:
        try:
            tps, spent, desc = cpu_reference_leg(w, 1, 1, tokens_per_step=4)
            out["cpu_baseline"] = dict(desc, value=tps, unit="tok/s", seconds_decoding=spent)
        except Exception as e:
            out["cpu_baseline"] = {"value": None, "unit": "tok/s", "cores": 0, "kind": "reference", "sample": f"failed: {str(e)[:150]}"}
    emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
