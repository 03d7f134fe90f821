#!/usr/bin/env python
"""bench.py -- decode tokens/s of a synthetic Llama-3-8B "v8-k65536-256" VPTQ stack on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One step = one decode token (batch 1) through every VPTQ-quantized linear of Llama-3-8B:
32 layers x (q 4096x4096, k/v 1024x4096, o 4096x4096, gate/up 14336x4096, down 4096x14336),
vector_len 8, 65536 centroids + 256 residual centroids (b = 24 index bits per 8 weights),
perm + norm enabled -- 224 fused GEMV launches chained by true data dependence
(h -> q,k,v ; q -> o ; o -> gate,up ; gate -> down -> next layer).  Attention, norms, the
fp16 embedding and lm_head are NOT on the VPTQ path and are not executed (stated in `config`).
Weights are synthetic (uniform random packed indices, random codebooks); 2.6 GB of indices per
token stream from HBM every step, ~20x the L2.

Printed JSON (one line, rank 0): the driver contract + `roofline`, `cpu_baseline`, `e2e`, `clocks`.
  value     tokens/s, inputs resident in HBM, one CUDA graph of the 224 launches per step
  e2e       tokens/s through the C ABI with HOST buffers: pinned x -> H2D -> 224 GEMVs -> D2H -> sync
  roofline  HBM: algorithmic bytes (packed indices + x + y of every launch) / step time
  N > 1     tensor-parallel over out_features; exchange fused into the GEMV over NVLink peer memory (tagged words;
            --tp-mode nccl: one NCCL all-reduce per launch, the north_star form), strong scaling; `tp_check`
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LLAMA3_8B = dict(name="llama3-8b", layers=32, hidden=4096, kv=1024, ffn=14336)
QUANT = dict(vector_len=8, num_centroids=65536, num_res_centroids=256)
METRIC = "decode tokens/sec Llama-3-8B 2-bit (VPTQ v8-k65536-256, b=24 index bits / 8 weights), batch 1"
# BASELINE.json configs[3]: Llama-3-70B, true 2-bit variant (K = 65536, no residual codebook: b = 16)
LLAMA3_70B = dict(name="llama3-70b", layers=80, hidden=8192, kv=1024, ffn=28672)
QUANT_70B = dict(vector_len=8, num_centroids=65536, num_res_centroids=-1)
MODELS = {"llama3-8b": (LLAMA3_8B, QUANT, METRIC, "BASELINE.json configs[1]"),
          "llama3-70b": (LLAMA3_70B, QUANT_70B,
                         "decode tokens/sec Llama-3-70B 2-bit (VPTQ v8-k65536-0, b=16 index bits / 8 weights), batch 1",
                         "BASELINE.json configs[3]")}


def model_linears(m):
    h, kv, f = m["hidden"], m["kv"], m["ffn"]
    # (name, in, out, input_of)
    return [("q", h, h), ("k", h, kv), ("v", h, kv), ("o", h, h), ("gate", h, f), ("up", h, f), ("down", f, h)]


def workload_string(m, q, cfg_name):
    Kr = q["num_res_centroids"]
    b = (q["num_centroids"].bit_length() - 1) + (Kr.bit_length() - 1 if Kr > 0 else 0)
    return (f"{cfg_name}: {m['name']} decode batch=1 seq=1, all {7 * m['layers']} VPTQ linears ({m['layers']} layers x "
            f"q,k,v,o,gate,up,down), v=8 K={q['num_centroids']} Kr={max(Kr, 0)} (b={b}), perm+norm on; "
            "attention/norm/lm_head not on the VPTQ path and not executed")


def algorithmic_bytes(m, q, tokens=1, world=1):
    """SURVEY.md 8(d): packed index bytes + x bytes + y bytes per GEMV launch, summed over a step."""
    b = (q["num_centroids"].bit_length() - 1) + max(q["num_res_centroids"].bit_length() - 1, 0)
    tot = 0
    for _, i, o in model_linears(m):
        ro = (o // world + q["vector_len"] - 1) // q["vector_len"]
        tot += ro * ((i * b + 31) // 32) * 4 + tokens * i * 2 + tokens * (o // world) * 2
    return tot * m["layers"]


# ------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def layer_tensors(m, q, li, name, i, o, device, dtype, rows=None):
    """Synthetic tensors of linear `name` of decoder layer `li`: a function of (li, name) only, so every rank
    (and the unsharded correctness check) sees the same layer; `rows` = (r0, r1) keeps that slice of the
    index rows (tensor parallelism shards out_features, tp.shard_bounds)."""
    import torch
    v, K, Kr = q["vector_len"], q["num_centroids"], q["num_res_centroids"]
    ib, rb = K.bit_length() - 1, max(Kr.bit_length() - 1, 0)
    ro, wd = o // v, (i * (ib + rb) + 31) // 32
    g = torch.Generator(device=device).manual_seed(1234 + 16 * li + [n for n, _, _ in model_linears(m)].index(name))
    t = dict(
        indices=torch.randint(-2 ** 31, 2 ** 31 - 1, (1, ro, wd), device=device, dtype=torch.int32, generator=g),
        # std 1/sqrt(in): unit gain, so activations stay O(1) through the chained layers
        centroids=(torch.randn(1, K * v, device=device, generator=g) / i ** 0.5).to(dtype),
        res_centroids=(0.25 * torch.randn(1, Kr * v, device=device, generator=g) / i ** 0.5).to(dtype) if Kr > 0 else None,
        # uint16 payload behind an int16 view: int64 -> int16 narrowing keeps the low 16 bits
        perm=torch.randperm(i, device=device, generator=g).to(torch.int16),
        weight_scale=(1 + 0.1 * torch.randn(i, device=device, generator=g)).to(dtype),
        weight_bias=(0.01 * torch.randn(i, device=device, generator=g) / i ** 0.5).to(dtype))
    if rows is not None:
        t["indices"] = t["indices"][:, rows[0]:rows[1], :].contiguous()
    return t


def make_layer_desc(q, t, i, o_loc, dtype, lists=None):
    from vptq_b200 import native
    return native.make_desc(
        dtype=dtype, in_features=i, out_features=o_loc, vector_len=q["vector_len"], num_centroids=q["num_centroids"],
        num_res_centroids=q["num_res_centroids"], num_codebooks=1, group_size=i, outlier_size=0, outlier_vector_len=-1,
        num_outlier_centroids=-1, indices=t["indices"], centroids=t["centroids"], res_centroids=t["res_centroids"],
        outlier_indices=None, outlier_centroids=None, perm=t["perm"], weight_scale=t["weight_scale"],
        weight_bias=t["weight_bias"], bias=None, lists=lists)


def make_module(q, t, i, o_loc, dtype, device):
    """The drop-in module (vptq_b200.VQuantLinear, reference constructor signature) holding these tensors."""
    import torch
    from vptq_b200 import VQuantLinear
    Kr = q["num_res_centroids"]
    mod = VQuantLinear(i, o_loc, vector_lens=[-1, q["vector_len"]], num_centroids=[-1, q["num_centroids"]],
                       num_res_centroids=[-1, Kr], group_num=1, group_size=i, outlier_size=0, indices_as_float=False,
                       enable_norm=True, enable_perm=True, is_indice_packed=True, bias=False, device=device, dtype=dtype,
                       enable_proxy_error=False)
    with torch.no_grad():
        mod.indices.data = t["indices"]
        mod.centroids.weight.data = t["centroids"]
        if Kr > 0:
            mod.res_centroids.weight.data = t["res_centroids"]
        mod.perm.data = t["perm"]
        mod.weight_scale.data, mod.weight_bias.data = t["weight_scale"], t["weight_bias"]
    return mod.eval().prepare(dtype)


def build_stack(m, q, device, rank, world, dtype):
    """This rank's out_features shard of every linear, as VQuantLinear modules; the C-ABI legs of the bench use the
    descriptors those modules built (one copy of the weights and of the load-time index lists)."""
    v = q["vector_len"]
    stack = []
    for li in range(m["layers"]):
        layer = {}
        for name, i, o in model_linears(m):
            o_loc = o // world
            t = layer_tensors(m, q, li, name, i, o, device, dtype, rows=(rank * o_loc // v, (rank + 1) * o_loc // v))
            t["module"] = make_module(q, t, i, o_loc, dtype, device)
            t["desc"] = t["module"]._desc_cache[0]
            t["in"], t["out"], t["out_loc"] = i, o, o_loc
            layer[name] = t
        stack.append(layer)
    return stack


def module_level(m, stack, device, dtype, x_host, steps, warmup, lm_head_rows=128256):
    """The same token through the MODULE API a Hugging Face model calls (VQuantLinear.forward per projection, in
    HF's order), three ways: eager and unfused (what a stock integration does), vptq_b200.fuse(model) + one CUDA
    graph per token + PDL, and the latter followed by the fp16 lm_head GEMV (cuBLAS through torch: not a VPTQ
    layer, SURVEY.md 8d) -- per-step H2D of x and D2H of the result inside the timed region."""
    import torch
    import torch.nn as nn
    import vptq_b200

    class Layer(nn.Module):
        def __init__(self, d):
            super().__init__()
            for n in ("q", "k", "v", "o", "gate", "up", "down"):
                setattr(self, n + "_proj", d[n]["module"])

        def forward(self, x):
            q, k, v = self.q_proj(x), self.k_proj(x), self.v_proj(x)      # (attention itself is not a VPTQ layer)
            o = self.o_proj(q)
            g, u = self.gate_proj(o), self.up_proj(o)
            return self.down_proj(g)

    model = nn.Sequential(*[Layer(d) for d in stack])
    x_dev = torch.zeros(1, m["hidden"], device=device, dtype=dtype)
    s = torch.cuda.Stream(device)
    s.wait_stream(torch.cuda.current_stream())
    out = {}

    def timed(fn, result, n_steps, n_warm):
        fn()
        s.synchronize()
        host = torch.empty_like(result(), device="cpu").pin_memory()
        def one():
            x_dev.copy_(x_host, non_blocking=True)
            fn()
            host.copy_(result(), non_blocking=True)
            s.synchronize()
        for _ in range(n_warm):
            one()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(n_steps):
            one()
        e1.record(s)
        s.synchronize()
        return 1e3 / (e0.elapsed_time(e1) / n_steps)

    with torch.cuda.stream(s), torch.no_grad():
        holder = {}
        def eager():
            holder["y"] = model(x_dev)
        out["eager_unfused_tokens_per_s"] = round(timed(eager, lambda: holder["y"], max(3, steps // 4), 2), 2)
        vptq_b200.fuse(model, pdl=True, prepare=False)
        model(x_dev); s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            y_graph = model(x_dev)
        out["fused_graph_tokens_per_s"] = round(timed(g.replay, lambda: y_graph, steps, max(warmup, 3)), 2)
        # + the fp16 lm_head (vocabulary 128256): 1.05 GB more per token, read by cuBLAS
        w_head = torch.randn(lm_head_rows, m["hidden"], device=device, dtype=dtype) * 0.02
        torch.matmul(y_graph, w_head.t()); s.synchronize()
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2, stream=s):
            logits = torch.matmul(model(x_dev), w_head.t())
        out["fused_graph_plus_lm_head_tokens_per_s"] = round(timed(g2.replay, lambda: logits, steps, max(warmup, 3)), 2)
        vptq_b200.unfuse(model)
    out["how"] = ("VQuantLinear.forward per projection in HF order (q,k,v,o,gate,up,down), host x -> H2D -> layers -> D2H "
                  "every step; eager_unfused = 7 eager module calls per layer; fused_graph = vptq_b200.fuse(model) + "
                  "CUDA graph + PDL; lm_head = fp16 128256 x hidden GEMV through torch (cuBLAS)")
    return out




def reference_hidden(m, q, device, dtype, x_in, lists=None):
    """The same token through the UNSHARDED layers on this GPU alone (one decoder layer resident at a time):
    what the tensor-parallel exchange must reproduce.  Same kernels, same chain as make_step."""
    import torch
    from vptq_b200 import native
    h, kv, f = m["hidden"], m["kv"], m["ffn"]
    x = x_in.clone()
    for li in range(m["layers"]):
        out = {}
        src = {"q": "x", "k": "x", "v": "x", "o": "q", "gate": "o", "up": "o", "down": "gate"}
        out["x"] = x
        for name, i, o in model_linears(m):
            t = layer_tensors(m, q, li, name, i, o, device, dtype)
            d = make_layer_desc(q, t, i, o, dtype, lists=lists)
            y = torch.empty(1, o, device=device, dtype=dtype)
            native.quant_gemv(d, out[src[name]], y)
            torch.cuda.synchronize()
            out[name] = y
            del d, t
        x = out["down"]
    return x


def make_step(m, stack, device, dtype, rank, world, flags, tp_mode="nccl"):
    """Returns (x_in, step, launches); step() enqueues one decode token on the current stream."""
    import torch
    import torch.distributed as dist
    from vptq_b200 import native
    h, kv, f = m["hidden"], m["kv"], m["ffn"]
    p2p = world > 1 and tp_mode in ("p2p", "p2p-plain")
    tagged = p2p and tp_mode != "p2p-plain"
    if p2p:
        # activations live in a symmetric arena mapped into every rank: the GEMV stores its slice into all peers'
        # buffers (no NCCL on the path).  Default wire format: tagged 8-byte words {2 values, tag} that the
        # consumer re-reads until the tag is current (no fence, no flag); "p2p-plain": plain values + epoch flags
        from vptq_b200 import tp
        nslots = 4 * len(stack)
        wb = 4 if tagged else 2   # bytes per output in the exchanged buffers
        arena = tp.PeerArena((h + 2 * kv + h + 2 * f + 2 * h) * wb + nslots * world * 4 + 8192, device)
        bdt, mul = (torch.uint8, wb) if tagged else (dtype, 1)
        qkv_x, off_qkv = arena.alloc((1, (h + 2 * kv) * mul), bdt)
        o_x, off_o = arena.alloc((1, h * mul), bdt)
        gu_x, off_gu = arena.alloc((1, 2 * f * mul), bdt)
        hs0_x, off_h0 = arena.alloc((1, h * mul), bdt)
        hs1_x, off_h1 = arena.alloc((1, h * mul), bdt)
        _, off_flags = arena.alloc((nslots, world), torch.int32)
        tp_epoch = torch.zeros(nslots, dtype=torch.int32, device=device)
        tp_done = torch.zeros(nslots, dtype=torch.int32, device=device)
        tp_error = torch.zeros(1, dtype=torch.int32, device=device)
        if tagged:   # the kernels also leave the plain local slice in ordinary full-width buffers
            qkv = torch.zeros(1, h + 2 * kv, device=device, dtype=dtype)
            gu = torch.zeros(1, 2 * f, device=device, dtype=dtype)
            o_buf = torch.zeros(1, h, device=device, dtype=dtype)
            hs0, hs1 = (torch.zeros(1, h, device=device, dtype=dtype) for _ in range(2))
        else:
            qkv, o_buf, gu, hs0, hs1 = qkv_x, o_x, gu_x, hs0_x, hs1_x
    else:
        # q|k|v and gate|up live side by side so that one memset + one all-reduce serve a fused launch
        qkv = torch.zeros(1, h + 2 * kv, device=device, dtype=dtype)
        gu = torch.zeros(1, 2 * f, device=device, dtype=dtype)
        o_buf = torch.zeros(1, h, device=device, dtype=dtype)
        hs0, hs1 = (torch.zeros(1, h, device=device, dtype=dtype) for _ in range(2))
    buf = {"q": qkv[:, :h], "k": qkv[:, h:h + kv], "v": qkv[:, h + kv:], "gate": gu[:, :f], "up": gu[:, f:], "o": o_buf}
    # x_in is read-only (so that replaying the graph repeats the same token); hidden states ping-pong
    x_in = torch.zeros(1, h, device=device, dtype=dtype)
    hs = [hs0, hs1]
    launches = [0]
    debug_sync = bool(os.environ.get("BENCH_DEBUG"))

    def own(t, y):
        """this rank's slice of a full-width output"""
        return y if world == 1 else y[:, rank * t["out_loc"]:(rank + 1) * t["out_loc"]]

    def linear(t, x, y):
        if world == 1:
            native.quant_gemv(t["desc"], x, y, flags=flags)
            if debug_sync and not torch.cuda.is_current_stream_capturing():
                torch.cuda.current_stream().synchronize()
        else:
            # this rank owns rows [rank*o_loc, (rank+1)*o_loc); y is full width and zero elsewhere,
            # one all-reduce(sum) over NVLink per layer completes it (north_star)
            y.zero_()
            native.quant_gemv(t["desc"], x, own(t, y), flags=0)
            dist.all_reduce(y)
        launches[0] += 1

    fuse = not os.environ.get("BENCH_NO_FUSE")
    fused = []
    if fuse and not p2p:   # horizontal fusion of the linears that share an input: 7 -> 4 launches per layer
        for layer in stack:
            fused.append((native.FusedGemv([layer[n]["desc"] for n in ("q", "k", "v")],
                                           [own(layer[n], buf[n]) for n in ("q", "k", "v")]),
                          native.FusedGemv([layer[n]["desc"] for n in ("gate", "up")],
                                           [own(layer[n], buf[n]) for n in ("gate", "up")])))

    def fused_linear(fn, x, full):
        if world == 1:
            fn(x, flags)
        else:   # one memset + one launch + ONE all-reduce for the whole group
            full.zero_()
            fn(x, 0)
            dist.all_reduce(full)
        launches[0] += 1

    p2p_launch = []
    if p2p:
        e2 = wb  # bytes per output in the exchanged buffers
        hs_off = [off_h0, off_h1]
        hs_x = [hs0_x, hs1_x]
        for li, layer in enumerate(stack):
            cur = li % 2

            def ex(slot_in_layer, wait, y_offsets, names, layer=layer, li=li):
                return tp.make_exchange(arena, slot=4 * li + slot_in_layer, wait_slot=wait, y_offsets=y_offsets,
                                        slice_bytes=[rank * layer[n]["out_loc"] * e2 for n in names],
                                        flags_offset=off_flags, epoch=tp_epoch, done=tp_done, error=tp_error,
                                        fmt=native.TP_TAGGED if tagged else native.TP_PLAIN, num_slots=nslots)

            def fz(names, ys_full, exch, layer=layer):
                return native.FusedGemvTP([layer[n]["desc"] for n in names],
                                          [own(layer[n], y) for n, y in zip(names, ys_full)], exch)

            wait_x = -1 if li == 0 else 4 * (li - 1) + 3
            p2p_launch.append((
                fz(("q", "k", "v"), (buf["q"], buf["k"], buf["v"]),
                   ex(0, wait_x, [off_qkv, off_qkv + h * e2, off_qkv + (h + kv) * e2], ("q", "k", "v"))),
                fz(("o",), (buf["o"],), ex(1, 4 * li, [off_o], ("o",))),
                fz(("gate", "up"), (buf["gate"], buf["up"]), ex(2, 4 * li + 1, [off_gu, off_gu + f * e2], ("gate", "up"))),
                fz(("down",), (hs[cur],), ex(3, 4 * li + 2, [hs_off[cur]], ("down",)))))

    h_plain = torch.zeros(1, h, device=device, dtype=dtype) if tagged else None

    def step():
        launches[0] = 0
        x, cur = x_in, 0
        if p2p:
            # (tagged: a consumer's x is its local tagged buffer; the q / gate part starts at offset 0 of qkv / gu)
            xq, xo, xg = (qkv_x, o_x, gu_x) if tagged else (buf["q"], buf["o"], buf["gate"])
            for f_qkv, f_o, f_gu, f_down in p2p_launch:
                f_qkv(x, flags)
                f_o(xq, flags)
                f_gu(xo, flags)
                f_down(xg, flags)
                launches[0] += 4
                x, cur = (hs_x[cur] if tagged else hs[cur]), 1 - cur
            if tagged:   # the last hidden state, every rank's slice (waits for their tags), as plain 16-bit values
                native.tp_untag(x, h_plain, p2p_launch[-1][3].ex)
                return h_plain
            return x
        for li, layer in enumerate(stack):
            if fuse:
                fused_linear(fused[li][0], x, qkv)
                linear(layer["o"], buf["q"], buf["o"])
                fused_linear(fused[li][1], buf["o"], gu)
            else:
                linear(layer["q"], x, buf["q"])
                linear(layer["k"], x, buf["k"])
                linear(layer["v"], x, buf["v"])
                linear(layer["o"], buf["q"], buf["o"])
                linear(layer["gate"], buf["o"], buf["gate"])
                linear(layer["up"], buf["o"], buf["up"])
            linear(layer["down"], buf["gate"], hs[cur])
            x, cur = hs[cur], 1 - cur
        return x

    step.tp_error = tp_error if p2p else None
    step.last_layer = buf      # after a step: the last decoder layer's projections (q, k, v, o, gate, up)
    return x_in, step, launches


def _log(msg):
    if os.environ.get("BENCH_VERBOSE"):
        print(f"[bench r{os.environ.get('RANK', '0')} {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def dump_outputs(out_dir, hidden, last_layer):
    """What the last timed step computed, as float32 .npy files: the hidden state the step returns and, on one GPU,
    the last layer's projections (k, v and up feed nothing downstream, so the hidden state alone would not show them).
    The weights and the token are seeded, so two builds can be compared file for file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"hidden": hidden, **{f"last_layer_{n}": t for n, t in last_layer.items()}}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import faulthandler
    import torch
    import torch.distributed as dist
    from vptq_b200 import native
    faulthandler.dump_traceback_later(int(os.environ.get("BENCH_WATCHDOG_S", "900")), exit=True)  # a hang leaves a trace

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _log("process group up")
    native.lib()
    dtype = torch.float16
    m, q, metric, cfg_name = MODELS[args.model]
    m = dict(m)
    if args.debug_layers:
        m["layers"] = args.debug_layers
    flags = 0 if args.no_pdl else native.FLAG_PDL

    stack = build_stack(m, q, device, rank, world, dtype)
    _log("weights built")
    tp_mode = args.tp_mode if world > 1 else "none"
    torch.manual_seed(4321)
    x_host = torch.randn(1, m["hidden"]).to(dtype).pin_memory()
    tp_fallback = None
    if tp_mode in ("p2p", "p2p-plain"):
        # peer-mapped activations need symmetric memory, and the fused exchange must get through one eager
        # token without a refused launch or a flag time-out; every rank must take the same decision
        ok = torch.ones(1, device=device)
        try:
            x_in, step, launches = make_step(m, stack, device, dtype, rank, world, flags, tp_mode)
            x_in.copy_(x_host, non_blocking=True)
            step()
            torch.cuda.synchronize()
            if int(step.tp_error.item()) != 0:
                raise RuntimeError("a tensor-parallel flag wait timed out")
        except Exception as e:  # noqa: BLE001
            _log(f"p2p exchange unavailable ({e!r}); falling back to NCCL all-reduce")
            tp_fallback = repr(e)[:200]
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok.item()) == 0.0:
            tp_mode, tp_fallback = "nccl", tp_fallback or "another rank could not set up the fused exchange"
            torch.cuda.synchronize()
    if tp_mode not in ("p2p", "p2p-plain"):
        x_in, step, launches = make_step(m, stack, device, dtype, rank, world, flags, tp_mode)
    y_host = torch.empty(1, m["hidden"], dtype=dtype).pin_memory()

    s = torch.cuda.Stream(device)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x_in.copy_(x_host, non_blocking=True)
        for _ in range(2):                      # eager warm-up: smem attributes, workspace, NCCL channels
            h_out = step()
        s.synchronize()
        _log("eager warm-up done")
        use_graph = not args.tp_eager or world == 1
        if use_graph:
            graph = torch.cuda.CUDAGraph()
            # thread_local: the NCCL watchdog thread may touch CUDA while this thread captures
            with torch.cuda.graph(graph, stream=s, capture_error_mode="thread_local"):
                h_out = step()
            replay = graph.replay
        else:
            def replay():
                nonlocal h_out
                h_out = step()
        n_launch = launches[0]
        _log("graph captured" if use_graph else "eager mode")

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        # ---- `value`: device-resident, W warm-up + K timed graph replays -------------------------
        for _ in range(max(args.warmup, 3)):
            replay()
        barrier()
        _log("warm-up replays done")
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        barrier()
        ev[0].record(s)
        for _ in range(args.steps):
            replay()
        ev[1].record(s)
        barrier()
        ms = ev[0].elapsed_time(ev[1])
        clk = clocks.stop() if rank == 0 else None
        assert torch.isfinite(h_out.float()).all(), "activations overflowed"
        tp_err = int(step.tp_error.item()) if step.tp_error is not None else 0
        if world > 1:
            te = torch.tensor([tp_err], device=device)
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            tp_err = int(te.item())
        assert tp_err == 0, "a tensor-parallel flag wait timed out"
        h_final = h_out.clone()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, h_out, step.last_layer if world == 1 else {})

        # ---- `e2e`: host buffers, H2D + D2H inside the timed region, per-step sync ------------------
        e2e_steps = args.steps
        for _ in range(3):
            x_in.copy_(x_host, non_blocking=True); replay(); y_host.copy_(h_out, non_blocking=True); s.synchronize()
        barrier()
        ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        t0 = time.perf_counter()
        ev2[0].record(s)
        for _ in range(e2e_steps):
            x_in.copy_(x_host, non_blocking=True)
            replay()
            y_host.copy_(h_out, non_blocking=True)
            s.synchronize()
        ev2[1].record(s)
        barrier()
        ms_e2e = ev2[0].elapsed_time(ev2[1])
        wall_e2e = (time.perf_counter() - t0) * 1e3
    _log("timed regions done")

    if world > 1:
        tms = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms, ms_e2e = tms.tolist()

    # ---- correctness of the measured computation: the same token through the unsharded layers on rank 0
    # alone (N > 1: checks the tensor-parallel exchange; N = 1: the list kernel against the generic one) ----
    lists_on = os.environ.get("VPTQ_B200_LISTS", native.LISTS_DEFAULT) != "0" and \
        "lists=0" not in os.environ.get("VPTQ_B200_GEMV_TUNE", "")
    check = None
    if rank == 0 and not args.no_check:
        with torch.cuda.stream(s):
            x_chk = torch.empty(1, m["hidden"], device=device, dtype=dtype)
            x_chk.copy_(x_host)
            # the reference runs the OTHER decode kernel (generic when the measured path used the lists and vice
            # versa): an independent implementation, and no list building for the unsharded layers
            h_ref = reference_hidden(m, q, device, dtype, x_chk, lists=not lists_on).float()
            s.synchronize()
        err = float((h_final.float() - h_ref).abs().max() / h_ref.abs().max())
        # 4 * layers chained 16-bit roundings: the bar is loose, a wrong or stale slice misses it by orders of magnitude
        check = {"max_rel_err": round(err, 6), "ok": bool(err <= 2e-2), "against":
                 ("unsharded layers on rank 0, " if world > 1 else "") + "the other decode kernel (generic <-> lists), same token"}
    if world > 1:
        dist.barrier()

    if rank == 0:
        ms_step = ms / args.steps
        value = 1e3 / ms_step
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        abytes = algorithmic_bytes(m, q, 1, world)         # per rank and step
        achieved = abytes / (ms_step * 1e-3) / 1e9
        traffic = None
        uses_lists = lists_on
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "gemv_traffic.json")))
            traffic = (tj["lists"] if uses_lists else tj)["dram_bytes_per_token"] // (n_launch * world)
        except Exception:
            pass
        line = {
            "metric": metric, "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": workload_string(m, q, cfg_name),
                       "parallelism": (f"tp{world} (out_features sharded; " +
                                       ("exchange fused into the GEMV: tagged 8-byte words stored into every peer over NVLink, "
                                        "no fence / flag / NCCL call" if tp_mode == "p2p" else
                                        "exchange fused into the GEMV: NVLink peer stores + epoch flags, no NCCL call"
                                        if tp_mode.startswith("p2p") else "1 NCCL all-reduce per launch: q|k|v, o, gate|up, down") + ")")
                                      if world > 1 else "single GPU",
                       "l2_policy": "inputs larger than L2: 2.6 GB of distinct packed indices streamed per step",
                       "index_lists": ("slice x tile lists, entries re-ordered at load time for shared-memory banks "
                                       "(vptq_b200_lists_deal_host)" if os.environ.get("VPTQ_B200_LISTS_DEAL", "1") not in ("0", "off", "")
                                       else "slice x tile lists, round-robin order") if uses_lists else "none (generic kernel)",
                       "fusion": "q+k+v and gate+up each in one launch (vptq_b200_quant_gemv_multi)" if
                                 not os.environ.get("BENCH_NO_FUSE") else "one launch per linear",
                       "launch": ("one CUDA graph per token" if use_graph else "eager launches") +
                                 ", PDL " + ("off" if (args.no_pdl or (world > 1 and not tp_mode.startswith("p2p"))) else "on")},
            "gpu_launches": n_launch * args.steps,
            "e2e": {"value": round(1e3 / (ms_e2e / e2e_steps), 2), "unit": "tokens/s",
                    "h2d_bytes_per_step": x_host.numel() * 2, "d2h_bytes_per_step": y_host.numel() * 2,
                    "wall_ms_per_step": round(wall_e2e / e2e_steps, 4)},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic,
                         "traffic_source": "ncu dram__bytes_read+write per launch, profiles/gemv_traffic.json (one --set full "
                                           "capture per shape, profiles/r02_ncu_shapes_metrics.csv); not measured in this run",
                         "kernel": ("gemv_lists_kernel<half,true> (csrc/gemv_lists.cu: 64 KiB codebook slices in shared "
                                    "memory, slice x tile index lists)") if uses_lists else
                                   "gemv_body<half,8,1,false,true> (entry points gemv_kernel / gemv_multi_kernel)",
                         "algorithmic_bytes_per_launch": abytes // n_launch,
                         "avg_launch_us": round(ms_step * 1e3 / n_launch, 3),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)"},
            "clocks": clk,
        }
        # resident bytes of this rank's weights: checkpoint tensors + load-time index lists of the decode kernel
        mem = {"packed_index_bytes": 0, "list_bytes": 0, "codebook_bytes": 0}
        for layer in stack:
            for t in layer.values():
                mem["packed_index_bytes"] += t["indices"].numel() * 4
                mem["codebook_bytes"] += t["centroids"].numel() * 2 + (t["res_centroids"].numel() * 2 if t["res_centroids"] is not None else 0)
                mem["list_bytes"] += sum(k.numel() * k.element_size() for k in getattr(t["desc"], "_keep", ())
                                         if k.dtype == torch.int32)
        mem["lists_over_packed"] = round(mem["list_bytes"] / max(mem["packed_index_bytes"], 1), 3)
        line["resident_bytes"] = mem
        if world > 1:
            line["tp_check"] = check
            line["config"]["tp_mode"] = tp_mode
            if tp_fallback:
                line["config"]["tp_fallback_reason"] = tp_fallback
        else:
            line["check"] = check
        if world == 1 and not args.no_module_level:
            try:
                line["module_api"] = module_level(m, stack, device, dtype, x_host, args.steps, args.warmup)
            except Exception as e:  # noqa: BLE001
                line["module_api"] = {"error": repr(e)[:300]}
        if world == 1 and not args.no_prefill:
            try:
                line["prefill"] = prefill_timing(m, q, stack, device, dtype)
            except Exception as e:  # noqa: BLE001
                line["prefill"] = {"error": repr(e)[:300]}
        if world == 1 and not args.no_ref_cuda:
            try:
                line["ref_cuda"] = ref_cuda_timing(m, q, device, dtype)
            except Exception as e:  # noqa: BLE001
                line["ref_cuda"] = {"unavailable": repr(e)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(m, q, budget_s=args.cpu_budget)
        print(json.dumps(line), flush=True)
    faulthandler.cancel_dump_traceback_later()
    if world > 1:
        # tearing down a process group whose collectives live in a captured CUDA graph can block
        # forever; every rank has its result out, so leave without the destructor chain
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's pure-torch path (ported, see oracle/torch_port.py) on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_threads():
    """All the host threads this process may use: torchrun pins OMP_NUM_THREADS=1, which would make the CPU arm
    look 60x slower than the box really is -- undo it (rank 0 is the only rank that runs the CPU arm)."""
    import torch
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # one thread per physical core: with all 128 hyper-threads of the GPU box the gather / GEMV mix of this path ran
    # 4x SLOWER than with 64 (measured, round 2), so that would understate the CPU
    n = n // 2 if n > 16 else n
    try:
        torch.set_num_threads(max(1, n))
    except Exception:
        pass
    return torch.get_num_threads()


_CPU_LAYERS = {}


def cpu_baseline(m, q, budget_s=20.0, min_reps=1):
    """Bounded sample: ONE decoder layer's seven VPTQ linears (q,k,v,o,gate,up,down at their real shapes) of the
    same workload, batch 1 = 1/layers of a token, through the reference's pure-torch path (oracle/torch_port.py)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch_port as tp
    threads = _cpu_threads()
    key = (m["name"], q["num_centroids"], q["num_res_centroids"])
    if key not in _CPU_LAYERS:
        _CPU_LAYERS[key] = [(tp.synthetic_layer(i, o, q["vector_len"], q["num_centroids"], q["num_res_centroids"], seed=k),
                             torch.randn(1, i).to(torch.float16)) for k, (_, i, o) in enumerate(model_linears(m))]
    layers = _CPU_LAYERS[key]
    times, t_start = [], time.perf_counter()
    while len(times) < min_reps or (time.perf_counter() - t_start < budget_s and len(times) < 50):
        t0 = time.perf_counter()
        for L, x in layers:
            tp.quant_gemm(x, L)
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    tok_s = 1.0 / (t * m["layers"])
    return {"value": round(tok_s, 5), "unit": "tokens/s", "cores": threads, "kind": "port", "host_cpus": os.cpu_count(),
            "sample": f"one decoder layer of {m['name']} (its 7 VPTQ linears at full size = 1/{m['layers']} of a token), "
                      f"median of {len(times)} passes of {t:.2f} s, scaled to a full token; oracle/torch_port.py = "
                      "reference torch fallback (unpack + gather + F.linear) in fp32"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, q, metric, cfg_name = MODELS[args.model]
    steps, warm = max(args.steps, 1), max(args.warmup, 1)
    cb, vals = None, []
    t_begin = time.perf_counter()
    for i in range(warm + steps):
        cb = cpu_baseline(m, q, budget_s=0.0, min_reps=1)             # one pass over the layer per step
        if i >= warm:
            vals.append(cb["value"])
        if time.perf_counter() - t_begin > 240 and len(vals) >= 3:    # keep the whole run within minutes
            break
    v = statistics.median(vals)
    cb["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": "tokens/s", "n_gpus": args.gpus, "steps": len(vals),
        "warmup": warm, "ms_per_step": round(1e3 / v, 1), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(m, q, cfg_name),
                   "sample": "each step = one decoder layer (7 linears) timed on the host cores, scaled to a whole token"},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU-vs-GPU bar: the reference's OWN CUDA kernels (oracle/_ref/libvptq.so, unmodified sources compiled for
# sm_100a by oracle/build_ref.sh) timed on the same box, eager, one launch pair per linear as the reference runs
# them (csrc/quant_gemv.cu:241-294 + its sum(-1) epilogue; prefill: csrc/dequant.cu:227-287 + F.linear).
# ------------------------------------------------------------------------------------------------
def prefill_timing(m, q, stack, device, dtype, tokens=8192):
    """BASELINE.json configs[2] (prefill, batch 4 x seq 2048 = 8192 tokens) on the three distinct linear shapes of one
    decoder layer: vptq_b200_quant_gemm (prep + dequant into the workspace + hand-written tcgen05 GEMM) next to OUR
    dequant kernel + cuBLAS through torch, and the tensor-pipe share of the bf16 sustained peak."""
    import torch
    from vptq_b200 import native
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops_sustained", 1436.0))
    out = {"tokens": tokens, "shapes": {}}
    for name in ("q", "gate", "down"):
        t = stack[0][name]
        i, o, d = t["in"], t["out"], t["desc"]
        x = torch.randn(tokens, i, device=device).to(dtype)
        y = torch.empty(tokens, o, device=device, dtype=dtype)
        W = torch.empty(o, i, device=device, dtype=dtype)

        def med(fn, n=7):
            fn(); torch.cuda.synchronize()
            ts = []
            for _ in range(n):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            return sorted(ts)[len(ts) // 2]
        ours = med(lambda: native.quant_gemm(d, x, y))

        def deq_cublas():
            native.dequant(d, W)
            torch.nn.functional.linear(x, W)
        cub = med(deq_cublas)
        tf = 2.0 * tokens * i * o / (ours * 1e-3) / 1e12
        out["shapes"][f"{name}_{o}x{i}"] = {"ms": round(ours, 4), "tflops": round(tf, 1), "frac_of_bf16_sustained": round(tf / peak, 3),
                                            "our_dequant_plus_cublas_ms": round(cub, 4)}
        del x, y, W
    out["how"] = ("median of 7, CUDA events, whole op (x' prep + dequant + GEMM); flops = 2*T*I*O; peak = "
                  "MEASURED_PEAKS.json bf16_tflops_sustained")
    return out


def ref_cuda_timing(m, q, device, dtype, prefill_tokens=8192):
    import importlib.util
    import torch
    so = os.path.join(ROOT, "oracle", "_ref", "libvptq.so")
    if not os.path.exists(so):
        return {"unavailable": "oracle/_ref/libvptq.so not built (oracle/build_ref.sh needs /root/reference)"}
    try:
        spec = importlib.util.spec_from_file_location("libvptq", so)
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"cannot load oracle/_ref/libvptq.so: {e!r}"[:200]}
    v = q["vector_len"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)      # > L2: every timed launch streams from HBM
    out = {"us_per_shape": {}, "how": "CUDA events around quant_gemv (kernel + sum(-1)), L2 flushed before each call, "
                                      "median of 7; tokens_per_s = 1 / (sum over the 7 linears x layers), eager launches "
                                      "excluded (kernel time only: favourable to the reference)"}
    per_layer_us = 0.0
    shapes = {}
    for name, i, o in model_linears(m):
        shapes.setdefault((i, o), []).append(name)
    prefill = {}
    for (i, o), names in shapes.items():
        t = layer_tensors(m, q, 0, names[0], i, o, device, dtype)
        x = torch.randn(1, i, device=device).to(dtype)
        args = (t["indices"], t["centroids"].view(1, -1, v), None,
                None if t["res_centroids"] is None else t["res_centroids"].view(1, -1, v), None, None,
                t["perm"], t["weight_scale"], t["weight_bias"], None, i, o)
        y = ref.quant_gemv(x, *args)
        torch.cuda.synchronize()
        ts = []
        for _ in range(7):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); ref.quant_gemv(x, *args); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        us = sorted(ts)[len(ts) // 2]
        for n in names:
            out["us_per_shape"][n] = round(us, 2)
            per_layer_us += us
        if prefill_tokens and names[0] in ("q", "gate", "down"):
            # the reference's prefill path on this shape: dequant kernel + cuBLAS (vptq/ops/quant_gemm.py:231-275)
            inv = torch.argsort(t["perm"].view(torch.uint16).to(torch.int64)).to(torch.uint16).view(torch.int16)
            dargs = (t["indices"], t["centroids"].view(1, -1, v), None,
                     None if t["res_centroids"] is None else t["res_centroids"].view(1, -1, v), None, None, inv,
                     t["weight_scale"], t["weight_bias"], v, i, o)
            xp = torch.randn(prefill_tokens, i, device=device).to(dtype)
            W = ref.dequant(*dargs)
            torch.nn.functional.linear(xp, W)
            torch.cuda.synchronize()
            tp_ = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); W = ref.dequant(*dargs); yy = torch.nn.functional.linear(xp, W); e1.record()
                torch.cuda.synchronize()
                tp_.append(e0.elapsed_time(e1))
            prefill[f"{names[0]}_{o}x{i}"] = {"tokens": prefill_tokens, "ms": round(sorted(tp_)[len(tp_) // 2], 4)}
            del xp, W
        del t
    out["tokens_per_s"] = round(1e6 / (per_layer_us * m["layers"]), 2)
    if prefill:
        out["prefill_dequant_plus_cublas"] = prefill
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefill", action="store_true", help="skip the BASELINE configs[2] prefill timings")
    ap.add_argument("--no-module-level", action="store_true", help="skip the VQuantLinear.forward / fuse(model) timings")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference's own CUDA kernels (oracle/_ref)")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--tp-mode", default="p2p", choices=["p2p", "p2p-plain", "nccl"],
                    help="N > 1: exchange fused into the GEMV over peer memory (p2p: tagged words; p2p-plain: plain "
                         "values + epoch flags) or memset + NCCL all-reduce (nccl)")
    ap.add_argument("--tp-eager", action="store_true", help="N > 1: launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--debug-layers", type=int, default=0, help="debugging only: truncate the model (invalid as a result)")
    ap.add_argument("--model", default="llama3-8b", choices=sorted(MODELS))
    ap.add_argument("--no-check", action="store_true", help="skip the unsharded recomputation of the token")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
