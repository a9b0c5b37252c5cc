#!/usr/bin/env python
"""bench.py -- ViL-Small 224x224 bf16 training throughput (images/sec) on N B200s, with the
Vision-Longformer attention hot path running on the vil_attn sm_100a kernels.

Contract (see the task statement):  python bench.py --gpus N --steps K --warmup W  prints ONE JSON line.
  value      : whole-job images/sec, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        : same step through the public module API with pinned-HOST images copied H2D and the loss
               read back D2H inside the timed region
  roofline   : the dominant hot-path kernel, timed alone with CUDA events inside this process
  cpu_baseline: the oracle port of the reference's CPU path (same model, small batch) on the host cores
  --impl reference : only the CPU arm (reference algorithm port), same metric / config
  --dump-outputs DIR: after the timed steps, what the last timed step computed, as DIR/<name>.npy (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it

PER_GPU_BATCH = 256           # BASELINE config 3: synthetic ImageNet-shape batch = 256 / GPU
MODEL, IMG = "vil_small", 224


def ncu_traffic(key):
    """DRAM bytes per launch measured by `ncu --set full` for this kernel (profiles/ncu_traffic.json, written by
    tools/ncu_traffic.py from the committed capture); None when the capture does not cover it."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            return json.load(f)[key]["dram_bytes"]
    except (OSError, KeyError, ValueError):
        return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d["hbm_gbs"], d["bf16_tflops"], "measured (MEASURED_PEAKS.json, burst)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.stop_flag, self.index = [], False, index
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [p.strip() for p in out.stdout.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.thread.join(timeout=3)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        mhz = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
                "samples": len(mhz)}


# ------------------------------------------------------------------------------------------ algorithmic work
def algorithmic_work(nx, ny, w, g, H, M, exact=0):
    """SURVEY.md section 8(d): FLOPs and bytes of ONE image, ONE layer, forward (bf16 I/O)."""
    Nloc, N = nx * ny, nx * ny + g

    def allowed_rows(n):
        out = []
        for r in range(n):
            if exact == 1:
                out.append(min(n - 1, r + w) - max(0, r - w) + 1)
            else:
                lo, hi = max(0, (r // w - 1) * w), min(n, (r // w + 2) * w)
                out.append(hi - lo)
        return sum(out)
    pairs = allowed_rows(nx) * allowed_rows(ny)
    flops = 4 * M * H * (pairs + Nloc * g + g * N)
    byts = 2 * H * M * (2 * Nloc + 2 * N + 2 * g) + 4 * H * Nloc
    return flops, byts


# ------------------------------------------------------------------------------------------ kernel microbench
def _gpu_backlog(cycles=400_000):
    """Keep the GPU busy (~0.2 ms spin kernel on the timing stream) while the host enqueues `start event, kernel(s), stop event`:
    otherwise the 15-30 us the host needs to fill the C-ABI struct and launch sit INSIDE the event bracket (the stream is idle,
    the start event fires at once) and inflate a 60-300 us kernel by 10-30 %."""
    torch.cuda._sleep(cycles)


def _heads(t, H, which=0, parts=1):
    B, T, C = t.shape
    return t.view(B, T, parts, H, C // (parts * H))[:, :, which].permute(0, 2, 1, 3)


def kernel_microbench(dev, reps=10, variants=True):
    """BASELINE config 2: attention-operator-only fwd / bwd at the ViL-Small hot-layer shapes, B=256, bf16, in the
    PRODUCTION layout (q / k / v = strided views of the query / kv Linear outputs, head-merged output, gradients written
    into Linear-layout buffers), timed with CUDA events on the launching stream; the tensors of one call (>= 0.6 GB per
    shape) are cycled through 3 distinct buffer sets so consecutive reps cannot hit L2 (126 MB).
    Per shape: the fused round-2 pipeline (default) and, for reference, the round-1 multi-kernel pipeline
    (VIL_FLAG_UNFUSED); `variants` adds exact=1 and rpe-on timings of the fused/default path."""
    from vision_longformer_b200 import _lib, vil_attention_raw_backward, vil_attention_raw_forward
    res = {}
    B = PER_GPU_BATCH
    for tag, (H, M, nx, ny) in {"S1": (3, 32, 56, 56), "S2": (3, 64, 28, 28)}.items():
        w, g = 7, 1
        N, C = g + nx * ny, H * M
        gen = torch.Generator(device=dev).manual_seed(300)
        mk = lambda *s: torch.randn(*s, generator=gen, device=dev, dtype=torch.float32).to(torch.bfloat16)
        sets = []
        for _ in range(3):
            q_all, kv, d_out = mk(B, N, C), mk(B, N, 2 * C), mk(B, N, C)
            out, dq_all, dkv = torch.empty_like(q_all), torch.empty_like(q_all), torch.empty_like(kv)
            sets.append(dict(q=_heads(q_all, H)[:, :, g:], qg=_heads(q_all, H)[:, :, :g], k=_heads(kv, H, 0, 2), v=_heads(kv, H, 1, 2),
                             o=_heads(out, H)[:, :, g:], og=_heads(out, H)[:, :, :g], go=_heads(d_out, H)[:, :, g:],
                             gog=_heads(d_out, H)[:, :, :g], dq=_heads(dq_all, H)[:, :, g:], dqg=_heads(dq_all, H)[:, :, :g],
                             dk=_heads(dkv, H, 0, 2), dv=_heads(dkv, H, 1, 2), keep=(q_all, kv, d_out, out, dq_all, dkv)))
        table = 0.02 * torch.randn((4 * w - 1) ** 2, H, device=dev)
        g2l, g2g = 0.02 * torch.randn(2, H, g, device=dev), 0.02 * torch.randn(H, g, g, device=dev)

        def timed(fn):
            for i in range(3):
                fn(i)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for i in range(reps):
                _gpu_backlog()
                ev[i][0].record()
                fn(i % 3)
                ev[i][1].record()
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b) for a, b in ev)
            return ts[len(ts) // 2]

        def bench_one(exact=0, rpe=False, flags=0, passes=True):
            kw = dict(nx=nx, ny=ny, w=w, exact=exact, mode=0, scale=M ** -0.5, flags=flags)
            tb, gl, gg = (table, g2l, g2g) if rpe else (None, None, None)
            dtb, dgl, dgg = (torch.zeros_like(table), torch.zeros_like(g2l), torch.zeros_like(g2g)) if rpe else (None, None, None)

            def run_f(s, skip=0):
                return vil_attention_raw_forward(s["q"], s["k"], s["v"], s["qg"], s["k"], s["v"], tb, gl, gg, s["o"], s["og"],
                                                 skip_mask=skip, **kw)

            def run_b(s, lse, lse_g, skip=0):
                vil_attention_raw_backward(s["q"], s["k"], s["v"], s["qg"], s["k"], s["v"], tb, gl, gg, s["o"], s["og"], lse, lse_g,
                                           s["go"], s["gog"], s["dq"], s["dk"], s["dv"], s["dqg"], s["dk"], s["dv"], dtb, dgl, dgg,
                                           skip_mask=skip, **kw)
            n0 = _lib.launch_count()
            lses = [run_f(s) for s in sets]
            n_f = (_lib.launch_count() - n0) // 3
            fam_f = _lib.last_impl()
            n0 = _lib.launch_count()
            for s, (l, lg) in zip(sets, lses):
                run_b(s, l, lg)
            n_b = (_lib.launch_count() - n0) // 3
            torch.cuda.synchronize()
            r = {"family_fwd": fam_f, "family_bwd": _lib.last_impl(), "launches_fwd": n_f, "launches_bwd": n_b,
                 "fwd_ms": timed(lambda i: run_f(sets[i])), "bwd_ms": timed(lambda i: run_b(sets[i], *lses[i]))}
            if passes:
                r["fwd_main_ms"] = timed(lambda i: run_f(sets[i], skip=1))                          # main forward kernel alone
                r["bwd_dq_ms"] = timed(lambda i: run_b(sets[i], *lses[i], skip=1 | 4 | 8))          # pass 1 alone
                r["bwd_dkv_ms"] = timed(lambda i: run_b(sets[i], *lses[i], skip=1 | 2 | 8))         # pass 2 alone
            return r

        flops, byts = algorithmic_work(nx, ny, w, g, H, M)
        r = {"layout": "strided views of the query / kv Linear outputs (production)", "flops_fwd": flops * B, "bytes_fwd": byts * B}
        r.update(bench_one())
        r["round1_pipeline"] = bench_one(flags=_lib.VIL_FLAG_UNFUSED)
        if variants:
            fl1, _ = algorithmic_work(nx, ny, w, g, H, M, exact=1)
            r["exact1"] = dict(bench_one(exact=1, passes=False), flops_fwd=fl1 * B)
            r["rpe_on"] = bench_one(rpe=True, passes=False)
        res[tag] = r
        del sets
        torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------ epilogue microbench
def epilogue_microbench(dev, reps=10):
    """SURVEY.md section 8 (f) row 4 kernels (residual add + DropPath scale + deferred bias + LayerNorm; bias + GELU; column-sum bias
    gradient) at the ViL-Small token streams, B=256, through the C ABI on preallocated buffers (no autograd / allocator in the
    timed region): pure HBM kernels, so the figure of merit is algorithmic bytes / time against the measured HBM peak.
    CUDA events on the launching stream, 3 buffer sets cycled (one call moves >= 0.2 GB: nothing survives in the 126 MB L2)."""
    from vision_longformer_b200 import _lib, epilogue as ep
    res = {}
    B = PER_GPU_BATCH
    peak = peaks()[0]
    bf = torch.bfloat16
    for tag, (N, C) in {"S1": (1 + 56 * 56, 96), "S2": (1 + 28 * 28, 192), "S3": (1 + 14 * 14, 384)}.items():
        rows = B * N
        f32 = lambda *s: torch.randn(*s, device=dev)
        gamma, beta, bias, scale = torch.ones(C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev), torch.ones(B, device=dev)
        b1 = torch.zeros(4 * C, device=dev)
        sets = [dict(x=f32(rows, C), br=f32(rows, C).to(bf), xo=torch.empty(rows, C, device=dev), y=torch.empty(rows, C, device=dev, dtype=bf),
                     mean=torch.empty(rows, device=dev), rstd=torch.empty(rows, device=dev), dy=f32(rows, C).to(bf), gres=f32(rows, C),
                     dx=torch.empty(rows, C, device=dev), dbr=torch.empty(rows, C, device=dev, dtype=bf),
                     z=f32(rows, 4 * C).to(bf), a=torch.empty(rows, 4 * C, device=dev, dtype=bf), da=f32(rows, 4 * C).to(bf),
                     dz=torch.empty(rows, 4 * C, device=dev, dtype=bf)) for _ in range(3)]
        dg, db, dbi, db1 = torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty(4 * C, device=dev)
        ws_an = ep.addnorm_workspace(rows, C, dev)
        ws_g = ep.bias_act_workspace(sets[0]["da"], _lib.VIL_ACT_GELU)
        ws_c = ep.bias_act_workspace(sets[0]["da"], _lib.VIL_ACT_NONE)

        def timed(fn):
            for i in range(3):
                fn(sets[i])
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for i in range(reps):
                _gpu_backlog()
                ev[i][0].record()
                fn(sets[i % 3])
                ev[i][1].record()
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b) for a, b in ev)
            return ts[len(ts) // 2]

        e = rows * C
        kernels = (
            ("addnorm_fwd", lambda s: ep.addnorm_raw_forward(s["x"], s["br"], bias, scale, gamma, beta, s["xo"], s["y"], s["mean"], s["rstd"], 1e-6, N),
             e * (4 + 2 + 4 + 2)),                                     # x, br -> xo, y
            ("addnorm_bwd", lambda s: ep.addnorm_raw_backward(s["xo"], gamma, s["mean"], s["rstd"], scale, s["dy"], s["gres"], s["dx"], s["dbr"],
                                                              dg, db, dbi, ws_an, 1e-6, N),
             e * (2 + 4 + 4 + 4 + 2)),                                 # dy, gres, xo -> dx, dbr (+ 3 column sums); 2 launches
            ("bias_gelu_fwd", lambda s: ep.bias_act_raw_forward(s["z"], b1, s["a"], _lib.VIL_ACT_GELU), 4 * e * (2 + 2)),
            ("bias_gelu_bwd", lambda s: ep.bias_act_raw_backward(s["da"], s["z"], b1, s["dz"], db1, ws_g, _lib.VIL_ACT_GELU),
             4 * e * (2 + 2 + 2)),                                     # da, z -> dz (+ d_bias); 2 launches
            ("colsum", lambda s: ep.bias_act_raw_backward(s["da"], None, None, None, db1, ws_c, _lib.VIL_ACT_NONE), 4 * e * 2),
            # context: what a plain device copy of the bias_gelu_fwd tensor achieves at THIS size (the 6571 GB/s peak was measured on
            # a 2 x 2 GiB copy; these streams are 0.15 - 1.2 GB and pay launch / ramp-up / tail on 60 - 300 us kernels)
            ("torch_copy_same_size", lambda s: s["a"].copy_(s["z"]), 4 * e * (2 + 2)))
        r = {"rows": rows, "C": C}
        for name, fn, byts in kernels:
            ms = timed(fn)
            r[name] = {"ms": round(ms, 4), "algorithmic_bytes": byts, "GBps": round(byts / ms / 1e6, 1),
                       "hbm_frac": round(byts / (ms * 1e-3) / (peak * 1e9), 3)}
        res[tag] = r
        del sets
        torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------ BASELINE config 5
def config5_sweep(dev, B=8, img=512, reps=10):
    """ViL-Base-Deep backbone forward at 512x512, window sweep w in {7,15,31} x nglo in {1,8} in the two longformer stages
    (arch README.md:236 of the reference with `f` / `g` overridden), bf16 autocast, batch 8, forward_features only.
    Per (w, g): backbone ms (CUDA events, median) and the attention operator alone at the stage-1 / stage-2 shapes with its
    fraction of the measured bf16 tensor peak (w >= 12 is the tensor-bound regime, SURVEY.md section 8(d))."""
    from vision_longformer_b200 import _lib, build_vil, vil_attention_raw_forward
    hbm, tflops, _ = peaks()
    out = []

    def timed(fn):
        for _ in range(3):
            fn()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) for a, b in ev)
        return ts[len(ts) // 2]

    x = torch.randn(B, 3, img, img, device=dev)
    for w in (7, 15, 31):
        for g in (1, 8):
            arch = (f"l1,h3,d96,n1,s1,g{g},p4,f{w}_l2,h3,d192,n8,s1,g{g},p2,f{w}_l3,h6,d384,n24,s0,g1,p2,f7_"
                    f"l4,h12,d768,n1,s0,g0,p2,f7")
            torch.manual_seed(0)
            net = build_vil(arch, img_size=img, drop_path_rate=0.0).to(dev).eval()

            def fwd():
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                    return net.forward_features(x)
            rec = {"w": w, "nglo": g, "backbone_fwd_ms": timed(fwd)}
            for stage, (H, M, n) in {"stage1": (3, 32, img // 4), "stage2": (3, 64, img // 8)}.items():
                N, C = g + n * n, H * M
                q_all = torch.randn(B, N, C, device=dev).bfloat16()
                kv = torch.randn(B, N, 2 * C, device=dev).bfloat16()
                o_all = torch.empty_like(q_all)
                hd = _heads
                args = (hd(q_all, H)[:, :, g:], hd(kv, H, 0, 2), hd(kv, H, 1, 2), hd(q_all, H)[:, :, :g], hd(kv, H, 0, 2), hd(kv, H, 1, 2),
                        None, None, None, hd(o_all, H)[:, :, g:], hd(o_all, H)[:, :, :g])
                ms = timed(lambda: vil_attention_raw_forward(*args, nx=n, ny=n, w=w, exact=0, mode=0, scale=M ** -0.5))
                fl, by = algorithmic_work(n, n, w, g, H, M)
                rec[stage] = {"tokens": f"{n}x{n}", "H": H, "D": M, "family": _lib.last_impl(), "attn_fwd_ms": ms,
                              "tensor_frac": fl * B / (ms * 1e-3) / 1e12 / tflops, "hbm_frac": by * B / (ms * 1e-3) / 1e9 / hbm,
                              "flop_per_byte": fl / by}
            out.append(rec)
            del net
            torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------ output dump
DUMP_SAMPLE = 1 << 21        # elements kept of the flattened gradients / parameters (8 MB each in float32)


def dump_outputs(out_dir, net, loss, logits):
    """Write what one training step hands back to its caller, so that two builds can be compared output for output:
    logits.npy (batch x classes), loss.npy, and grads.npy / params.npy - the gradients and the updated parameters of
    net.parameters(), flattened in order and sampled at DUMP_SAMPLE fixed (seed 0) positions.  All float32, 17 MB for
    ViL-Small."""
    params = list(net.parameters())
    flat_p = torch.cat([p.detach().reshape(-1) for p in params]).float().cpu()
    flat_g = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1) for p in params]).float().cpu()
    n = flat_p.numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values if n > DUMP_SAMPLE else None
    arrays = {"logits": logits.detach().float().cpu(), "loss": loss.detach().float().cpu(),
              "params": flat_p if idx is None else flat_p[idx], "grads": flat_g if idx is None else flat_g[idx]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_training_throughput(steps, warmup, batch=4):
    """The reference's CPU path, restated (oracle port, `chunked_attention` with the hand-written backward
    structure of SlidingChunk2D) inside the same MsViT harness: ViL-Small 224 fwd+bwd+AdamW, fp32."""
    from oracle.vil_oracle import OracleLong2DSCSelfAttention
    from vision_longformer_b200 import build_vil
    torch.manual_seed(0)
    # torch's CPU thread pool collapses on many-core hosts for this op mix (measured on the 128-core GPU box:
    # 157 s/step with 128 threads vs ~2 s/step with 8): cap the pool and report the threads actually used.
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    net = build_vil(MODEL, img_size=IMG, attn_cls=OracleLong2DSCSelfAttention).train()
    opt = torch.optim.AdamW(net.parameters(), lr=5e-4, weight_decay=0.05)
    x = torch.randn(batch, 3, IMG, IMG)
    y = torch.randint(0, 1000, (batch,))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = torch.nn.functional.cross_entropy(net(x), y)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return batch * len(times) / total, total / len(times) * 1e3, cores, batch


def port_cost_note():
    """The CPU arm is the oracle PORT of the reference algorithm (the reference tree does not exist on the GPU box).  Its
    cost relative to the real reference MsViT on identical cores was measured in the authoring container
    (tools/port_vs_reference.py -> profiles/r02_port_vs_reference.json) and is reported with the number."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_port_vs_reference.json")))
        return {"port_over_reference_time_ratio": d["port_over_reference_time_ratio"],
                "ratio_source": "profiles/r02_port_vs_reference.json (reference MsViT vs oracle port, same cores, authoring container)"}
    except (OSError, KeyError, ValueError):
        return {}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, min(args.warmup, 3))
    ips, ms, cores, batch = cpu_training_throughput(steps, warmup)
    line = {"impl": "reference", "metric": "images/sec ViL-Small 224x224 training", "value": ips, "unit": "images/sec",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"ViL-Small 224x224 training step (fwd+bwd+AdamW), batch {batch} (bounded CPU sample "
                                   f"of the {PER_GPU_BATCH}/GPU workload)", "attn": "oracle port of ATTN_TYPE=longformerhand"},
            "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": cores, "kind": "port",
                             "sample": f"{steps} timed steps of batch {batch}, fp32, torch CPU threads={cores}", **port_cost_note()},
            "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH)
    ap.add_argument("--arch", default=MODEL, help="side configs only (e.g. vil_medium_deep with --img-size 384, BASELINE "
                                                  "config 4); the headline metric is the default vil_small / 224")
    ap.add_argument("--img-size", type=int, default=IMG)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-microbench", action="store_true")
    ap.add_argument("--micro-only", action="store_true", help="only the attention-kernel microbench (BASELINE config 2)")
    ap.add_argument("--config5", action="store_true", help="BASELINE config 5: ViL-Base-Deep 512x512 backbone-forward window sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the logits, loss and a fixed sample of the "
                                                          "gradients and updated parameters of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs CUDA devices; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from vision_longformer_b200 import _lib, build_vil
    _lib.load()                 # built by __graft_entry__.build(); raises when it is missing
    if args.config5:
        sweep = config5_sweep(dev)
        base = next(r for r in sweep if r["w"] == 7 and r["nglo"] == 1)
        print(json.dumps({"metric": "ms backbone forward ViL-Base-Deep 512x512 (BASELINE config 5)", "value": base["backbone_fwd_ms"],
                          "unit": "ms", "n_gpus": 1, "higher_is_better": False, "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": "ViL-Base-Deep backbone forward_features, 512x512, batch 8, bf16 autocast, window sweep "
                                                 "w in {7,15,31} x nglo in {1,8} in stages 1-2; value = the (w=7, nglo=1) point"},
                          "sweep": sweep}))
        return
    if args.micro_only:
        mb = kernel_microbench(dev)
        for tag, r in mb.items():
            print(tag, json.dumps({k: v for k, v in r.items() if k not in ("flops_fwd", "bytes_fwd")}))
        print("epilogue", json.dumps(epilogue_microbench(dev)))
        return
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    warmup = max(3, args.warmup)
    steps = args.steps
    B = args.batch

    torch.manual_seed(1234 + rank)
    arch, img = args.arch, args.img_size
    net = build_vil(arch, img_size=img).to(dev).train()
    model = net
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local], gradient_as_bucket_view=True,
                                                          static_graph=True)
    opt = torch.optim.AdamW(model.parameters(), lr=5e-4, weight_decay=0.05, fused=True)
    x_dev = torch.randn(B, 3, img, img, device=dev)
    y_dev = torch.randint(0, 1000, (B,), device=dev)
    x_host = torch.randn(B, 3, img, img).pin_memory()
    y_host = torch.randint(0, 1000, (B,)).pin_memory()

    def step(x, y):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = model(x)
            loss = torch.nn.functional.cross_entropy(logits, y)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss, logits

    def sync_all():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    for _ in range(warmup):
        step(x_dev, y_dev)
    sync_all()

    # ---- device-resident timing
    launches0 = _lib.launch_count()
    with ClockSampler(local) as clk:
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last_step = step(x_dev, y_dev)
        e1.record()
        sync_all()
    launches = _lib.launch_count() - launches0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net, *last_step)
    del last_step

    # ---- end-to-end timing: every step's images / labels are copied from PINNED HOST memory inside the timed region and
    # the loss is read back every step.  The copy of step i+1 runs on a side stream while step i computes (double-buffered
    # device staging, event-ordered) - what a real input pipeline does; round 1 issued it on the compute stream (7 % loss).
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [(torch.empty_like(x_dev), torch.empty_like(y_dev)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        xb, yb = stage[i & 1]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[i & 1])             # the step that last used this staging buffer has finished
            xb.copy_(x_host, non_blocking=True)
            yb.copy_(y_host, non_blocking=True)
            ready[i & 1].record(copy_stream)

    def e2e_loop(n):
        cur = torch.cuda.current_stream(dev)
        for b in range(2):
            freed[b].record(cur)
        prefetch(0)
        last = 0.0
        for i in range(n):
            if i + 1 < n:
                prefetch(i + 1)
            cur.wait_event(ready[i & 1])
            xb, yb = stage[i & 1]
            loss, _ = step(xb, yb)
            freed[i & 1].record(cur)
            last = loss.item()                                # D2H read of the step's result
        return last

    e2e_loop(2)
    sync_all()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    loss_value = e2e_loop(steps)
    e3.record()
    sync_all()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))

    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return

    hbm, tflops, peak_src = peaks()
    side = (arch, img) != (MODEL, IMG)
    s1 = [c for c in net.layer_cfgs if c["s"]][:2]
    wins = "/".join(str(c["f"]) for c in s1)
    line = {"metric": "images/sec ViL-Small 224x224 training" if not side else f"images/sec {arch} {img}x{img} training (side config)",
            "value": world * B * steps / (ms_total / 1e3),
            "unit": "images/sec", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{arch} {img}x{img} bf16 training step (fwd+bwd+fused AdamW), {B} img/GPU, "
                                   f"ATTN_TYPE=longformerhand -> vil_attn sm_100a kernels, w={wins} in the longformer stages, "
                                   f"SW_EXACT=0, rpe off (published arch string), DDP over NCCL when n_gpus>1",
                       "arch": arch, "img_size": img, "global_batch": world * B, "parallelism": f"dp{world}",
                       "l2": "per-step activation working set is several GB (>> 126 MB L2); no explicit flush",
                       "harness": "reference block structure; residual add + DropPath + deferred bias + LayerNorm and bias + GELU in the "
                                  "vil_addnorm / vil_bias_act kernels (fused_residual=True), NHWC patch-merge convolutions; GEMMs cuBLAS, dense "
                                  "s0-stage attention cuDNN SDPA"},
            "e2e": {"value": world * B * steps / (ms_e2e / 1e3), "unit": "images/sec",
                    "h2d_bytes_per_step": x_host.numel() * 4 + y_host.numel() * 8, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / steps, "last_loss": loss_value,
                    "h2d": "pinned host -> device every step on a side stream, overlapped with the previous step"},
            "gpu_launches": launches, "clocks": clocks, "attn_family": _lib.last_impl()}

    if world == 1 and not args.no_microbench:
        mb = kernel_microbench(dev)
        # dominant hot-path kernel = the slowest single kernel among the timed ones
        cands = []
        for tag, r in mb.items():
            cands += [(r["fwd_main_ms"], tag, "fwd"), (r["bwd_dq_ms"], tag, "bwd_dq"), (r["bwd_dkv_ms"], tag, "bwd_dkv")]
        ms, tag, name = max(cands)
        r = mb[tag]
        # algorithmic bytes of that launch (DESIGN.md section 5, SURVEY.md section 8(d) per-image figure x 256 images):
        # fwd: read q,k,v write o (4 token-tensors);  pass 1: read q,k,v,dO,o write dq (6);  pass 2: read q,k,v,dO write dk,dv
        # (6);  fp32 lse/delta ignored.  FLOPs: fwd 2 GEMMs, pass 1: 3 (S, dP, dQ), pass 2: 4 (S, dP, dK, dV) - the recomputed
        # GEMMs ARE counted for a single pass because each pass is its own launch.
        kbytes = r["bytes_fwd"] * {"fwd": 1.0, "bwd_dq": 6 / 4, "bwd_dkv": 6 / 4}[name]
        kflops = r["flops_fwd"] * {"fwd": 1.0, "bwd_dq": 3 / 2, "bwd_dkv": 4 / 2}[name]
        achieved = kbytes / (ms * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": f"{name}[{tag}] ({r['family_fwd'] if name == 'fwd' else r['family_bwd']})",
                            "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                            "traffic": ncu_traffic(f"{name}[{tag}]"),
                            "traffic_source": "profiles/ncu_traffic.json (ncu --set full capture of this build, committed)",
                            "algorithmic_bytes": kbytes, "peak_source": peak_src, "kernel_ms": ms,
                            "tensor_frac": kflops / (ms * 1e-3) / 1e12 / tflops}
        # whole operator (SURVEY.md section 8(d) accounting: backward = 2 x forward bytes / flops), 1 x S1 + 2 x S2 layers
        op_ms = sum(r2["fwd_ms"] + r2["bwd_ms"] for r2 in mb.values()) + mb["S2"]["fwd_ms"] + mb["S2"]["bwd_ms"]
        op_bytes = 3 * (mb["S1"]["bytes_fwd"] + 2 * mb["S2"]["bytes_fwd"])
        op_flops = 3 * (mb["S1"]["flops_fwd"] + 2 * mb["S2"]["flops_fwd"])
        old_ms = sum(r2["round1_pipeline"]["fwd_ms"] + r2["round1_pipeline"]["bwd_ms"] for r2 in mb.values()) + \
            mb["S2"]["round1_pipeline"]["fwd_ms"] + mb["S2"]["round1_pipeline"]["bwd_ms"]
        line["roofline"]["operator"] = {"ms_fwd_bwd_3_layers": op_ms, "hbm_frac": op_bytes / (op_ms * 1e-3) / 1e9 / hbm,
                                        "tensor_frac": op_flops / (op_ms * 1e-3) / 1e12 / tflops,
                                        "round1_pipeline_ms": old_ms}
        line["kernel_bench"] = mb
        line["kernel_bench"]["hot_path_ms_per_256img"] = op_ms      # 1x S1 + 2x S2 layers, fwd+bwd
        line["kernel_bench"]["hot_path_images_per_sec"] = PER_GPU_BATCH / (op_ms * 1e-3)
        # SURVEY.md section 8 (f) row 4 kernels around the operator: HBM-bound, reported against the same measured HBM peak
        line["epilogue_bench"] = epilogue_microbench(dev)
    if world == 1 and not args.no_cpu_baseline:
        ips, ms, cores, batch = cpu_training_throughput(steps=2, warmup=1)
        line["cpu_baseline"] = {"value": ips, "unit": "images/sec", "cores": cores, "kind": "port",
                                "sample": f"2 timed ViL-Small training steps of batch {batch}, fp32 CPU, oracle port of "
                                          f"the reference's sliding-chunk algorithm ({ms:.0f} ms/step)",
                                **port_cost_note()}
    print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
