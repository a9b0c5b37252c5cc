"""Cost of the oracle PORT (bench.py's CPU arm) relative to the real, unmodified reference MsViT on identical cores.
Imports the reference checkout through oracle/make_golden.py's timm shim and writes profiles/r02_port_vs_reference.json,
which bench.py attaches to `cpu_baseline`.
usage: python tools/port_vs_reference.py <vision-longformer checkout> [threads]"""
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import import_reference  # noqa: E402
from oracle.vil_oracle import OracleLong2DSCSelfAttention  # noqa: E402
from vision_longformer_b200 import ARCHS, build_vil  # noqa: E402

threads = int(sys.argv[2]) if len(sys.argv) > 2 else min(os.cpu_count() or 1, 16)
torch.set_num_threads(threads)
_, _, RefMsViT = import_reference(sys.argv[1])
B, IMG = 4, 224


def time_steps(net, steps=3, warmup=1):
    opt = torch.optim.AdamW(net.parameters(), lr=5e-4, weight_decay=0.05)
    x, y = torch.randn(B, 3, IMG, IMG), torch.randint(0, 1000, (B,))
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = torch.nn.functional.cross_entropy(net(x), y)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts)


torch.manual_seed(0)
ref = RefMsViT(arch=ARCHS["vil_small"], img_size=IMG, drop_path_rate=0.1, norm_embed=True, sharew=True, attn_type="longformerhand",
               sw_exact=0, mode=0, ln_eps=1e-6).train()
port = build_vil("vil_small", img_size=IMG, attn_cls=OracleLong2DSCSelfAttention).train()
t_port0 = time_steps(port)
t_ref = time_steps(ref)
t_port = 0.5 * (t_port0 + time_steps(port))          # port measured before and after the reference (drift check)
out = {"port_s_per_step_before_after": [t_port0, 2 * t_port - t_port0], "threads": threads, "batch": B, "reference_s_per_step": t_ref, "port_s_per_step": t_port,
       "port_over_reference_time_ratio": t_port / t_ref,
       "what": "ViL-Small 224 fwd+bwd+AdamW, fp32 CPU: unmodified reference MsViT(attn_type='longformerhand') vs the MsViT harness with "
               "the oracle port of the sliding-chunk algorithm"}
print(json.dumps(out, indent=1))
with open(os.path.join(ROOT, "profiles", "r02_port_vs_reference.json"), "w") as f:
    json.dump(out, f, indent=1)
