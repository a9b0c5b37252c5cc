"""bench.py's roofline accounting is pinned to the algorithmic work SURVEY.md section 8(d) computed for the BASELINE
configs (per image, per layer, forward) - the `roofline.achieved` figure is built from these numbers."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

# (nx, ny, w, g, H, M, exact) -> GFLOP per image (SURVEY.md 8(d) "Values [computed]")
SURVEY_GF = [
    ((56, 56, 7, 1, 3, 32, 0), 0.4486), ((56, 56, 7, 1, 3, 32, 1), 0.2384),      # ViL-Small stage 1
    ((28, 28, 7, 1, 3, 64, 0), 0.1856), ((28, 28, 7, 1, 3, 64, 1), 0.1030),      # ViL-Small stage 2
    ((96, 96, 8, 1, 3, 32, 0), 1.825), ((48, 48, 12, 1, 3, 64, 0), 1.596),        # Medium-Deep 384
    ((128, 128, 7, 1, 3, 32, 0), 2.57), ((128, 128, 15, 1, 3, 32, 0), 10.61), ((128, 128, 31, 1, 3, 32, 0), 37.45),
    ((64, 64, 7, 1, 3, 64, 0), 1.19), ((64, 64, 15, 1, 3, 64, 0), 4.38), ((64, 64, 31, 1, 3, 64, 0), 12.12),
]


@pytest.mark.parametrize("args,gf", SURVEY_GF, ids=lambda v: str(v))
def test_flops_match_survey(args, gf):
    nx, ny, w, g, H, M, exact = args
    flops, _ = bench.algorithmic_work(nx, ny, w, g, H, M, exact=exact)
    assert flops / 1e9 == pytest.approx(gf, rel=5e-3)      # SURVEY quotes 3-4 significant digits


def test_bytes_match_survey():
    # SURVEY.md: S1 2.41 MB (+ LSE) and S2 1.21 MB per image forward; all three hot layers 4.82 MB (rounded)
    _, b1 = bench.algorithmic_work(56, 56, 7, 1, 3, 32)
    _, b2 = bench.algorithmic_work(28, 28, 7, 1, 3, 64)
    assert b1 / 1e6 == pytest.approx(2.41, rel=2e-2)
    assert b2 / 1e6 == pytest.approx(1.21, rel=2e-2)


def test_committed_ncu_traffic_is_close_to_the_algorithmic_bytes():
    """DRAM traffic measured by ncu (profiles/ncu_traffic.json) must stay within 30 % of the algorithmic bytes of the
    launch: a larger gap would mean wasted re-reads (the first thing the roofline section is there to catch)."""
    with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
        tr = json.load(f)
    # pass 1 reads q, k, v, dO and O and writes dq (6 tensors: O is read here since round 2); pass 2 reads q, k, v, dO, writes dk, dv
    factor = {"fwd": 1.0, "fwd_local": 1.0, "bwd_dq": 6 / 4, "bwd_dkv": 6 / 4}
    shapes = {"S1": (56, 56, 7, 1, 3, 32), "S2": (28, 28, 7, 1, 3, 64)}
    # epilogue kernels (tools/epilogue_only.py streams, bf16 branch): bytes per (row, channel of the C-wide stream)
    epi = {"addnorm_fwd": 4 + 2 + 4 + 2, "addnorm_bwd": 2 + 4 + 4 + 4 + 2, "bias_gelu_fwd": 4 * (2 + 2), "bias_gelu_bwd": 4 * (2 + 2 + 2),
           "colsum": 2 * 2}
    streams = {"S1": (256 * (1 + 56 * 56), 96), "S2": (256 * (1 + 28 * 28), 192)}
    for key, rec in tr.items():
        name, tag = key[:-4], key[-3:-1]
        assert bench.ncu_traffic(key) == rec["dram_bytes"]
        if name in epi:                                  # pure streaming kernels: nothing is read twice
            rows, C = streams[tag]
            algo = rows * C * epi[name]
            assert 0.90 * algo < rec["dram_bytes"] < 1.10 * algo, (key, rec["dram_bytes"], algo)
            continue
        _, b = bench.algorithmic_work(*shapes[tag])
        if name.endswith("merge"):                       # per-unit partials of the global rows: a few MB per launch
            assert rec["dram_bytes"] < 0.03 * 256 * b, (key, rec["dram_bytes"])
            continue
        algo = 256 * b * factor[name]
        assert 0.75 * algo < rec["dram_bytes"] < 1.30 * algo, (key, rec["dram_bytes"], algo)


def test_dump_outputs_writes_the_step_results(tmp_path, monkeypatch):
    """--dump-outputs: float32 .npy files of the logits, loss and a fixed sample of the gradients / updated parameters."""
    import numpy as np
    import torch
    from oracle.vil_oracle import OracleLong2DSCSelfAttention
    from vision_longformer_b200 import build_vil
    torch.manual_seed(0)
    net = build_vil("l1,h2,d16,n1,s1,g1,p4,f4,a0_l2,h2,d32,n1,s1,g1,p2,f4_l3,h2,d32,n1,s0,g1,p2,f7", img_size=32,
                    num_classes=7, attn_cls=OracleLong2DSCSelfAttention)
    logits = net(torch.randn(2, 3, 32, 32))
    loss = torch.nn.functional.cross_entropy(logits, torch.tensor([1, 5]))
    loss.backward()
    n = sum(p.numel() for p in net.parameters())
    monkeypatch.setattr(bench, "DUMP_SAMPLE", n // 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), net, loss, logits)
    got = {f: np.load(tmp_path / "a" / f"{f}.npy") for f in ("logits", "loss", "grads", "params")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["logits"].shape == (2, 7) and got["loss"].shape == () and got["grads"].shape == got["params"].shape == (n // 3,)
    assert np.array_equal(got["logits"], logits.detach().numpy()) and got["loss"] == loss.item()
    flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).numpy()
    assert np.isin(got["params"], flat).all() and np.abs(got["grads"]).sum() > 0
    for f, a in got.items():                         # the sample positions are fixed
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{f}.npy")), f
