"""CPU: pin the oracle (oracle/vil_oracle.py) against golden vectors produced by
the UNMODIFIED reference (oracle/make_golden.py) and against itself."""
import pytest
import torch

from oracle import vil_oracle as vo
from tests.util import attn_cases, load_attn, load_golden, load_state, relerr


def run_module(gold, dense):
    kw = dict(gold["kwargs"])
    mod = vo.OracleLong2DSCSelfAttention(dense=dense, **kw).double()
    load_state(mod, gold["state_dict"])
    pick = gold["picked_mode"]
    mod.train(pick is not None)
    x = gold["x"].double().requires_grad_(True)
    y = mod(x, gold["nx"], gold["ny"], mode_override=pick)
    (y * gold["gy"].double()).sum().backward()
    grads = {n: p.grad for n, p in mod.named_parameters() if p.grad is not None}
    return y, x.grad, grads


@pytest.mark.parametrize("name", attn_cases())
@pytest.mark.parametrize("dense", [False, True], ids=["chunked", "dense"])
def test_oracle_matches_reference_golden(name, dense):
    gold = load_attn(name)
    y, dx, grads = run_module(gold, dense)
    assert relerr(y, gold["y"]) < 1e-12
    assert relerr(dx, gold["dx"]) < 1e-11
    for n, gref in gold["param_grads"].items():
        assert relerr(grads[n], gref) < 1e-6, n      # golden param grads are stored in fp32


def test_relative_position_index_matches_reference_buffer():
    for name in attn_cases():
        gold = load_attn(name)
        if "relative_position_index" in gold["state_dict"]:
            w = gold["kwargs"]["w"]
            assert torch.equal(vo.relative_position_index(w).int(), gold["state_dict"]["relative_position_index"])


def test_mask_closed_forms_match_reference_builders():
    masks = load_golden("masks.pt")
    for (kind, nx, ny, w), (ref_mask, ninv) in masks.items():
        exact = {"zero": 0, "exact": 1, "cyclic": -1}[kind]
        padx, pady, mx, my = vo.geometry(nx, ny, w)
        mine = vo.chunk_mask(nx, ny, w, exact, 0)[0]
        w2 = w * w
        if exact == 1:
            assert torch.equal(mine.reshape(mx * my, w2, 9 * w2), ref_mask)
            assert int(mine.sum()) == ninv
        else:
            assert torch.equal(mine.reshape(mx * my, 9 * w2), ref_mask)
            assert w2 * int(mine.sum()) == ninv          # the reference counts the w2 query rows


def test_exact1_rejects_modes():
    with pytest.raises(ValueError):
        vo.chunk_mask(14, 14, 7, 1, 3)
    with pytest.raises(ValueError):
        vo.visit_weights(14, 14, 7, 2, 0, None, 1)


@pytest.mark.parametrize("cfg", [(9, 11, 4, 2, 0, 0, True), (9, 11, 4, 1, 1, 0, True), (8, 8, 4, 1, 0, 5, False),
                                 (7, 6, 3, 3, -1, 0, True), (6, 6, 3, 1, 0, -1, True)])
def test_dense_and_chunked_agree(cfg):
    nx, ny, w, g, exact, mode, rpe = cfg
    torch.manual_seed(7)
    B, H, D = 2, 2, 8
    N = g + nx * ny
    mk = lambda *s: torch.randn(*s, dtype=torch.float64, requires_grad=True)
    q, k, v, qg = mk(B, H, nx * ny, D), mk(B, H, N, D), mk(B, H, N, D), mk(B, H, g, D)
    table = mk((4 * w - 1) ** 2, H) if rpe else None
    g2l = mk(2, H, g) if rpe else None
    g2g = mk(H, g, g) if rpe else None
    kw = dict(nx=nx, ny=ny, w=w, exact=exact, mode=mode, scale=D ** -0.5)
    o1, og1, _, _ = vo.dense_attention(q, k, v, qg, k, v, table, g2l, g2g, **kw)
    o2, og2 = vo.chunked_attention(q, k, v, qg, k, v, table, g2l, g2g, **kw)
    assert relerr(o1, o2) < 1e-12 and relerr(og1, og2) < 1e-12
    ins = [t for t in (q, k, v, qg, table, g2l, g2g) if t is not None]
    go, gog = torch.randn_like(o1), torch.randn_like(og1)
    g1 = torch.autograd.grad((o1 * go).sum() + (og1 * gog).sum(), ins)
    g2 = torch.autograd.grad((o2 * go).sum() + (og2 * gog).sum(), ins)
    for a, b in zip(g1, g2):
        assert relerr(a, b) < 1e-11


def test_oracle_against_reference_fresh_seed():
    """Beyond the attn_* cases: a configuration none of them uses (w=3, two global tokens, rpe, separate global
    weights, 8x10), against the reference's float64 forward."""
    gold = load_golden("reference_fresh_seed.pt")
    mine = vo.OracleLong2DSCSelfAttention(**gold["kwargs"]).double().eval()
    mine.load_state_dict(gold["state_dict"])
    assert relerr(mine(gold["x"], gold["nx"], gold["ny"]), gold["y"]) < 1e-13
