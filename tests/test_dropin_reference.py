"""The reference-side binding of INTEGRATION.md section 1, checked against what the UNMODIFIED reference exposes.

CPU part: `make_dropin_class` bound to a stand-in base class with the reference's constructor signature, placed at the
attention seam of the MsViT harness (`AttnBlock.__init__`, reference msvit.py:269-276), against the stock reference
`MsViT` (src/models/msvit.py:343) and `Long2DSCSelfAttention` as recorded by oracle/make_golden.py
(tests/golden/dropin_reference.pt): construction, state_dict layout and round trips, `reset_vil_mode`
(msvit.py:532-541), the public attributes and `compute_macs` (longformer2d.py:231-280).

GPU part: the same class factory run forward + backward and compared with the plain B200 module.
"""
import pytest
import torch
from torch import nn

from tests.util import load_golden
from vision_longformer_b200 import B200Long2DSCSelfAttention, MsViT, make_dropin_class


class _StandIn(nn.Module):
    """Same constructor signature as the reference class (longformer2d.py:13-14)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0., proj_drop=0., w=7, d=1,
                 autoregressive=False, sharew=False, nglo=1, only_glo=False, exact=0, autograd=False, rpe=False, mode=0):
        raise AssertionError("the base-class constructor must never run in the drop-in class")


def _tied(sd):
    """{key: the first key sharing its storage} for the state_dict entries that alias an earlier one."""
    first = {}
    return {k: t for k, t in ((k, first.setdefault(v.data_ptr(), k)) for k, v in sd.items()) if t != k}


def test_dropin_class_binds_into_reference_msvit():
    gold = load_golden("dropin_reference.pt")["msvit"]
    DropIn = make_dropin_class(_StandIn)
    torch.manual_seed(0)
    net = MsViT(attn_cls=DropIn, **gold["kwargs"])
    attn = [m for m in net.modules() if isinstance(m, _StandIn)]
    assert len(attn) == len(gold["attn"]) == 2 and all(type(m) is DropIn for m in attn)      # the two s1 stages
    assert all(m.forward.__func__ is B200Long2DSCSelfAttention.forward for m in attn)
    # one parameter set only, laid out like the stock reference model's
    sd = net.state_dict()
    assert {k: (tuple(v.shape), v.dtype) for k, v in sd.items()} == gold["state_dict"]
    assert sum(p.numel() for p in net.parameters()) == gold["n_params"]
    assert _tied(sd) == gold["tied"]                    # sharew: the global-token Linears are the local ones
    # checkpoints flow both ways: a checkpoint with the reference's layout loads strictly and reads back unchanged
    gen = torch.Generator().manual_seed(0)
    ckpt = {k: torch.randn(shape, generator=gen).to(dtype) for k, (shape, dtype) in gold["state_dict"].items()}
    ckpt.update({k: ckpt[t] for k, t in gold["tied"].items()})
    net.load_state_dict(ckpt, strict=True)
    for k, v in net.state_dict().items():
        assert torch.equal(v, ckpt[k]), k
    # reset_vil_mode reaches every longformer attention  (msvit.py:532-541)
    net.reset_vil_mode(0)
    assert all(m.mode == 0 for m in attn)
    net.reset_vil_mode(-1)
    assert all(m.mode == -1 for m in attn)
    # public attributes read elsewhere in the reference, and the reference's MAC count (longformer2d.py:231-280)
    for a, ref in zip(attn, gold["attn"]):
        for name, want in ref.items():
            if name != "macs_56x56":
                assert getattr(a, name) == want, name
        assert a.query is a.query_global and a.kv is a.kv_global and a.proj is a.proj_global      # sharew
        a.__flops__ = 0
        type(a).compute_macs(a, (torch.zeros(1, a.Nglo + 56 * 56, a.num_heads * a.head_dim),), None)
        assert a.__flops__ == ref["macs_56x56"] > 0
    # no CPU path: the MsViT with the B200 class refuses CPU tensors loudly
    with pytest.raises(RuntimeError, match="no CPU"):
        net.eval()(torch.zeros(1, 3, 224, 224))


def test_dropin_nonshared_weights_and_rpe_state_dict():
    gold = load_golden("dropin_reference.pt")["nonshared"]
    DropIn = make_dropin_class(_StandIn)
    torch.manual_seed(1)
    mod = DropIn(autograd=False, **gold["kwargs"])
    assert sorted(mod.state_dict().keys()) == sorted(gold["state_dict"].keys())
    assert torch.equal(mod.relative_position_index, gold["state_dict"]["relative_position_index"])
    mod.load_state_dict(gold["state_dict"], strict=True)
    assert mod.query is not mod.query_global


def test_dropin_mro_never_runs_the_base_constructor():
    DropIn = make_dropin_class(_StandIn)
    m = DropIn(32, num_heads=2, w=4, nglo=1, sharew=True, rpe=True)
    assert isinstance(m, _StandIn) and isinstance(m, B200Long2DSCSelfAttention)
    assert DropIn.__name__ == "B200_StandIn"
    assert len(list(m.parameters())) == len(list(B200Long2DSCSelfAttention(32, num_heads=2, w=4, nglo=1, sharew=True, rpe=True).parameters()))


@pytest.mark.gpu
def test_dropin_class_runs_on_gpu():
    DropIn = make_dropin_class(_StandIn)
    kw = dict(dim=96, num_heads=3, qkv_bias=True, w=7, nglo=1, sharew=True, rpe=False)
    torch.manual_seed(0)
    a = B200Long2DSCSelfAttention(**kw).cuda().bfloat16()
    b = DropIn(**kw).cuda().bfloat16()
    b.load_state_dict(a.state_dict())
    x = torch.randn(2, 1 + 14 * 14, 96, device="cuda", dtype=torch.bfloat16)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ya, yb = a(xa, 14, 14), b(xb, 14, 14)
    ya.sum().backward()
    yb.sum().backward()
    assert torch.equal(ya, yb) and torch.equal(xa.grad, xb.grad)
