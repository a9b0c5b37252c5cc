"""Generate golden vectors by IMPORTING THE UNMODIFIED REFERENCE (a checkout of microsoft/vision-longformer).

    python oracle/make_golden.py <vision-longformer checkout>

Outputs small fixtures under tests/golden/*.pt which ARE committed, so that the
test-suite never needs the reference itself.

What is pinned
--------------
* `attn_*.pt`  : `Long2DSCSelfAttention` (src/models/layers/longformer2d.py:12)
  built exactly like `AttnBlock` builds it for ATTN_TYPE='longformerhand'
  (src/models/msvit.py:269-276: autograd=False), float64 on CPU (the
  `@autocast()` decorators of slidingchunk_2d.py:203,235 are inert on CPU).
  Stored: ctor kwargs, state_dict, x, y=forward(x,nx,ny), dL/dx and all
  parameter grads for L = sum(y * gy), plus the tensors at the core-op seam
  (outputs of the q / kv Linears and the inputs of proj / proj_global) so the
  fused op can be checked without the Linears.
* `msvit_*.pt` : a tiny `MsViT` (src/models/msvit.py:343) forward + loss grads,
  pinning the stock-PyTorch harness in vision_longformer_b200/msvit.py.
* `mask_*.pt`  : raw outputs of the three reference mask builders
  (slidingchunk_2d.py:249-318) for the oracle's closed forms.
* `dropin_reference.pt` : what the reference MsViT and `Long2DSCSelfAttention`
  expose to a drop-in class (state_dict keys / shapes, public attributes, MAC
  counts), for tests/test_dropin_reference.py.
* `reference_fresh_seed.pt` : one more `Long2DSCSelfAttention` forward at a
  configuration none of the `attn_*.pt` cases uses, for the oracle.
"""
import os
import random
import sys
import types

import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def install_timm_shim():
    """timm is not installed; the reference only needs three helpers from it
    (src/models/layers/longformer2d.py:8, src/models/msvit.py:6)."""
    if "timm" in sys.modules:
        return
    layers = types.ModuleType("timm.models.layers")
    layers.trunc_normal_ = torch.nn.init.trunc_normal_
    layers.to_2tuple = lambda v: tuple(v) if isinstance(v, (tuple, list)) else (v, v)

    class DropPath(torch.nn.Module):
        def __init__(self, p=0.):
            super().__init__()
            self.p = p

        def forward(self, x):
            if self.p == 0. or not self.training:
                return x
            keep = 1 - self.p
            m = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
            return x.div(keep) * m
    layers.DropPath = DropPath
    timm = types.ModuleType("timm")
    models = types.ModuleType("timm.models")
    timm.models, models.layers = models, layers
    sys.modules.update({"timm": timm, "timm.models": models, "timm.models.layers": layers})


def import_reference(checkout):
    install_timm_shim()
    src = os.path.join(os.path.abspath(checkout), "src")
    if src not in sys.path:
        sys.path.insert(0, src)
    from models.layers.longformer2d import Long2DSCSelfAttention
    from models.layers import slidingchunk_2d
    from models.msvit import MsViT
    return Long2DSCSelfAttention, slidingchunk_2d, MsViT


ATTN_CASES = {
    # name: (B, nx, ny, ctor kwargs, train_mode_pick)
    "w7_g1_exact0_rpe":      (2, 14, 14, dict(dim=32, num_heads=2, w=7, nglo=1, exact=0, rpe=True, sharew=True), None),
    "w7_g1_exact1_rpe":      (2, 14, 14, dict(dim=32, num_heads=2, w=7, nglo=1, exact=1, rpe=True, sharew=True), None),
    "w4_g2_exact1_rpe_pad":  (2, 10, 9, dict(dim=24, num_heads=3, w=4, nglo=2, exact=1, rpe=True, sharew=True), None),
    "w4_g2_exact0_norpe_nosharew": (2, 10, 9, dict(dim=24, num_heads=3, w=4, nglo=2, exact=0, rpe=False, sharew=False), None),
    "w4_g1_cyclic_rpe_pad":  (2, 10, 9, dict(dim=16, num_heads=2, w=4, nglo=1, exact=-1, rpe=True, sharew=True), None),
    "w4_g1_cyclic_small":    (1, 8, 5, dict(dim=16, num_heads=2, w=4, nglo=1, exact=-1, rpe=True, sharew=True), None),
    "w4_g1_modeneg1_rpe_pad": (2, 10, 9, dict(dim=16, num_heads=2, w=4, nglo=1, exact=0, rpe=True, sharew=True, mode=-1), None),
    "w4_g2_mode3_rpe_pad":   (2, 10, 9, dict(dim=16, num_heads=2, w=4, nglo=2, exact=0, rpe=True, sharew=True, mode=1), 3),
    "w4_g1_mode6_norpe_pad": (2, 9, 10, dict(dim=16, num_heads=2, w=4, nglo=1, exact=0, rpe=False, sharew=True, mode=1), 6),
    "w5_g0_exact0_rpe":      (1, 12, 13, dict(dim=16, num_heads=2, w=5, nglo=0, exact=0, rpe=True, sharew=False), None),
    "w8_g1_exact0_d32":      (1, 24, 16, dict(dim=64, num_heads=2, w=8, nglo=1, exact=0, rpe=False, sharew=True), None),
    "w7_g1_exact0_d64_28":   (1, 28, 28, dict(dim=64, num_heads=1, w=7, nglo=1, exact=0, rpe=True, sharew=True), None),
}


def gen_attn(name, B, nx, ny, kw, pick, Cls):
    torch.manual_seed(300)   # the reference tests' seed (src/tests/test_slidingchunk_2d.py:56-60)
    mod = Cls(qkv_bias=True, autograd=False, **kw)
    # give the bias tables visible magnitude so the parity check is not vacuous
    with torch.no_grad():
        for n, p in mod.named_parameters():
            if "relative_position" in n:
                p.normal_(0, 0.5)
    mod = mod.double()      # parameters / inputs are fp32-representable, the math is fp64
    g = kw["nglo"]
    x = torch.randn(B, g + nx * ny, kw["dim"]).double().requires_grad_(True)
    seam = {}
    def grab(key, pick_input):
        def hook(m, i, o):          # first call only (sharew re-uses the Linears for the global rows)
            if key not in seam:
                seam[key] = (i[0] if pick_input else o).detach().clone()
        return hook
    hooks = [mod.query.register_forward_hook(grab("q_lin", False)),
             mod.kv.register_forward_hook(grab("kv_lin", False)),
             mod.proj.register_forward_hook(grab("proj_in", True))]
    if pick is not None:       # pin the random-shift mode the reference draws (longformer2d.py:118)
        mod.train()
        orig = random.randrange
        random.randrange = lambda *a, **k: pick
    else:
        mod.eval()
    try:
        y = mod(x, nx, ny)
    finally:
        if pick is not None:
            random.randrange = orig
    gy = torch.randn(y.shape).double()
    (y * gy).sum().backward()
    for h in hooks:
        h.remove()

    def small(t):           # exact for the fp32-representable inputs; 6e-8 rounding for derived tensors
        return t.detach().to(torch.int32 if t.dtype == torch.int64 else torch.float32).clone()
    out = dict(name=name, B=B, nx=nx, ny=ny, kwargs=dict(qkv_bias=True, **kw), picked_mode=pick,
               state_dict={k: small(v) for k, v in mod.state_dict().items()},
               x=small(x), gy=small(gy), y=y.detach().clone(), dx=x.grad.clone(),
               param_grads={n: small(p.grad) for n, p in mod.named_parameters() if p.grad is not None},
               seam={"proj_in": small(seam["proj_in"])})
    torch.save(out, os.path.join(OUT, f"attn_{name}.pt"))
    print("wrote attn_%s  y.norm=%.4f" % (name, y.norm().item()))


MSVIT_CASES = {
    "tiny_rpe": dict(arch="l1,h2,d16,n1,s1,g1,p4,f4,a0_l2,h2,d32,n2,s1,g1,p2,f4,a0_l3,h4,d48,n2,s0,g1,p2,f7,a0_l4,h4,d64,n1,s0,g0,p2,f7,a0",
                     img_size=64),
    "tiny_ape": dict(arch="l1,h2,d16,n1,s1,g1,p4,f4_l2,h2,d32,n1,s1,g2,p2,f4_l3,h4,d48,n1,s0,g1,p2,f7_l4,h4,d64,n1,s0,g0,p2,f7",
                     img_size=64),
}


def gen_msvit(name, kw, MsViT):
    torch.manual_seed(300)
    net = MsViT(num_classes=10, attn_type="longformerhand", sharew=True, norm_embed=True, ln_eps=1e-6,
                drop_path_rate=0.0, **kw).double().eval()
    x = torch.randn(2, 3, kw["img_size"], kw["img_size"]).double().requires_grad_(True)
    y = net(x)
    gy = torch.randn(y.shape).double()
    (y * gy).sum().backward()
    grads = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
    keep = sorted(grads)[::7]          # a spread of parameter grads, to bound the file size
    out = dict(name=name, kwargs=dict(num_classes=10, attn_type="longformerhand", sharew=True, norm_embed=True,
                                      ln_eps=1e-6, drop_path_rate=0.0, **kw),
               state_dict={k: (v.detach().to(torch.int32) if v.dtype == torch.int64 else v.detach().float())
                           for k, v in net.state_dict().items()},
               x=x.detach().float(), y=y.detach().clone(), gy=gy, dx=x.grad.clone(),
               param_grads={n: grads[n].float() for n in keep}, n_params=sum(p.numel() for p in net.parameters()))
    torch.save(out, os.path.join(OUT, f"msvit_{name}.pt"))
    print("wrote msvit_%s  params=%d" % (name, out["n_params"]))


def gen_masks(sc):
    out = {}
    for (nx, ny, w) in [(14, 14, 7), (10, 9, 4), (8, 5, 4), (16, 24, 8), (5, 5, 5)]:
        padx, pady = (w - nx % w) % w, (w - ny % w) % w
        mx, my = (nx + padx) // w, (ny + pady) // w
        for nm, fn in [("zero", sc._get_invalid_locations_mask_zero), ("exact", sc._get_invalid_locations_mask_exact),
                       ("cyclic", sc._get_invalid_locations_mask_cyclic)]:
            mask, ninv = fn(mx, my, padx, pady, w, "cpu")
            out[(nm, nx, ny, w)] = (mask.clone(), int(ninv))
    torch.save(out, os.path.join(OUT, "masks.pt"))
    print("wrote masks.pt", len(out))


# a 224x224 MsViT with two longformer stages (s1) and two dense ones, built the way `build_model` builds ViL
DROPIN_MSVIT = dict(arch="l1,h1,d48,n1,s1,g1,p4,f7_l2,h3,d96,n1,s1,g1,p2,f7_l3,h3,d192,n2,s0,g1,p2,f7_l4,h6,d384,n1,s0,g0,p2,f7",
                    img_size=224, num_classes=10, drop_path_rate=0.1, norm_embed=True, sharew=True,
                    attn_type="longformerhand", sw_exact=0, mode=1, ln_eps=1e-6)
# public attributes of Long2DSCSelfAttention that the rest of the reference reads
DROPIN_ATTRS = ("Nglo", "num_heads", "head_dim", "attention_window", "only_glo", "scale", "exact", "rpe")


def gen_dropin(Cls, MsViT):
    """What a drop-in class must reproduce: the stock MsViT's state_dict layout and parameter count, the attributes and
    the MAC count (compute_macs, longformer2d.py:231-280, at a 56x56 token grid) of each longformer attention, and the
    state_dict of a non-shared-weight, rpe, exact=1 module."""
    torch.manual_seed(0)
    net = MsViT(**DROPIN_MSVIT)
    attn = []
    for m in net.modules():
        if isinstance(m, Cls):
            m.__flops__ = 0
            Cls.compute_macs(m, (torch.zeros(1, m.Nglo + 56 * 56, m.num_heads * m.head_dim),), None)
            attn.append(dict({a: getattr(m, a) for a in DROPIN_ATTRS}, macs_56x56=m.__flops__))
    sd = net.state_dict()
    first = {}                  # sharew: the global-token Linears ARE the local ones, so their entries share storage
    tied = {k: first.setdefault(v.data_ptr(), k) for k, v in sd.items()}
    msvit = dict(kwargs=DROPIN_MSVIT, attn=attn, n_params=sum(p.numel() for p in net.parameters()),
                 state_dict={k: (tuple(v.shape), v.dtype) for k, v in sd.items()}, tied={k: t for k, t in tied.items() if t != k})
    kw = dict(dim=48, num_heads=3, qkv_bias=True, w=4, nglo=2, sharew=False, rpe=True, exact=1, mode=0)
    torch.manual_seed(1)
    ref = Cls(autograd=False, **kw)
    nonshared = dict(kwargs=kw, state_dict={k: v.detach().clone() for k, v in ref.state_dict().items()})
    torch.save(dict(msvit=msvit, nonshared=nonshared), os.path.join(OUT, "dropin_reference.pt"))
    print("wrote dropin_reference.pt  attn modules=%d" % len(attn))


def gen_fresh_seed(Cls):
    """Float64 eval forward at a configuration (w=3, two global tokens, rpe, separate global weights, 8x10) that the attn_*
    cases do not cover."""
    torch.manual_seed(1234)
    kw = dict(dim=24, num_heads=2, w=3, nglo=2, exact=0, rpe=True, sharew=False, qkv_bias=True)
    ref = Cls(autograd=False, **kw).double().eval()
    x = torch.randn(2, 2 + 8 * 10, 24, dtype=torch.float64)
    with torch.no_grad():
        y = ref(x, 8, 10)
    out = dict(kwargs=kw, nx=8, ny=10, state_dict={k: v.detach().clone() for k, v in ref.state_dict().items()}, x=x, y=y)
    torch.save(out, os.path.join(OUT, "reference_fresh_seed.pt"))
    print("wrote reference_fresh_seed.pt  y.norm=%.4f" % y.norm().item())


def main(checkout):
    os.makedirs(OUT, exist_ok=True)
    Cls, sc, MsViT = import_reference(checkout)
    gen_masks(sc)
    for name, (B, nx, ny, kw, pick) in ATTN_CASES.items():
        gen_attn(name, B, nx, ny, kw, pick, Cls)
    for name, kw in MSVIT_CASES.items():
        gen_msvit(name, kw, MsViT)
    gen_dropin(Cls, MsViT)
    gen_fresh_seed(Cls)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
