"""`segmentron._C` drop-in (segmentron_b200/c_shim.py over csrc/ca_nchw.cu): the four functions of the reference's pybind module
(segmentron/modules/csrc/vision.cpp:6-11, ca.h:25-72).

CPU part: the module object exposes exactly the four names, CPU tensors raise the reference's "Not implemented on the CPU".
GPU part (through the C ABI):
  * each function against the oracle's restatement (oracle/segref.py ca_weight / ca_map, pinned to a scalar transcription of
    ca_cuda.cu by tests/golden) and, for the two backward functions, against autograd through that restatement -- fp32 to 1e-5 of
    the output's max, fp16 / bf16 on 16-bit-representable inputs to 2^-10 / 2^-7;
  * CrissCrossAttention (cc_attention.py:11-72) with the four functions on the shim, differentiated the way the reference's
    autograd Functions _CAWeight / _CAMap do -- forward and every gradient against the oracle and against the reference's own
    module, stored in tests/golden/cca_module.pt;
  * CCNet (models/ccnet.py) with its criss-cross attention on the shim, against the committed fixture of the reference's model,
    tests/golden/ccnet_resnet101_65x97.pt.
"""
import os

import pytest
import torch

from oracle import segref as R

G = os.path.join(os.path.dirname(__file__), "golden")


def test_shim_surface_cpu():
    from segmentron_b200 import c_shim
    m = c_shim.make_module()
    assert sorted(n for n in dir(m) if n.startswith("ca_")) == ["ca_backward", "ca_forward", "ca_map_backward", "ca_map_forward"]
    t = torch.zeros(1, 8, 4, 5)
    for call in (lambda: m.ca_forward(t, t), lambda: m.ca_backward(torch.zeros(1, 8, 4, 5), t, t),
                 lambda: m.ca_map_forward(torch.zeros(1, 8, 4, 5), t), lambda: m.ca_map_backward(t, torch.zeros(1, 8, 4, 5), t)):
        with pytest.raises(RuntimeError, match="Not implemented on the CPU"):       # ca.h:34,46,58,70
            call()


def _rt(shape, seed, dtype):
    t = torch.randn(*shape, generator=torch.Generator().manual_seed(seed))
    return t.to(dtype).float()                          # representable in the kernel dtype


def _close(a, b, tol, what, floor=0.0):
    err = float((a.float().cpu() - b).abs().max() / max(float(b.abs().max()), floor, 1e-30))
    assert err <= tol, (what, err, tol)
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.float16, 2.0 ** -10), (torch.bfloat16, 2.0 ** -7)],
                         ids=["f32", "f16", "bf16"])
@pytest.mark.parametrize("shape", [(2, 8, 5, 7), (1, 64, 33, 49), (2, 16, 40, 129), (1, 3, 1, 37), (1, 5, 33, 1)],
                         ids=lambda s: "x".join(map(str, s)))
def test_c_functions_vs_oracle(shape, dtype, tol):
    from segmentron_b200 import c_shim as S
    n, c, h, w = shape
    t, f = _rt(shape, 1, dtype), _rt(shape, 2, dtype)
    g = _rt((n, 2 * c, h, w), 3, dtype)
    a = torch.softmax(_rt((n, h + w - 1, h, w), 4, torch.float32), 1).to(dtype).float()
    dwt = _rt((n, h + w - 1, h, w), 5, dtype)
    dout = _rt((n, 2 * c, h, w), 6, dtype)
    dev = lambda v: v.to("cuda", dtype)                     # noqa: E731
    # ca_forward / ca_map_forward
    _close(S.ca_forward(dev(t), dev(f)), R.ca_weight(t, f), tol, "ca_forward")
    _close(S.ca_map_forward(dev(a), dev(g)), R.ca_map(a, g), tol, "ca_map_forward")
    # ca_backward == autograd of ca_weight;  ca_map_backward == autograd of ca_map
    tt, ff = t.clone().requires_grad_(), f.clone().requires_grad_()
    R.ca_weight(tt, ff).backward(dwt)
    dt_, df_ = S.ca_backward(dev(dwt), dev(t), dev(f))
    _close(dt_, tt.grad, tol, "ca_backward dt")
    _close(df_, ff.grad, tol, "ca_backward df")
    aa, gg = a.clone().requires_grad_(), g.clone().requires_grad_()
    R.ca_map(aa, gg).backward(dout)
    dw_, dg_ = S.ca_map_backward(dev(dout), dev(a), dev(g))
    _close(dw_, aa.grad, tol, "ca_map_backward dw")
    _close(dg_, gg.grad, tol, "ca_map_backward dg")
    # non-contiguous inputs are accepted like the reference's (.contiguous() inside, ca_cuda.cu:205-207)
    tn = dev(t).permute(0, 1, 3, 2).contiguous().permute(0, 1, 3, 2)
    assert not tn.is_contiguous() or h == 1 or w == 1
    _close(S.ca_forward(tn, dev(f)), R.ca_weight(t, f), tol, "ca_forward (strided input)")


class _CAWeight(torch.autograd.Function):
    """ca_weight differentiated through the shim's ca_forward / ca_backward, the calls the reference's _CAWeight makes."""
    @staticmethod
    def forward(ctx, t, f):
        from segmentron_b200 import c_shim as S
        ctx.save_for_backward(t, f)
        return S.ca_forward(t, f)

    @staticmethod
    def backward(ctx, dw):
        from segmentron_b200 import c_shim as S
        return S.ca_backward(dw, *ctx.saved_tensors)


class _CAMap(torch.autograd.Function):
    """ca_map differentiated through the shim's ca_map_forward / ca_map_backward, the calls the reference's _CAMap makes."""
    @staticmethod
    def forward(ctx, weight, g):
        from segmentron_b200 import c_shim as S
        ctx.save_for_backward(weight, g)
        return S.ca_map_forward(weight, g)

    @staticmethod
    def backward(ctx, dout):
        from segmentron_b200 import c_shim as S
        return S.ca_map_backward(dout, *ctx.saved_tensors)


def _oracle_on_shim(monkeypatch):
    """From here on the oracle's ca_weight / ca_map are served by the shim (GPU only), with TF32 off for the oracle's 1x1 convs."""
    monkeypatch.setattr(R, "ca_weight", _CAWeight.apply)
    monkeypatch.setattr(R, "ca_map", _CAMap.apply)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)


@pytest.mark.gpu
def test_cca_autograd_on_the_shim_matches_reference_module(monkeypatch):
    """CrissCrossAttention forward and every gradient with its four `_C` functions on the shim, against the CPU oracle and against
    the reference's own module and autograd Functions (cc_attention.py:11-72), stored in tests/golden/cca_module.pt."""
    fx = torch.load(os.path.join(G, "cca_module.pt"))
    n, c, h, w = fx["shape"]
    P = R.Params(fx["params_seed"])
    x = torch.randn(n, c, h, w, generator=torch.Generator().manual_seed(fx["x_seed"]))
    dy = torch.randn(n, c, h, w, generator=torch.Generator().manual_seed(fx["dy_seed"]))
    with torch.no_grad():
        R.criss_cross_attention(P, x, "cca", gamma=fx["gamma"])             # creates the seeded parameters
    Pg = P.to("cuda:0")                 # the device the leaves live on, so that the oracle uses them as they are
    for k in P.t:
        P.t[k].requires_grad_()
        Pg.t[k] = Pg.t[k].detach().requires_grad_()
    xo = x.clone().requires_grad_()
    yo = R.criss_cross_attention(P, xo, "cca", gamma=fx["gamma"])          # fp32 oracle on the CPU
    yo.backward(dy)
    _oracle_on_shim(monkeypatch)
    xr = x.cuda().requires_grad_()
    yr = R.criss_cross_attention(Pg, xr, "cca", gamma=fx["gamma"])
    yr.backward(dy.cuda())
    refs = {"oracle": dict(y=yo.detach(), dx=xo.grad, grads={k: P.t["cca." + k].grad for k in fx["grads"]}),
            "reference": dict(y=fx["y"], dx=fx["dx"], grads=fx["grads"])}
    # fp32 on both sides, but cuDNN / cuBLAS and the CPU sum in different orders and the softmax sits on energies of O(10):
    # forward to 2e-5, gradients to 1e-3 of their max
    errs = {}
    for tag, ref in refs.items():
        errs[tag + " y"] = _close(yr.detach(), ref["y"], 2e-5, f"CrissCrossAttention forward vs {tag}")
        errs[tag + " dx"] = _close(xr.grad, ref["dx"], 1e-3, f"dx vs {tag}")
        wscale = float(ref["grads"]["value_conv.weight"].abs().max())
        for name, g in ref["grads"].items():
            # key_conv.bias: adding a constant to every key shifts all energies of a query equally -> the softmax, hence the loss, does
            # not depend on it; its gradient is pure rounding noise (1e-5) on both sides, so it is measured against the weight-gradient
            # scale
            mine = Pg.t["cca." + name].grad
            errs[f"{tag} d{name}"] = _close(mine, g.reshape(mine.shape), 1e-3, f"d{name} vs {tag}",
                                            floor=1e-3 * wscale if name == "key_conv.bias" else 0.0)
    print("\n[CrissCrossAttention on the segb200 _C shim] max-rel errors:", {k: f"{v:.1e}" for k, v in errs.items()})


@pytest.mark.gpu
def test_ccnet_on_the_shim_matches_reference_fixture(monkeypatch):
    """CCNet (models/ccnet.py, the model that needs `segmentron._C`) with its criss-cross attention on the shim: output == the
    committed fixture of the reference's own model, tests/golden/ccnet_resnet101_65x97.pt."""
    fx = torch.load(os.path.join(G, "ccnet_resnet101_65x97.pt"))
    P = R.build_params(fx["model"], fx["seed"]).to("cuda:0")
    x = torch.randn(*fx["shape"], generator=torch.Generator().manual_seed(fx["input_seed"]))
    _oracle_on_shim(monkeypatch)
    y = R.forward(fx["model"], P, x.cuda()).float().cpu()
    err = float((y - fx["y_ref"].float()).norm() / fx["y_ref"].float().norm())
    print(f"\n[CCNet on the segb200 _C shim] rel-L2 vs committed reference fixture: {err:.2e}")
    assert err < 1e-4, err
