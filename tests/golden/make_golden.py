"""Generate the golden fixtures that pin oracle/segref.py to the REAL reference.

Run in the build container only (needs /root/reference, read-only):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

For every case it (1) builds the oracle's seeded parameter dict, (2) builds the reference
nn.Module from its own YAML config / module class and ``load_state_dict(strict=True)``s that
dict (so key names and shapes are proven to be the reference's), (3) runs the reference on a
seeded input, (4) asserts the oracle reproduces it, and (5) stores the reference output
(fp16-compressed where large) in ``tests/golden/<case>.pt``.  One reference config per process
(the reference's ``cfg`` is a frozen global, SURVEY.md App. B10), hence the subprocess fan-out.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"

MODEL_CASES = {
    # case: (oracle model name, reference yaml, input shape, seed)
    "dlv3p_xception65_65x129": ("deeplabv3plus_xception65", "cityscapes_deeplabv3_plus.yaml", (1, 3, 65, 129), 0),
    "dlv3p_xception65_97x161_b2": ("deeplabv3plus_xception65", "cityscapes_deeplabv3_plus.yaml", (2, 3, 97, 161), 1),
    "dlv3p_mobilenetv2_64x128": ("deeplabv3plus_mobilenet_v2", "cityscapes_deeplabv3_plus_mobilenet.yaml", (1, 3, 64, 128), 2),
    "dlv3p_resnet101_65x129": ("deeplabv3plus_resnet101", "cityscapes_deeplabv3_plus_resnet.yaml", (1, 3, 65, 129), 4),
    "danet_resnet101_64x96": ("danet_resnet101", "cityscapes_danet_resnet.yaml", (1, 3, 64, 96), 5),
    "ccnet_resnet101_65x97": ("ccnet_resnet101", "cityscapes_ccnet_resnet.yaml", (1, 3, 65, 97), 6),
    "hrnet_w18s_128x192": ("hrnet_w18_small_v1", "cityscapes_hrnet_w18_small_v1.yaml", (2, 3, 128, 192), 7),
    "pspnet_resnet101_65x97": ("pspnet_resnet101", "cityscapes_pspnet_resnet.yaml", (1, 3, 65, 97), 8),
    "ocnet_resnet50_65x97": ("ocnet_resnet50", "cityscapes_ocnet.yaml", (1, 3, 65, 97), 9),
}


def run_model_case(case):
    import numpy as np
    np.int = int                                    # SURVEY App. B1
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    from oracle import segref as R
    name, yaml_file, shape, seed = MODEL_CASES[case]
    if name == "ccnet_resnet101":
        # The reference's CCNet needs the pybind module `segmentron._C`, which cannot be built (THC headers, App. B5) and
        # is commented out of models/__init__.py.  Provide a stand-in whose two forward functions are the oracle's
        # ca_weight / ca_map (themselves pinned to a scalar transcription of ca_cuda.cu in run_module_cases), so the
        # fixture pins the reference's MODEL structure (_RCCAModule, recurrence, cat order, bottleneck) around them.
        import types
        import segmentron
        fake = types.ModuleType("segmentron._C")
        fake.ca_forward = lambda t, f: R.ca_weight(t, f)
        fake.ca_map_forward = lambda w, g: R.ca_map(w, g)
        sys.modules["segmentron._C"] = fake
        segmentron._C = fake
        import segmentron.models.ccnet  # noqa: F401  (registers "CCNet")
    if name == "pspnet_resnet101":
        # The reference's PSPNet() cannot be constructed as shipped: _PSPHead passes norm_kwargs=None down to _ConvBNReLU, which has
        # no such parameter (pspnet.py:47 -> module.py:90 -> basic.py:66; SURVEY.md App. B2).  Harness-side workaround, outside the
        # reference tree: drop that one keyword in PyramidPooling's constructor.  No forward code is touched.
        import segmentron.modules.module as _mm
        _orig_init = _mm.PyramidPooling.__init__

        def _init(self, in_channels, sizes=(1, 2, 3, 6), norm_layer=torch.nn.BatchNorm2d, **kwargs):
            kwargs.pop("norm_kwargs", None)
            _orig_init(self, in_channels, sizes=sizes, norm_layer=norm_layer, **kwargs)
        _mm.PyramidPooling.__init__ = _init
    from segmentron.config import cfg
    from segmentron.models.model_zoo import get_segmentation_model
    cfg.update_from_file(os.path.join(REF, "configs", yaml_file))
    cfg.PHASE = "test"
    cfg.check_and_freeze()
    model = get_segmentation_model().eval()
    # tools/eval.py:50-53 : BN eps override for the encoder
    if cfg.MODEL.BN_EPS_FOR_ENCODER:
        for m in model.encoder.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.eps = cfg.MODEL.BN_EPS_FOR_ENCODER
    P = R.build_params(name, seed)
    missing = model.load_state_dict(P.state_dict(), strict=True)
    if name == "pspnet_resnet101":                      # two outputs (main, aux): check both, store the first
        g_ = torch.Generator().manual_seed(1000 + seed)
        x_ = torch.randn(*shape, generator=g_)
        with torch.no_grad():
            yr, yo = model(x_), R.forward(name, P, x_, all=True)
        assert len(yr) == 2
        for a_, b_ in zip(yr, yo):
            assert float((a_ - b_).abs().max() / a_.abs().max()) < 1e-5
    if name == "danet_resnet101":                       # three outputs (sasc, sa, sc): check all, store the first
        g_ = torch.Generator().manual_seed(1000 + seed)
        x_ = torch.randn(*shape, generator=g_)
        with torch.no_grad():
            yr, yo = model(x_), R.forward(name, P, x_, all=True)
        for a_, b_ in zip(yr, yo):
            assert float((a_ - b_).abs().max() / a_.abs().max()) < 1e-5
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.randn(*shape, generator=g)
    with torch.no_grad():
        y_ref = model(x)[0]
        y_orc = R.forward(name, P, x)
    err = float((y_ref - y_orc).abs().max() / y_ref.abs().max())
    assert err < 1e-5, f"oracle != reference for {case}: {err}"
    out = dict(case=case, model=name, seed=seed, input_seed=1000 + seed, shape=shape,
               y_ref=y_ref.contiguous(), argmax=y_ref.argmax(1).to(torch.uint8),
               oracle_vs_ref_maxrel=err, n_params=len(P.t))
    torch.save(out, os.path.join(HERE, case + ".pt"))
    print(f"{case}: oracle vs reference max-rel {err:.2e}; saved {tuple(y_ref.shape)}")


TRAIN_CASES = {
    # case: (oracle model name, reference yaml, input shape, seed)
    "train_dlv3p_resnet101_65x97_b4": ("deeplabv3plus_resnet101", "cityscapes_deeplabv3_plus_resnet.yaml", (4, 3, 65, 97), 21),
    "train_dlv3p_xception65_65x97_b4": ("deeplabv3plus_xception65", "cityscapes_deeplabv3_plus.yaml", (4, 3, 65, 97), 22),
    "train_dlv3p_mobilenetv2_64x96_b4": ("deeplabv3plus_mobilenet_v2", "cityscapes_deeplabv3_plus_mobilenet.yaml", (4, 3, 64, 96), 23),
    "train_ccnet_resnet101_65x97_b2": ("ccnet_resnet101", "cityscapes_ccnet_resnet.yaml", (2, 3, 65, 97), 24),
    "train_hrnet_w18s_64x96_b2": ("hrnet_w18_small_v1", "cityscapes_hrnet_w18_small_v1.yaml", (2, 3, 64, 96), 25),
    "train_danet_resnet101_64x96_b2": ("danet_resnet101", "cityscapes_danet_resnet.yaml", (2, 3, 64, 96), 26),
}


def grad_digest(grads, seed=12345):
    """Per-parameter (norm, projection on a seeded random direction): 2 numbers per tensor pin a gradient to ~1e-6 without
    storing 190 MB of them."""
    import torch
    out = {}
    for i, k in enumerate(sorted(grads)):
        g = grads[k].detach().double().flatten()
        r = torch.randn(g.numel(), generator=torch.Generator().manual_seed(seed + i), dtype=torch.float64)
        out[k] = (float(g.norm()), float((g * r).sum()))
    return out


def _install_oracle_c(R):
    """Install a CPU stand-in for `segmentron._C` whose four functions are the oracle's ca_weight / ca_map and their torch-autograd
    gradients (the reference's extension cannot be built, App. B5)."""
    import types
    import torch
    import segmentron

    def _vjp(fn, args, gout):
        with torch.enable_grad():
            leaves = [a.detach().requires_grad_(True) for a in args]
            out = fn(*leaves)
            return torch.autograd.grad(out, leaves, gout)
    fake = types.ModuleType("segmentron._C")
    fake.ca_forward = lambda t, f: R.ca_weight(t, f)
    fake.ca_map_forward = lambda w, g: R.ca_map(w, g)
    fake.ca_backward = lambda dw, t, f: _vjp(R.ca_weight, (t, f), dw)
    fake.ca_map_backward = lambda dout, w, g: _vjp(R.ca_map, (w, g), dout)
    sys.modules["segmentron._C"] = fake
    segmentron._C = fake


def run_train_case(case):
    """One training iteration of tools/train.py:135-147 on the REAL reference model (train mode, the reference's own
    criterion and optimizer) vs the oracle's loss_and_grads: loss, every parameter gradient, BatchNorm running statistics and
    the parameters after one optimizer.step() must agree."""
    import numpy as np
    np.int = int
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    from oracle import segref as R
    name, yaml_file, shape, seed = TRAIN_CASES[case]
    if name == "ccnet_resnet101":
        # `segmentron._C` cannot be built (App. B5): stand-in whose four functions are the oracle's ca_weight / ca_map and their
        # torch-autograd gradients (ca_weight / ca_map are pinned to a scalar transcription of ca_cuda.cu in run_module_cases),
        # so this fixture pins the reference's MODEL graph, its custom autograd Functions (cc_attention.py:11-45) and its
        # training recipe around them.
        _install_oracle_c(R)
        import segmentron.models.ccnet  # noqa: F401  (registers "CCNet")
    if name == "pspnet_resnet101":
        # The reference's PSPNet() cannot be constructed as shipped: _PSPHead passes norm_kwargs=None down to _ConvBNReLU, which has
        # no such parameter (pspnet.py:47 -> module.py:90 -> basic.py:66; SURVEY.md App. B2).  Harness-side workaround, outside the
        # reference tree: drop that one keyword in PyramidPooling's constructor.  No forward code is touched.
        import segmentron.modules.module as _mm
        _orig_init = _mm.PyramidPooling.__init__

        def _init(self, in_channels, sizes=(1, 2, 3, 6), norm_layer=torch.nn.BatchNorm2d, **kwargs):
            kwargs.pop("norm_kwargs", None)
            _orig_init(self, in_channels, sizes=sizes, norm_layer=norm_layer, **kwargs)
        _mm.PyramidPooling.__init__ = _init
    from segmentron.config import cfg
    from segmentron.models.model_zoo import get_segmentation_model
    cfg.update_from_file(os.path.join(REF, "configs", yaml_file))
    cfg.PHASE = "test"                                   # only suppresses the pretrained-weights download (App. B9)
    cfg.check_and_freeze()
    from segmentron.solver.loss import get_segmentation_loss
    from segmentron.solver.optimizer import get_optimizer
    model = get_segmentation_model()
    P = R.build_params(name, seed)
    model.load_state_dict(P.state_dict(), strict=True)
    model.train()
    n, _, h, w = shape
    g = torch.Generator().manual_seed(2000 + seed)
    x = torch.randn(*shape, generator=g)
    target = torch.randint(-1, 19, (n, h, w), generator=g)
    criterion = get_segmentation_loss(cfg.MODEL.MODEL_NAME, use_ohem=cfg.SOLVER.OHEM, aux=cfg.SOLVER.AUX,
                                      aux_weight=cfg.SOLVER.AUX_WEIGHT, ignore_index=-1)
    optimizer = get_optimizer(model)
    # Dropout2d mask: torch draws a [N,C,1,1] Bernoulli(0.9) tensor; re-create it from the same RNG state for the oracle
    mask_c, mask_key = (512, "head.rcca.bottleneck.dropout") if name == "ccnet_resnet101" else (256, "head.aspp.dropout")
    torch.manual_seed(777)
    mask = torch.empty(n, mask_c, 1, 1).bernoulli_(0.9) / 0.9         # (unused by the ASPP-less MobileNetV2 head)
    more_masks = {}
    if name == "danet_resnet101":                                    # three Dropout2d(0.1): conv6, conv7, conv8 in call order
        torch.manual_seed(777)
        for key in ("head.conv6.0", "head.conv7.0", "head.conv8.0"):
            more_masks[key] = torch.empty(n, 512, 1, 1).bernoulli_(0.9) / 0.9
        mask, mask_key = more_masks["head.conv6.0"], "head.conv6.0"
    torch.manual_seed(777)
    outputs = model(x)
    loss = sum(criterion(outputs, target).values())
    optimizer.zero_grad()
    loss.backward()
    ref_grads = {k: v.grad.detach().clone() for k, v in model.named_parameters() if v.grad is not None}
    P.dropout_masks[mask_key] = mask
    P.dropout_masks.update(more_masks)
    # MODEL.BN_MOMENTUM (None -> torch's 0.1) is applied to every BatchNorm by get_optimizer (solver/optimizer.py:37-39); the
    # HRNet YAML sets 0.01
    bn_momentum = float(cfg.MODEL.BN_MOMENTUM) if cfg.MODEL.BN_MOMENTUM else 0.1
    P.bn_momentum = bn_momentum
    o_loss, o_grads, o_out, o_low = R.loss_and_grads(name, P, x, target)
    assert abs(float(loss) - float(o_loss)) < 1e-5 * abs(float(loss)), (float(loss), float(o_loss))
    worst = 0.0
    gmax = max(float(v.norm()) for v in ref_grads.values())       # floor: analytically-zero gradients are rounding noise
    for k, gr in ref_grads.items():
        e = float((gr - o_grads[k]).norm() / (gr.norm() + 1e-6 * gmax))
        worst = max(worst, e)
        assert e < 2e-4, f"grad mismatch {k}: {e}"
    assert set(ref_grads) == set(k for k in o_grads if float(o_grads[k].abs().max()) > 0 or k in ref_grads)
    sd = model.state_dict()
    for k in sd:
        if k.endswith(("running_mean", "running_var")):
            e = float((sd[k] - P.t[k]).abs().max())
            assert e < 1e-5, f"running stat mismatch {k}: {e}"
    optimizer.step()
    lrs = {}
    for gi, grp in enumerate(optimizer.param_groups):
        for q in grp["params"]:
            lrs[id(q)] = (grp["lr"], grp["weight_decay"], grp["momentum"])
    hyper = {k: lrs[id(v)] for k, v in model.named_parameters() if id(v) in lrs}
    stepped = {k: v.detach().clone() for k, v in model.named_parameters()}
    small = ["encoder.conv1.weight", "encoder.bn1.weight", "encoder.bn1.bias",
             "encoder.layer4.2.bn3.weight" if "resnet" in name else "encoder.block21.sep_conv3.block.bn_point.weight",
             "head.block.2.weight", "head.block.2.bias", "head.aspp.image_pooling.bn.weight", "head.c1_block.bn.bias"]
    if name == "ccnet_resnet101":
        small = ["encoder.conv1.weight", "head.rcca.cca.gamma", "head.rcca.cca.query_conv.weight", "head.rcca.cca.key_conv.bias",
                 "head.out.weight", "head.out.bias", "head.rcca.bottleneck.1.weight"]
    if "danet" in name:
        small = ["encoder.conv1.weight", "encoder.layer4.2.bn2.weight", "head.conv5a.1.weight", "head.sa.gamma", "head.sa.query_conv.weight",
                 "head.sa.key_conv.bias", "head.sa.value_conv.bias", "head.sc.gamma", "head.conv52.1.weight", "head.conv6.1.weight",
                 "head.conv7.1.bias", "head.conv8.1.weight"]
    if "hrnet" in name:
        small = ["encoder.conv1.weight", "encoder.bn2.bias", "encoder.layer1.0.conv3.weight", "encoder.transition1.1.0.0.weight",
                 "encoder.stage2.0.fuse_layers.0.1.0.weight", "encoder.stage4.0.fuse_layers.3.0.1.0.weight",
                 "encoder.stage4.0.fuse_layers.3.0.1.1.bias", "encoder.stage4.0.branches.3.1.conv2.weight",
                 "hrnet_head.last_layer.0.weight", "hrnet_head.last_layer.0.bias", "hrnet_head.last_layer.1.weight",
                 "hrnet_head.last_layer.3.weight", "hrnet_head.last_layer.3.bias"]
    if "mobilenet" in name:
        small = ["encoder.conv1.conv.weight", "encoder.conv1.bn.weight", "encoder.block5.3.conv.3.bias", "head.block.2.weight",
                 "head.block.2.bias", "head.block.0.block.depthwise.weight"]
    out = dict(case=case, model=name, seed=seed, input_seed=2000 + seed, shape=shape, loss=float(loss), mask=mask, mask_key=mask_key,
               low=outputs[0].detach()[:, :, ::8, ::8].contiguous(), digest=grad_digest(ref_grads),
               grads_small={k: ref_grads[k] for k in small}, hyper=hyper, stepped_digest=grad_digest(stepped, 999),
               running={k: sd[k].clone() for k in sd if k.endswith(("running_mean", "running_var")) and
                        (k.startswith("encoder.bn1") or "image_pooling" in k or "layer4.2.bn3" in k or "block21.sep_conv3.block.bn_point" in k
                         or k.startswith("encoder.conv1.bn") or "block5.3.conv.3" in k or "hrnet_head.last_layer.1" in k
                         or "stage4.0.fuse_layers.3.0.1.1" in k)},
               bn_momentum=bn_momentum, more_masks=more_masks, oracle_vs_ref_worst_grad_rel=worst)
    torch.save(out, os.path.join(HERE, case + ".pt"))
    print(f"{case}: loss {float(loss):.6f}; worst grad rel-L2 oracle vs reference {worst:.2e}; {len(ref_grads)} grads")


def run_module_cases():
    """Module-level fixtures: PAM, CAM, PyramidPooling from the reference classes; criss-cross
    attention from a line-by-line python transcription of ca_cuda.cu's index map (the CUDA
    extension cannot be built: THC headers are gone, SURVEY App. B5)."""
    import numpy as np
    np.int = int
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    from oracle import segref as R
    from segmentron.modules.module import PAM_Module, CAM_Module, PyramidPooling
    out = {}
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2, 64, 12, 20, generator=g)
    # PAM
    P = R.Params(11)
    with torch.no_grad():
        y_o = R.pam(P, x, "pam")
        m = PAM_Module(64).eval()
        m.load_state_dict({k[len("pam."):]: v for k, v in P.state_dict().items()}, strict=True)
        y_r = m(x)
    assert float((y_r - y_o).abs().max()) < 1e-4
    out["pam"] = dict(x=x, y=y_r, seed=11)
    # CAM
    P = R.Params(12)
    with torch.no_grad():
        y_o = R.cam(P, x * 0.2, "cam")
        m = CAM_Module(64).eval()
        m.load_state_dict({k[len("cam."):]: v for k, v in P.state_dict().items()}, strict=True)
        y_r = m(x * 0.2)
    assert float((y_r - y_o).abs().max()) < 1e-4
    out["cam"] = dict(x=x * 0.2, y=y_r, seed=12)
    # PyramidPooling (PSPNet() itself cannot be constructed: App. B2)
    P = R.Params(13)
    xp = torch.randn(1, 64, 17, 33, generator=g)
    with torch.no_grad():
        y_o = R.pyramid_pooling(P, xp, "psp")
        m = PyramidPooling(64).eval()
        m.load_state_dict({k[len("psp."):]: v for k, v in P.state_dict().items()}, strict=True)
        y_r = m(xp)
    assert float((y_r - y_o).abs().max()) < 1e-4
    out["psp"] = dict(x=xp, y=y_r, seed=13)
    # criss-cross: scalar loops written from ca_cuda.cu:8-36 and :94-120
    n, c, h, w = 1, 4, 5, 7
    t = torch.randn(n, c, h, w, generator=g); f = torch.randn(n, c, h, w, generator=g)
    wgt = torch.zeros(n, h + w - 1, h, w)
    for b in range(n):
        for y in range(h):
            for xx in range(w):
                for z in range(h + w - 1):
                    for pl in range(c):
                        if z < w:
                            wgt[b, z, y, xx] += t[b, pl, y, xx] * f[b, pl, y, z]
                        else:
                            i = z - w
                            j = i if i < y else i + 1
                            wgt[b, w + i, y, xx] += t[b, pl, y, xx] * f[b, pl, j, xx]
    assert float((wgt - R.ca_weight(t, f)).abs().max()) < 1e-5
    gv = torch.randn(n, 6, h, w, generator=g)
    att = torch.softmax(wgt, 1)
    o = torch.zeros(n, 6, h, w)
    for b in range(n):
        for pl in range(6):
            for y in range(h):
                for xx in range(w):
                    for i in range(w):
                        o[b, pl, y, xx] += gv[b, pl, y, i] * att[b, i, y, xx]
                    for i in range(h):
                        if i == y:
                            continue
                        j = i if i < y else i - 1
                        o[b, pl, y, xx] += gv[b, pl, i, xx] * att[b, w + j, y, xx]
    assert float((o - R.ca_map(att, gv)).abs().max()) < 1e-5
    out["cca"] = dict(t=t, f=f, weight=wgt, g=gv, att=att, out=o)
    torch.save(out, os.path.join(HERE, "modules.pt"))
    print("modules: pam/cam/psp/cca OK")


def run_cca_module_case():
    """The reference's own CrissCrossAttention module and autograd Functions (cc_attention.py:11-72) on the oracle stand-in for
    `segmentron._C`: forward and every gradient for the seeded case of tests/test_c_shim.py, checked against the oracle and stored in
    tests/golden/cca_module.pt so that the GPU test compares the `segmentron._C` drop-in with the reference module without it."""
    import numpy as np
    np.int = int
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    from oracle import segref as R
    _install_oracle_c(R)
    from segmentron.modules.cc_attention import CrissCrossAttention
    n, c, h, w = 2, 64, 17, 23
    P = R.Params(7)
    x = torch.randn(n, c, h, w, generator=torch.Generator().manual_seed(8))
    dy = torch.randn(n, c, h, w, generator=torch.Generator().manual_seed(9))
    with torch.no_grad():
        R.criss_cross_attention(P, x, "cca", gamma=0.7)                 # creates the seeded parameters
    m = CrissCrossAttention(c)
    m.load_state_dict({k[len("cca."):]: v for k, v in P.t.items() if k.startswith("cca.")}, strict=True)
    xr = x.clone().requires_grad_()
    y = m(xr)
    y.backward(dy)
    y = y.detach()
    for k in P.t:
        P.t[k].requires_grad_()
    xo = x.clone().requires_grad_()
    yo = R.criss_cross_attention(P, xo, "cca", gamma=0.7)
    yo.backward(dy)
    yo = yo.detach()
    assert float((y - yo).abs().max() / yo.abs().max()) < 1e-5
    assert float((xr.grad - xo.grad).abs().max() / xo.grad.abs().max()) < 1e-4
    grads = {name: p.grad.detach().clone() for name, p in m.named_parameters()}
    out = dict(shape=(n, c, h, w), params_seed=7, x_seed=8, dy_seed=9, gamma=0.7, y=y, dx=xr.grad.detach(), grads=grads)
    torch.save(out, os.path.join(HERE, "cca_module.pt"))
    print(f"cca_module: reference CrissCrossAttention {tuple(y.shape)}, {len(grads)} parameter gradients")


if __name__ == "__main__":
    if len(sys.argv) > 1:
        c = sys.argv[1]
        (run_module_cases() if c == "modules" else run_cca_module_case() if c == "cca_module" else
         run_train_case(c) if c in TRAIN_CASES else run_model_case(c))
    else:
        env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
        for c in list(MODEL_CASES) + list(TRAIN_CASES) + ["modules", "cca_module"]:
            subprocess.check_call([sys.executable, os.path.abspath(__file__), c], env=env)
