"""GPU tests of the product model graph: against the golden fixture from the reference's own graph, against the oracle
network on fresh inputs, the cascade, a training step, and the mx shim's operator call style on the CUDA operators."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from maskflownet_b200 import _lib, network, ops  # noqa: E402
from oracle import network_ref  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, G)
from make_golden import named_init, seeded_images  # noqa: E402


@pytest.fixture(autouse=True)
def _fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


def _named_model(cls=network.MaskFlownetS):
    m = cls()
    with torch.no_grad():
        for k, p in m.named_parameters():
            p.copy_(named_init(k.replace("MaskFlownet_S.", ""), p.shape) if cls is network.MaskFlownetS
                    else named_init(k, p.shape))
    return m.cuda().eval()


def test_product_graph_matches_reference_graph_fixture():
    d = np.load(os.path.join(G, "net_ref_graph.npz"))
    model = _named_model()
    im1, im2 = seeded_images()
    n0 = _lib.launch_count()
    with torch.no_grad():
        preds, occ, srcs = model(im1.cuda(), im2.cuda(), want_cascade_inputs=True)
    # 5 correlations, 4 fused warps, 1 cascade-input kernel, 27 tensor-core convolutions (+ their one-time weight packs)
    assert _lib.launch_count() - n0 >= 5 + 4 + 1 + 27
    for k, p in zip(("pred6", "pred5", "pred4", "pred3", "pred2"), preds):
        err = np.abs(p.cpu().numpy() - d[k]).max()
        assert err < 2e-3, (k, err)                       # flows reach ~12 px; 2e-3 px absolute = 1e-4 * scale
    assert np.abs(occ[0].cpu().numpy() - d["occ"]).max() < 1e-4
    assert np.abs(srcs[4].cpu().numpy() - d["c40"].astype(np.float32)).max() < 3e-3


def test_product_graph_matches_oracle_network_batch2():
    model = _named_model()
    a1, a2 = seeded_images(seed=5, n=2, h=64, w=192)
    params = {k: v.detach().cpu() for k, v in model.named_parameters()}
    with torch.no_grad():
        preds = model(a1.cuda(), a2.cuda())[0]
        ref = network_ref.maskflownet_s_forward(params, a1, a2, threads=8)[0]
    for p, r in zip(preds, ref):
        assert (p.cpu() - r).abs().max().item() < 2e-3


def test_predict_flow_pipeline():
    model = _named_model()
    rng = np.random.default_rng(0)
    u1 = torch.from_numpy(rng.integers(0, 256, (1, 3, 64, 128), dtype=np.uint8))
    u2 = torch.from_numpy(rng.integers(0, 256, (1, 3, 64, 128), dtype=np.uint8))
    flow = network.predict_flow(model, u1.cuda(), u2.cuda())
    params = {k: v.detach().cpu() for k, v in model.named_parameters()}
    ref = network_ref.predict_flow(params, u1, u2, threads=8)
    assert flow.shape == (1, 2, 64, 128)
    assert (flow.cpu() - ref).abs().max().item() < 5e-3


def test_cascade_matches_reference_graph_fixture():
    """network.MaskFlownet == the reference's own MaskFlownet.hybrid_forward (network/MaskFlownet.py:443-545) run unchanged
    through the shim with the oracle's operators (tests/golden/net_ref_graph_cascade.npz): pins the dual pyramid, the md=2
    correlations, deform6 and the c2s quirk (:306).  Bound: 1e-4 relative to the flow scale (x20) = 2e-3 px."""
    d = np.load(os.path.join(G, "net_ref_graph_cascade.npz"))
    model = _named_model(network.MaskFlownet)
    assert sum(p.numel() for p in model.parameters()) == int(d["n_params"])
    im1, im2 = seeded_images()
    with torch.no_grad():
        preds, vis, _ = model(im1.cuda(), im2.cuda())
    errs = {}
    for k, p in zip(("pred6", "pred5", "pred4", "pred3", "pred2"), preds):
        errs[k] = float(np.abs(p.cpu().numpy() - d[k]).max())
    print("cascade max abs errors (px):", errs)
    assert max(errs.values()) < 2e-3, errs
    assert np.abs(vis[0].cpu().numpy() - d["vis"]).max() < 1e-4


def test_cascade_matches_oracle_network_fresh_inputs():
    model = _named_model(network.MaskFlownet)
    a1, a2 = seeded_images(seed=11, n=2, h=64, w=128)
    params = {k: v.detach().cpu() for k, v in model.named_parameters()}
    with torch.no_grad():
        preds = model(a1.cuda(), a2.cuda())[0]
        ref = network_ref.maskflownet_forward(params, a1, a2, threads=8)[0]
    for p, r in zip(preds, ref):
        assert (p.cpu() - r).abs().max().item() < 2e-3


def test_cascade_forward_runs_and_uses_md2_kernels():
    model = network.MaskFlownet().cuda().eval()
    a1, a2 = seeded_images(seed=7, n=1, h=64, w=128)
    n0 = _lib.launch_count()
    with torch.no_grad():
        preds, vis, _ = model(a1.cuda(), a2.cuda())
    assert [tuple(p.shape) for p in preds] == [(1, 2, 1, 2), (1, 2, 2, 4), (1, 2, 4, 8), (1, 2, 8, 16), (1, 2, 16, 32)]
    assert all(torch.isfinite(p).all() for p in preds)
    assert _lib.launch_count() - n0 >= 10 + 10 + 5   # S head (5 corr, 4 warp, 1 image warp) + cascade (10 corr, 5 warp) + convs


def test_training_step_gradients_flow_through_cuda_backward():
    model = _named_model().train()
    a1, a2 = seeded_images(seed=9, n=2, h=64, w=128)
    preds = model(a1.cuda(), a2.cuda())[0]
    loss = sum(w * p.square().mean() for w, p in zip((.005, .01, .02, .08, .32), preds))
    loss.backward()
    for name in ("deform5.weight", "deform2.bias", "conv2f.weight", "conv1a.weight", "pred_mask3.weight"):
        g = dict(model.named_parameters())[name].grad
        assert g is not None and torch.isfinite(g).all() and g.abs().max().item() > 0, name


def test_shim_operator_call_style_on_cuda():
    """The call style of network/MaskFlownet.py:195,230 and network/layer.py:17-18,119 through the F shim."""
    from maskflownet_b200.mx import ndarray as F
    from oracle import cref
    rng = np.random.default_rng(1)
    c1 = rng.standard_normal((1, 32, 8, 12)).astype(np.float32)
    c2 = rng.standard_normal((1, 32, 8, 12)).astype(np.float32)
    out = F.Correlation(F.NDArray(torch.from_numpy(c1).cuda()), F.NDArray(torch.from_numpy(c2).cuda()), pad_size=4,
                        kernel_size=1, max_displacement=4, stride1=1, stride2=1, is_multiply=1)
    assert np.abs(out.asnumpy() - cref.correlation_forward(c1, c2)).max() < 1e-4
    flow = F.NDArray(torch.from_numpy((rng.standard_normal((1, 2, 8, 12)) * 0.2).astype(np.float32)).cuda())
    w = (rng.standard_normal((32, 32, 3, 3)) * 0.1).astype(np.float32)
    offs = F.repeat(F.expand_dims(flow * 20. / 8, axis=1), 9, axis=1).reshape((0, -3, -2))
    warp = F.contrib.DeformableConvolution(F.NDArray(torch.from_numpy(c2).cuda()), offs,
                                           F.NDArray(torch.from_numpy(w).cuda()), name='fwd', kernel=(3, 3),
                                           stride=(1, 1), dilate=(1, 1), pad=(1, 1), num_filter=32, num_group=1,
                                           no_bias=True, layout='NCHW', num_deformable_group=1)
    assert np.abs(warp.asnumpy() - cref.deformable_conv_forward(c2, offs.asnumpy(), w, None)).max() < 1e-4
    img = rng.standard_normal((1, 3, 8, 12)).astype(np.float32)
    grid = F.GridGenerator(data=flow.flip(axis=1), transform_type="warp")
    rec = F.BilinearSampler(F.NDArray(torch.from_numpy(img).cuda()), grid)
    assert np.abs(rec.asnumpy() - cref.reconstruction2d(img, flow.asnumpy())).max() < 1e-4


def test_multiscale_epe_loss_matches_oracle_and_backprops():
    from maskflownet_b200 import losses
    from oracle import torch_ref
    rng = np.random.default_rng(3)
    H, W = 64, 128
    preds_np = [rng.standard_normal((2, 2, H // s, W // s)).astype(np.float32) for s in losses.SCALES]
    flow = rng.standard_normal((2, 2, H, W)).astype(np.float32)
    mask = (rng.random((2, 1, H, W)) > 0.3).astype(np.float32)
    gp = [torch.from_numpy(p).cuda().requires_grad_() for p in preds_np]
    rp = [torch.from_numpy(p).clone().requires_grad_() for p in preds_np]
    lg = losses.multiscale_epe(torch.from_numpy(flow).cuda(), torch.from_numpy(mask).cuda(), gp)
    lr = losses.multiscale_epe(torch.from_numpy(flow), torch.from_numpy(mask), rp, upsample=torch_ref.upsample)
    assert (lg.cpu() - lr).abs().max().item() < 1e-5
    lg.sum().backward()
    lr.sum().backward()
    for a, b in zip(gp, rp):
        assert (a.grad.cpu() - b.grad).abs().max().item() < 1e-6


@pytest.mark.gpu
def test_flow_predictor_cuda_graph_equals_eager():
    """network.FlowPredictor (predict_flow captured in a CUDA graph, static input buffers) returns exactly what the eager
    call returns, also when it is replayed with new inputs."""
    torch.manual_seed(3)
    model = network.MaskFlownetS().cuda().eval()
    pred = network.FlowPredictor(model)
    for seed in (0, 1):
        g = torch.Generator().manual_seed(seed)
        a = torch.randint(0, 256, (2, 3, 64, 128), generator=g, dtype=torch.uint8).cuda()
        b = torch.randint(0, 256, (2, 3, 64, 128), generator=g, dtype=torch.uint8).cuda()
        ref = network.predict_flow(model, a, b).clone()
        got = pred(a, b).clone()
        assert torch.equal(ref, got)



def test_predict_any_size_matches_oracle_pipeline():
    """network.predict (PipelineFlownet.predict: resize to x64, forward, Upsample(4), resize back, flip) on a 50x100 pair
    against the oracle network + oracle pre/post-processing."""
    from oracle import prepost_ref
    model = _named_model()
    rng = np.random.default_rng(3)
    u1 = rng.integers(0, 256, (1, 3, 50, 100), dtype=np.uint8)
    u2 = rng.integers(0, 256, (1, 3, 50, 100), dtype=np.uint8)
    flow, occ = network.predict(model, torch.from_numpy(u1).cuda(), torch.from_numpy(u2).cuda())
    assert flow.shape == (1, 50, 100, 2) and occ.shape == (1, 50, 100, 1)
    a, b, _ = prepost_ref.preprocess(u1, u2, prepost_ref.padded_size(50, 100))
    params = {k: v.detach().cpu() for k, v in model.named_parameters()}
    with torch.no_grad():
        preds, o, _ = network_ref.maskflownet_s_forward(params, torch.from_numpy(a), torch.from_numpy(b), threads=8)
    ref = prepost_ref.postprocess(preds[-1].numpy(), 50, 100)
    assert np.abs(flow.cpu().numpy() - ref).max() < 5e-3
    assert np.abs(occ.cpu().numpy() - prepost_ref.postprocess(o[0].numpy(), 50, 100, False, False)).max() < 1e-3


@pytest.mark.parametrize("cls", [network.MaskFlownetS, network.MaskFlownet])
def test_fused_heads_equal_separate_heads(cls):
    """fuse_heads (pred_flow / pred_mask partial sums computed by conv{L}_4's launch through the linear-prefix epilogue, plus a
    32-channel tail convolution) == the separate 3-output head convolution over the whole block output."""
    model = _named_model(cls)
    a1, a2 = seeded_images(seed=13, n=2, h=64, w=128)
    with torch.no_grad():
        model.fuse_heads = True
        if cls is network.MaskFlownet:
            model.MaskFlownet_S.fuse_heads = True
        fused = model(a1.cuda(), a2.cuda())[0]
        model.fuse_heads = False
        if cls is network.MaskFlownet:
            model.MaskFlownet_S.fuse_heads = False
        plain = model(a1.cuda(), a2.cuda())[0]
    for f, p in zip(fused, plain):
        assert (f - p).abs().max().item() <= 1e-4 * max(1.0, p.abs().max().item())
