"""The training-side rows of SURVEY.md 8f: N4, GPU-side augmentation (/root/reference/augmentation.py:168-339), and the fused
MultiscaleEpe of row N2 (network/MaskFlownet.py:563-611).

CPU part (`-m "not gpu"`): the numpy restatement (oracle/augment_ref.py) against the fixture produced by the reference's own
augmentation.py (tests/golden/make_golden_aug.py); the product's host logic (draws -> parameter blocks) against the oracle;
and the kernel SOURCE of csrc/augment.cu compiled for the host (tests/host_emu/) against the oracle.
GPU part (`-m gpu`): mfn_geometry_augment_forward / mfn_color_augment_forward / mfn_multiscale_epe_* through the C ABI
against the oracle.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import augment_ref

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "aug_ref_graph.npz")
sys.path.insert(0, os.path.join(HERE, "golden"))
GEO_NAMES = ["rotation", "aspect_ratio", "scale", "tx_unit", "tx_range", "ty_unit", "ty_range", "rel_rotation", "rel_scale",
             "rel_translation"]


@pytest.fixture(autouse=True)
def _fp32():
    # cuDNN / cuBLAS references in fp32 (torch's default lets cuDNN convolutions use TF32: 1e-3 relative error)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


@pytest.fixture(scope="module")
def fx():
    return dict(np.load(FIX))


def geo_draws(fx, prefix="geo"):
    return {k: fx[f"{prefix}_draw_{k}"] for k in GEO_NAMES}


def col_draws(fx, prefix):
    return {k[len(prefix) + 6:]: v for k, v in fx.items() if k.startswith(prefix + "_draw_")}


def shapes(fx):
    return tuple(int(v) for v in fx["orig_shape"]), tuple(int(v) for v in fx["target_shape"])


# ---------------------------------------------------------------------------------------------------------------
# oracle vs the reference's own graph
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prefix", ["geo", "geob"])
def test_oracle_geometry_matches_reference_graph(fx, prefix):
    orig, target = shapes(fx)
    P = augment_ref.geometry_params(geo_draws(fx, prefix), orig, target)
    mask = fx["mask"] if prefix == "geo" else np.ones((fx["img1"].shape[0], 1, 1, 1), np.float32)
    out = augment_ref.geometry_augment(fx["img1"], fx["img2"], fx["flow"], mask, P, target)
    for name, got in zip(("img1", "img2", "flow", "mask"), out):
        ref = fx[f"{prefix}_{name}"]
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() < (2e-4 if name == "flow" else 2e-5), name
    assert np.abs(out[2]).max() > 1.0 and (prefix == "geob" or 0 < out[3].mean() < 1)


def test_oracle_color_matches_reference_graph(fx):
    d = col_draws(fx, "col")
    P = augment_ref.color_params(d, gamma=True, eigen=False)
    sigma = float(d["noise_sigma"][0])
    assert sigma > 0
    for k, img in (("1", fx["geo_img1"]), ("2", fx["geo_img2"])):
        got = augment_ref.color_augment_one(img, P, noise=d["noise" + k], noise_sigma=sigma)
        assert np.abs(got - fx["col_img" + k]).max() < 2e-5
    e = col_draws(fx, "eig")
    Pe = augment_ref.color_params(e, gamma=False, eigen=True)
    for k, img in (("1", fx["geo_img1"]), ("2", fx["geo_img2"])):
        got = augment_ref.color_augment_one(img, Pe)
        assert np.abs(got - fx["eig_img" + k]).max() < 2e-5


# ---------------------------------------------------------------------------------------------------------------
# product host logic (draws -> parameter blocks)
# ---------------------------------------------------------------------------------------------------------------
def make_geo(orig, target, N, seed=None):
    from maskflownet_b200 import augment
    return augment.GeometryAugmentation(angle_range=(-17, 17), zoom_range=(0.5, 1 / 0.9), aspect_range=(0.9, 1 / 0.9),
                                        translation_range=0.1, target_shape=target, orig_shape=orig, batch_size=N,
                                        relative_angle=0.25, relative_scale=(0.96, 1 / 0.96), relative_translation=0.25, seed=seed)


def test_host_geometry_params_match_oracle(fx):
    orig, target = shapes(fx)
    geo = make_geo(orig, target, 3)
    for prefix in ("geo", "geob"):
        d = geo_draws(fx, prefix)
        got = geo.params({k: torch.from_numpy(v) for k, v in d.items()}).numpy()
        want = augment_ref.geometry_params(d, orig, target)
        assert got.shape == want.shape == (3, 22)
        assert np.abs(got - want).max() < 1e-5 * max(1.0, np.abs(want).max())


def test_host_color_params_match_oracle(fx):
    from maskflownet_b200 import augment
    _, target = shapes(fx)
    kitti = augment.ColorAugmentation(contrast_range=(-0.2, 0.4), brightness_sigma=0.05, channel_range=(0.9, 1.2), batch_size=3,
                                      shape=target, noise_range=(0, 0.02), saturation=0.25, hue=0.1, gamma_range=(-0.5, 0.5))
    d = col_draws(fx, "col")
    got = kitti.params({k: torch.from_numpy(np.asarray(v)) for k, v in d.items() if not k.startswith("noise") or k == "noise_sigma"})
    assert np.abs(got.numpy() - augment_ref.color_params(d, gamma=True)).max() < 1e-6
    sintel = augment.ColorAugmentation(contrast_range=(-0.4, 0.8), brightness_sigma=0.1, channel_range=(0.8, 1.4), batch_size=3,
                                       shape=target, noise_range=(0, 0), saturation=0.5, hue=0.5, eigen_aug=True)
    e = col_draws(fx, "eig")
    got = sintel.params({k: torch.from_numpy(np.asarray(v)) for k, v in e.items()})
    assert np.abs(got.numpy() - augment_ref.color_params(e, eigen=True)).max() < 1e-6


def test_host_sampling_ranges_and_determinism():
    geo = make_geo((384, 512), (320, 448), 8, seed=11)
    d = geo.sample()
    assert list(d) == GEO_NAMES and d["rel_translation"].shape == (8, 2)
    assert (d["rotation"].abs() <= 17 / 180 * np.pi + 1e-6).all() and (d["scale"] >= 0.5).all() and (d["scale"] <= 1 / 0.9 + 1e-6).all()
    assert (d["rel_translation"].abs() <= 0.05 + 1e-6).all()      # 0.25 * (2 * 0.1)
    P = geo.params(d)
    assert P.shape == (8, 22) and torch.isfinite(P).all()
    assert torch.equal(make_geo((384, 512), (320, 448), 8, seed=11).sample()["scale"], d["scale"])
    with pytest.raises(Exception):
        from maskflownet_b200 import augment
        augment.GeometryAugmentation((-1, 1), (1, 1), 0.1, (8, 8), (8, 8), 1)     # the reference has no non-relative path


# ---------------------------------------------------------------------------------------------------------------
# the kernel source compiled for the host (no GPU in the development container)
# ---------------------------------------------------------------------------------------------------------------
def _build_emu(tmp_path_factory, name):
    out = str(tmp_path_factory.mktemp("emu") / f"lib{name}.so")
    src = os.path.join(HERE, "host_emu", name + ".cpp")
    subprocess.run(["g++", "-O1", "-ffp-contract=off", "-shared", "-fPIC", "-I", os.path.join(HERE, "host_emu"), "-o", out, src],
                   check=True)
    return ctypes.CDLL(out)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    return _build_emu(tmp_path_factory, "augment_emu")


@pytest.fixture(scope="module")
def emu_loss(tmp_path_factory):
    return _build_emu(tmp_path_factory, "loss_emu")


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def emu_geometry(emu, img1, img2, flow, mask, P, target):
    N, _, H, W = img1.shape
    TH, TW = target
    o1, o2 = np.zeros((N, 3, TH, TW), np.float32), np.zeros((N, 3, TH, TW), np.float32)
    of, om = np.zeros((N, 2, TH, TW), np.float32), np.zeros((N, 1, TH, TW), np.float32)
    arrs = [np.ascontiguousarray(a) for a in (img1, img2, flow, mask, P)]
    emu.emu_geometry_augment(_ptr(arrs[0]), _ptr(arrs[1]), int(img1.dtype == np.uint8), _ptr(arrs[2]), _ptr(arrs[3]),
                             int(mask.shape[2:] == (1, 1) and (H, W) != (1, 1)), _ptr(arrs[4]), _ptr(o1), _ptr(o2), _ptr(of),
                             _ptr(om), N, H, W, TH, TW)
    return o1, o2, of, om


def geometry_case(seed, N, orig, target, uint8, bcast):
    rng = np.random.default_rng(seed)
    H, W = orig
    if uint8:
        img1 = rng.integers(0, 256, (N, 3, H, W), dtype=np.uint8)
        img2 = rng.integers(0, 256, (N, 3, H, W), dtype=np.uint8)
        mask = np.full((N, 1, 1, 1), 255, np.uint8) if bcast else (rng.random((N, 1, H, W)) > 0.2).astype(np.uint8) * 255
    else:
        img1, img2 = rng.random((N, 3, H, W), dtype=np.float32), rng.random((N, 3, H, W), dtype=np.float32)
        mask = np.ones((N, 1, 1, 1), np.float32) if bcast else (rng.random((N, 1, H, W)) > 0.2).astype(np.float32)
    flow = (rng.standard_normal((N, 2, H, W)) * 4).astype(np.float32)
    geo = make_geo(orig, target, N, seed=seed)
    d = geo.sample()
    P = geo.params(d).numpy()
    P[0, 12:14] += np.float32(0.7)      # sample 0: a relative translation that pushes the second grid out of the image (zero padding)
    return img1, img2, flow, mask, P, geo, d


def oracle_geometry(img1, img2, flow, mask, P, target):
    if img1.dtype == np.uint8:
        img1, img2, mask = (a.astype(np.float32) / np.float32(255) for a in (img1, img2, mask))
    return augment_ref.geometry_augment(img1, img2, flow, mask, P, target)


def check_geometry(got, want, tag=""):
    for name, a, b in zip(("img1", "img2", "flow", "mask"), got, want):
        tol = 1e-5 if name != "flow" else 1e-5 * max(1.0, float(np.abs(b).max()))
        assert np.abs(a - b).max() < tol, (tag, name, float(np.abs(a - b).max()))


@pytest.mark.parametrize("uint8,bcast", [(False, False), (True, True), (True, False), (False, True)])
def test_kernel_source_geometry_on_host(emu, fx, uint8, bcast):
    orig, target = (30, 44), (20, 28)
    img1, img2, flow, mask, P, _, _ = geometry_case(5 + uint8 + 2 * bcast, 3, orig, target, uint8, bcast)
    want = oracle_geometry(img1, img2, flow, mask, P, target)
    assert (want[1][0] == 0).mean() > 0.1 and (want[1][1] == 0).mean() < 0.05      # the zero-padded region is exercised
    check_geometry(emu_geometry(emu, img1, img2, flow, mask, P, target), want)


def test_kernel_source_geometry_on_host_reference_fixture(emu, fx):
    orig, target = shapes(fx)
    P = augment_ref.geometry_params(geo_draws(fx), orig, target)
    got = emu_geometry(emu, fx["img1"], fx["img2"], fx["flow"], fx["mask"], P, target)
    check_geometry(got, [fx["geo_" + k] for k in ("img1", "img2", "flow", "mask")], "fixture")


def test_kernel_source_color_on_host(emu, fx):
    d = col_draws(fx, "col")
    P = np.ascontiguousarray(augment_ref.color_params(d, gamma=True))
    sigma = float(d["noise_sigma"][0])
    i1, i2 = np.ascontiguousarray(fx["geo_img1"]), np.ascontiguousarray(fx["geo_img2"])
    n1, n2 = np.ascontiguousarray(d["noise1"]), np.ascontiguousarray(d["noise2"])
    N, _, H, W = i1.shape
    # partial sums as color_sum_kernel lays them out: ws[image][n][slice][3]; everything in slice 0 here
    ws = np.zeros((2, N, 64, 3), np.float32)
    for k, (img, nz) in enumerate(((i1, n1), (i2, n2))):
        pre = np.zeros_like(img)
        emu.emu_color_pre_mean(_ptr(img), _ptr(nz), _ptr(P), ctypes.c_float(sigma), ctypes.c_longlong(0), k, _ptr(pre), N, H, W)
        ws[k, :, 0, :] = pre.sum(axis=(2, 3), dtype=np.float64)
    o1, o2 = np.zeros_like(i1), np.zeros_like(i2)
    emu.emu_color_apply(_ptr(i1), _ptr(i2), _ptr(P), _ptr(n1), _ptr(n2), ctypes.c_float(sigma), ctypes.c_longlong(0), _ptr(ws),
                        _ptr(o1), _ptr(o2), N, H, W, 1)
    assert np.abs(o1 - fx["col_img1"]).max() < 2e-5 and np.abs(o2 - fx["col_img2"]).max() < 2e-5


def test_kernel_source_philox_noise_on_host(emu):
    N, H, W, seed = 2, 5, 7, 0x1234567890ABCDEF & 0x7FFFFFFFFFFFFFFF
    P = np.zeros((N, 26), np.float32)            # zero hue matrix: the pre-mean image IS noise * sigma
    img = np.zeros((N, 3, H, W), np.float32)
    for image in (0, 1):
        pre = np.zeros_like(img)
        emu.emu_color_pre_mean(_ptr(img), None, _ptr(P), ctypes.c_float(1.0), ctypes.c_longlong(seed), image, _ptr(pre), N, H, W)
        want = augment_ref.philox_normal(N, H, W, seed, image)
        assert np.abs(pre - want).max() < 2e-5
    z = augment_ref.philox_normal(8, 64, 64, 99, 0)
    assert abs(float(z.mean())) < 0.02 and abs(float(z.std()) - 1.0) < 0.02     # a standard normal stream
    # Philox4x32-10 known-answer test (Random123 kat_vectors: counter = key = 0)
    r = augment_ref.philox4x32_10([0], [0], [0], [0], 0, 0)
    assert [int(x[0]) for x in r] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


# ---------------------------------------------------------------------------------------------------------------
# GPU: the C ABI against the oracle
# ---------------------------------------------------------------------------------------------------------------
def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("uint8,bcast,N,orig,target", [
    (False, False, 3, (30, 44), (20, 28)),
    (True, True, 2, (64, 96), (48, 80)),
    (True, False, 4, (96, 128), (64, 112)),
    (False, True, 2, (384, 512), (320, 448)),          # FlyingChairs shapes of main.py (orig 384x512 -> target 320x448)
])
def test_geometry_augment_parity(uint8, bcast, N, orig, target):
    from maskflownet_b200 import augment
    img1, img2, flow, mask, P, _, _ = geometry_case(17 + N, N, orig, target, uint8, bcast)
    got = augment.geometry_augment(_cuda(img1), _cuda(img2), _cuda(flow), _cuda(mask), _cuda(P), target)
    check_geometry([g.cpu().numpy() for g in got], oracle_geometry(img1, img2, flow, mask, P, target), "gpu")


@pytest.mark.gpu
def test_geometry_augment_reference_fixture_and_class(fx):
    from maskflownet_b200 import augment
    orig, target = shapes(fx)
    geo = make_geo(orig, target, 3)
    d = {k: torch.from_numpy(v) for k, v in geo_draws(fx).items()}
    got = geo(_cuda(fx["img1"]), _cuda(fx["img2"]), _cuda(fx["flow"]), _cuda(fx["mask"]), draws=d)
    check_geometry([g.cpu().numpy() for g in got], [fx["geo_" + k] for k in ("img1", "img2", "flow", "mask")], "fixture")
    # own draws: runs, finite, images stay in [0, 1], mask in [0, 1]
    o1, o2, of, om = geo(_cuda(fx["img1"]), _cuda(fx["img2"]), _cuda(fx["flow"]), _cuda(fx["mask"]))
    assert all(torch.isfinite(t).all() for t in (o1, o2, of, om))
    assert 0 <= float(o1.min()) and float(o1.max()) <= 1 and 0 <= float(om.min()) and float(om.max()) <= 1 + 1e-6
    with pytest.raises(augment.MaskflowError):
        augment.geometry_augment(torch.zeros(1, 3, 8, 8), torch.zeros(1, 3, 8, 8), torch.zeros(1, 2, 8, 8), torch.zeros(1, 1, 8, 8),
                                 torch.zeros(1, 22), (4, 4))       # CPU tensors: no fallback


@pytest.mark.gpu
def test_color_augment_parity(fx):
    from maskflownet_b200 import augment
    d = col_draws(fx, "col")
    P = augment_ref.color_params(d, gamma=True)
    sigma = float(d["noise_sigma"][0])
    o1, o2 = augment.color_augment(_cuda(fx["geo_img1"]), _cuda(fx["geo_img2"]), _cuda(P), noise_sigma=sigma,
                                   noise=(_cuda(d["noise1"]), _cuda(d["noise2"])), has_gamma=True)
    assert np.abs(o1.cpu().numpy() - fx["col_img1"]).max() < 2e-5 and np.abs(o2.cpu().numpy() - fx["col_img2"]).max() < 2e-5
    e = col_draws(fx, "eig")
    Pe = augment_ref.color_params(e, eigen=True)
    o1, o2 = augment.color_augment(_cuda(fx["geo_img1"]), _cuda(fx["geo_img2"]), _cuda(Pe))
    assert np.abs(o1.cpu().numpy() - fx["eig_img1"]).max() < 2e-5 and np.abs(o2.cpu().numpy() - fx["eig_img2"]).max() < 2e-5


@pytest.mark.gpu
def test_color_augment_in_kernel_noise_and_class():
    from maskflownet_b200 import augment
    rng = np.random.default_rng(3)
    N, H, W, seed, sigma = 4, 96, 160, 123456789012345, 0.03
    i1, i2 = rng.random((N, 3, H, W), dtype=np.float32), rng.random((N, 3, H, W), dtype=np.float32)
    col = augment.ColorAugmentation(contrast_range=(-0.2, 0.4), brightness_sigma=0.05, channel_range=(0.9, 1.2), batch_size=N,
                                    shape=(H, W), noise_range=(0, 0.02), saturation=0.25, hue=0.1, gamma_range=(-0.5, 0.5), seed=5)
    d = col.sample()
    P = col.params(d)
    o1, o2 = augment.color_augment(_cuda(i1), _cuda(i2), P.cuda(), noise_sigma=sigma, seed=seed, has_gamma=True)
    for image, (img, out) in enumerate(((i1, o1), (i2, o2))):
        want = augment_ref.color_augment_one(img, P.numpy(), noise=augment_ref.philox_normal(N, H, W, seed, image), noise_sigma=sigma)
        assert np.abs(out.cpu().numpy() - want).max() < 2e-5
    # bit-reproducible (no atomics), and the class call runs end to end
    p1, p2 = augment.color_augment(_cuda(i1), _cuda(i2), P.cuda(), noise_sigma=sigma, seed=seed, has_gamma=True)
    assert torch.equal(p1, o1) and torch.equal(p2, o2)
    c1, c2 = col(_cuda(i1), _cuda(i2))
    assert torch.isfinite(c1).all() and 0 <= float(c1.min()) and float(c2.max()) <= 1


# ---------------------------------------------------------------------------------------------------------------
# fused MultiscaleEpe (row N2): kernel source on the host, then the C ABI on the GPU, against torch autograd of the
# operator-by-operator composition on the oracle's Upsample
# ---------------------------------------------------------------------------------------------------------------
def epe_case(seed, N, H, W, scales):
    rng = np.random.default_rng(seed)
    preds = [np.ascontiguousarray(rng.standard_normal((N, 2, H // s, W // s)).astype(np.float32) * 2) for s in scales]
    flow = (rng.standard_normal((N, 2, H, W)) * 2).astype(np.float32)
    mask = (rng.random((N, 1, H, W)) > 0.3).astype(np.float32)
    gl = rng.random(N).astype(np.float32) + 0.5
    return preds, flow, mask, gl


def epe_oracle(preds, flow, mask, gl, scales, weights, eps, q):
    from maskflownet_b200 import losses
    from oracle import torch_ref
    rp = [torch.from_numpy(p).clone().requires_grad_() for p in preds]
    loss = losses.multiscale_epe(torch.from_numpy(flow), torch.from_numpy(mask), rp, scales=scales, weights=weights, eps=eps, q=q,
                                 upsample=torch_ref.upsample)
    (loss * torch.from_numpy(gl)).sum().backward()
    return loss.detach().numpy(), [p.grad.numpy() for p in rp]


@pytest.mark.parametrize("q", [None, 0.4])
def test_kernel_source_multiscale_epe_on_host(emu_loss, q):
    scales, weights, eps = (16, 8, 4, 2), (.01, .02, .08, .32), 1e-8 if q is None else 0.01
    N, H, W = 2, 32, 48
    preds, flow, mask, gl = epe_case(4, N, H, W, scales)
    want_loss, want_grads = epe_oracle(preds, flow, mask, gl, scales, weights, eps, q)
    n = len(scales)
    pa = (ctypes.c_void_p * n)(*[p.ctypes.data for p in preds])
    sa, wa = (ctypes.c_int * n)(*scales), (ctypes.c_float * n)(*weights)
    loss, msum = np.zeros(N, np.float32), np.zeros(N, np.float32)
    qf = ctypes.c_float(-1.0 if q is None else q)
    emu_loss.emu_epe_forward(_ptr(flow), _ptr(mask), pa, sa, wa, n, ctypes.c_float(eps), qf, _ptr(loss), _ptr(msum), N, H, W)
    assert np.abs(loss - want_loss).max() < 1e-5 * max(1.0, np.abs(want_loss).max())
    assert np.abs(msum - mask.sum(axis=(1, 2, 3))).max() < 0.5
    grads = [np.full_like(p, np.nan) for p in preds]
    ga = (ctypes.c_void_p * n)(*[g.ctypes.data for g in grads])
    emu_loss.emu_epe_backward(_ptr(flow), _ptr(mask), pa, sa, wa, n, ctypes.c_float(eps), qf, _ptr(gl), _ptr(msum), ga, N, H, W)
    for g, w in zip(grads, want_grads):
        assert np.isfinite(g).all() and np.abs(g - w).max() < 1e-5 * max(1e-3, np.abs(w).max())


def test_multiscale_epe_autograd_function_on_host_emulation(emu_loss, monkeypatch):
    """losses.multiscale_epe's autograd Function (argument marshalling, saved tensors, order / count of the returned gradients,
    once_differentiable) end to end on CPU tensors: the two C-ABI calls are routed to the host build of the same kernels."""
    from maskflownet_b200 import losses, ops

    def fake_call(name, dev, *args):
        conv = [ctypes.c_float(a) if isinstance(a, float) else a for a in args]
        if name == "mfn_multiscale_epe_forward":       # (..., loss, mask_sum, workspace, workspace_bytes, N, H, W)
            emu_loss.emu_epe_forward(*conv[:10], *conv[12:15])
        elif name == "mfn_multiscale_epe_backward":
            emu_loss.emu_epe_backward(*conv)
        else:
            raise AssertionError(name)
    monkeypatch.setattr(ops, "_call", fake_call)
    monkeypatch.setattr(ops, "_chk", lambda t, name, optional=False: t if t is None else t.contiguous())
    scales, weights = (16, 8, 4), (.02, .08, .32)
    N, H, W = 2, 32, 48
    preds, flow, mask, gl = epe_case(11, N, H, W, scales)
    want_loss, want_grads = epe_oracle(preds, flow, mask, gl, scales, weights, 1e-8, None)
    tp = [torch.from_numpy(p).clone().requires_grad_() for p in preds]
    loss = losses.multiscale_epe(torch.from_numpy(flow), torch.from_numpy(mask), tp, scales=scales, weights=weights, fused=True)
    assert np.abs(loss.detach().numpy() - want_loss).max() < 1e-5 * max(1.0, np.abs(want_loss).max())
    (loss * torch.from_numpy(gl)).sum().backward()
    for t, w in zip(tp, want_grads):
        assert t.grad is not None and np.abs(t.grad.numpy() - w).max() < 1e-5 * max(1e-3, np.abs(w).max())
    with pytest.raises(Exception):                       # the label is data: no gradient is defined for it
        losses.multiscale_epe(torch.from_numpy(flow).requires_grad_(), torch.from_numpy(mask), tp, scales=scales, weights=weights, fused=True)


@pytest.mark.gpu
@pytest.mark.parametrize("q,N,H,W", [(None, 2, 64, 128), (0.4, 3, 128, 192), (None, 8, 384, 512)])
def test_multiscale_epe_fused_parity(q, N, H, W):
    from maskflownet_b200 import losses
    eps = 1e-8 if q is None else 0.01
    preds, flow, mask, gl = epe_case(9, N, H, W, losses.SCALES)
    want_loss, want_grads = epe_oracle(preds, flow, mask, gl, losses.SCALES, losses.WEIGHTS, eps, q)
    gp = [_cuda(p).requires_grad_() for p in preds]
    loss = losses.multiscale_epe(_cuda(flow), _cuda(mask), gp, eps=eps, q=q)
    assert loss.shape == (N,) and np.abs(loss.detach().cpu().numpy() - want_loss).max() < 2e-5 * max(1.0, np.abs(want_loss).max())
    (loss * _cuda(gl)).sum().backward()
    for a, w in zip(gp, want_grads):
        assert np.abs(a.grad.cpu().numpy() - w).max() < 2e-5 * max(1e-3, np.abs(w).max())
    # the unfused composition (ops.upsample + torch) agrees, and the fused path is bit-reproducible
    gq = [_cuda(p).requires_grad_() for p in preds]
    ref = losses.multiscale_epe(_cuda(flow), _cuda(mask), gq, eps=eps, q=q, fused=False)
    assert (ref - loss).detach().abs().max().item() < 2e-5 * max(1.0, ref.detach().abs().max().item())
    again = losses.multiscale_epe(_cuda(flow), _cuda(mask), [_cuda(p) for p in preds], eps=eps, q=q)
    assert torch.equal(again, loss.detach())


# ---------------------------------------------------------------------------------------------------------------
# training-mode convolutions: tensor-core forward + cuDNN backward (ops.conv3x3_train, network.train_tc_forward)
# ---------------------------------------------------------------------------------------------------------------
def test_conv3x3_train_backward_wiring_on_cpu(monkeypatch):
    """The autograd wiring of ops._Conv3x3TrainFn (activation mask from the saved output, aten.convolution_backward argument
    order, frozen input, missing bias) against plain autograd, with the CUDA forward replaced by a torch stub."""
    import torch.nn.functional as tF
    from maskflownet_b200 import ops

    def stub(x, packed, bias, Cout, slope, dil, stride):
        y = tF.conv2d(x, packed, bias, stride=stride, padding=dil, dilation=dil)
        return y if slope == 1.0 else tF.leaky_relu(y, slope)
    monkeypatch.setattr(ops, "conv3x3", stub)
    torch.manual_seed(0)
    for slope, dil, stride, has_bias in [(0.1, 1, 1, True), (0.1, 1, 2, True), (1.0, 1, 1, True), (0.1, 4, 1, True), (0.1, 1, 1, False)]:
        x = torch.randn(2, 5, 9, 11, requires_grad=True)
        w = torch.randn(4, 5, 3, 3, requires_grad=True)
        b = torch.randn(4, requires_grad=True) if has_bias else None
        y = ops._Conv3x3TrainFn.apply(x, w, b, w.detach(), slope, dil, stride)
        g = torch.randn_like(y)
        y.backward(g)
        got = [t.grad.clone() for t in (x, w) + ((b,) if has_bias else ())]
        for t in (x, w) + ((b,) if has_bias else ()):
            t.grad = None
        stub(x, w, b, 4, slope, dil, stride).backward(g)
        for a, t in zip(got, (x, w) + ((b,) if has_bias else ())):
            assert torch.allclose(a, t.grad, atol=1e-6)
    x = torch.randn(2, 3, 8, 8)                                     # the image layer: no input gradient requested
    w = torch.randn(4, 3, 3, 3, requires_grad=True)
    ops._Conv3x3TrainFn.apply(x, w, None, w.detach(), 0.1, 1, 2).sum().backward()
    assert w.grad.abs().sum() > 0


@pytest.mark.gpu
def test_conv3x3_train_matches_cudnn_autograd():
    import torch.nn.functional as tF
    from maskflownet_b200 import ops
    torch.manual_seed(1)
    for Cin, Cout, H, W, dil, stride in [(16, 32, 24, 40, 1, 1), (3, 16, 32, 64, 1, 2), (128, 96, 16, 32, 8, 1)]:
        x = torch.randn(2, Cin, H, W, device="cuda", requires_grad=Cin != 3)
        w = (torch.randn(Cout, Cin, 3, 3, device="cuda") * (2.0 / (9 * Cin)) ** 0.5).requires_grad_()
        b = (torch.randn(Cout, device="cuda") * 0.1).requires_grad_()
        y = ops.conv3x3_train(x, w, b, ops.conv3x3_pack(w), 0.1, dil, stride)
        ref = tF.leaky_relu(tF.conv2d(x, w, b, stride=stride, padding=dil, dilation=dil), 0.1)
        err = (y - ref).abs().max().item()
        assert err < 1e-4 * max(1.0, ref.abs().max().item()), (Cin, Cout, dil, stride, err, ref.abs().max().item())
        # backward: the same activation mask on both sides (ours comes from the saved output; a pre-activation within the
        # forward's 1e-5 of zero may legitimately fall on the other side of the LeakyReLU kink in the cuDNN forward, which
        # moves single weight-gradient entries by O(|g x|) -- seen on the B200: 1 of 98 k outputs flipped), so the
        # reference is the LINEAR convolution's autograd fed with the masked gradient
        g = torch.randn_like(ref)
        wrt = [w, b] + ([x] if x.requires_grad else [])
        gy = torch.autograd.grad(y, wrt, g)
        lin = tF.conv2d(x, w, b, stride=stride, padding=dil, dilation=dil)
        gr = torch.autograd.grad(lin, wrt, torch.where(y.detach() > 0, g, g * 0.1))
        for a, r in zip(gy, gr):
            assert (a - r).abs().max().item() < 1e-4 * max(1.0, r.abs().max().item()), (Cin, Cout, dil, stride, tuple(a.shape),
                                                                                      (a - r).abs().max().item(), r.abs().max().item())
        flips = ((y.detach() > 0) != (ref.detach() > 0)).float().mean().item()
        assert flips < 1e-4, flips


@pytest.mark.gpu
def test_training_step_with_tensor_core_forward_matches_cudnn_forward():
    """One MaskFlownet-S training step (MultiscaleEpe loss) with train_tc_forward on / off: same loss, same gradients up to the
    1e-5-relative difference of the two forward convolutions."""
    from maskflownet_b200 import losses, network
    torch.manual_seed(3)
    model = network.MaskFlownetS().cuda().train()
    g = torch.Generator().manual_seed(5)
    a = torch.rand(2, 3, 128, 192, generator=g).cuda() - 0.5
    b = torch.rand(2, 3, 128, 192, generator=g).cuda() - 0.5
    flow = (torch.randn(2, 2, 128, 192, generator=g) * 2).cuda()
    mask = torch.ones(2, 1, 128, 192).cuda()
    res = {}
    for mode in (False, True):
        model.train_tc_forward = mode
        model.zero_grad(set_to_none=True)
        preds = model(a, b)[0]
        loss = losses.multiscale_epe(flow, mask, preds).sum()
        loss.backward()
        res[mode] = (loss.item(), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None})
    assert abs(res[True][0] - res[False][0]) < 1e-4 * max(1.0, abs(res[False][0])), (res[True][0], res[False][0])
    assert res[True][1].keys() == res[False][1].keys() and len(res[True][1]) > 100
    worst = max(((res[True][1][k] - res[False][1][k]).abs().max().item() / max(res[False][1][k].abs().max().item(), 1e-6), k)
                for k in res[False][1])
    # LeakyReLU kinks / floor() in the warps may flip on 1e-5 forward differences: single entries move, a wiring error would be O(1)
    assert worst[0] < 5e-2, worst


# ---------------------------------------------------------------------------------------------------------------
# pipeline.PipelineFlownet (the reference's network/pipeline.py:19-223): host plumbing on the CPU with the CUDA operators
# replaced by the oracle; the same calls on the GPU
# ---------------------------------------------------------------------------------------------------------------
class _TinyNet(torch.nn.Module):
    """Stand-in for MaskFlownetS with the same output contract: ([flow6..flow2], [mask2], None)."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(6, 3, 3, padding=1)

    def forward(self, a, b):
        import torch.nn.functional as tF
        y = self.conv(torch.cat([a, b], dim=1))
        preds = [tF.avg_pool2d(y[:, :2], s) * 20.0 for s in (64, 32, 16, 8, 4)]
        return preds, [torch.sigmoid(tF.avg_pool2d(y[:, 2:3], 4))], None


def _cpu_pipeline(monkeypatch):
    from maskflownet_b200 import network, ops, pipeline
    from oracle import cref, prepost_ref, torch_ref
    t = torch.from_numpy
    monkeypatch.setattr(network, "MaskFlownetS", _TinyNet)
    monkeypatch.setattr(ops, "upsample", lambda x, f, scale=1.0: torch_ref.upsample(x, f) * scale)
    monkeypatch.setattr(ops, "preprocess", lambda a, b, hw=None: tuple(t(v) for v in prepost_ref.preprocess(a.numpy(), b.numpy(), hw)))
    monkeypatch.setattr(ops, "postprocess", lambda p, H, W, flip_channels=True, is_flow=True: t(
        prepost_ref.postprocess(p.numpy(), H, W, flip_channels, is_flow)))
    monkeypatch.setattr(ops, "grid_generator_warp", lambda f: t(cref.grid_generator_warp(f.numpy())))
    monkeypatch.setattr(ops, "bilinear_sampler", lambda d, g: t(cref.bilinear_sampler(d.numpy(), g.numpy())))
    return pipeline.PipelineFlownet(device="cpu", lr_schedule=[(2, 1e-4), (5, 5e-5)])


def test_pipeline_host_plumbing_on_cpu(monkeypatch):
    pipe = _cpu_pipeline(monkeypatch)
    rng = np.random.default_rng(0)
    n, H, W = 2, 128, 192

    def geo(i1, i2, fl, mk):          # stand-in with the augmentation's contract: uint8 in, float32 [0,1] + (x,y) flow + mask out
        return i1.float() / 255, i2.float() / 255, fl.clone(), (mk.float() / 255).expand(n, 1, H, W).contiguous()
    img1 = rng.integers(0, 256, (n, 3, H, W), dtype=np.uint8)
    img2 = rng.integers(0, 256, (n, 3, H, W), dtype=np.uint8)
    label = (rng.standard_normal((n, 2, H, W)) * 2).astype(np.float32)
    w0 = pipe.network.conv.weight.detach().clone()
    out = pipe.train_batch(img1, img2, label, geo, lambda a, b: (a, b))
    assert np.isfinite(out["epe"]) and out["epe"] > 0
    assert not torch.equal(pipe.network.conv.weight, w0)                  # the optimizer stepped
    g = pipe._bucket.flat.clone()
    out2 = pipe.train_batch(img1, img2, label, geo, lambda a, b: (a, b), global_batch=4 * n)
    assert np.isfinite(out2["epe"]) and pipe._bucket.flat.abs().max() < g.abs().max()      # gradients rescaled by 1 / global batch
    # learning-rate schedule (pipeline.py:65-76)
    assert pipe.set_learning_rate(1) and pipe.lr == 1e-4 and pipe.set_learning_rate(3) and pipe.lr == 5e-5
    assert pipe.trainer.param_groups[0]["lr"] == 5e-5 and not pipe.set_learning_rate(9)
    # validation / prediction loops over lists of HWC samples of a size that needs the x64 resize
    Hs, Ws = 100, 150
    s1 = [rng.integers(0, 256, (Hs, Ws, 3), dtype=np.uint8) for _ in range(3)]
    s2 = [rng.integers(0, 256, (Hs, Ws, 3), dtype=np.uint8) for _ in range(3)]
    lab = [(rng.standard_normal((Hs, Ws, 2)) * 3).astype(np.float32) for _ in range(3)]
    epe = pipe.validate(s1, s2, lab, batch_size=2)
    f1 = pipe.validate(s1, s2, lab, batch_size=2, return_type="f1")
    assert np.isfinite(epe) and epe > 0 and 0 <= f1 <= 1
    res = list(pipe.predict(s1, s2, batch_size=2))
    assert len(res) == 3 and res[0][0].shape == (Hs, Ws, 2) and res[0][1].shape == (Hs, Ws, 1) and res[0][2].shape == (Hs, Ws, 3)
    # predict's flow is do_batch's flow, channels-last and flipped to (x, y)
    a = torch.from_numpy(np.transpose(np.stack(s1[:1]), (0, 3, 1, 2)).copy())
    b = torch.from_numpy(np.transpose(np.stack(s2[:1]), (0, 3, 1, 2)).copy())
    flow, _, warp, _ = pipe.do_batch(a, b)
    assert np.allclose(res[0][0], flow[0].permute(1, 2, 0).flip(-1).numpy()) and warp.shape == (1, 3, Hs, Ws)
    with pytest.raises(Exception):
        pipe.fix_head()                      # only the cascade has a head to freeze


def test_pipeline_load_head_and_fix_head_on_cpu(tmp_path):
    """main.py:133-139: a MaskFlownet-S checkpoint goes into the cascade's head (load_head), which is then frozen (fix_head);
    the trainer only keeps the cascade's own parameters.  The checkpoint is the shipped one's byte layout, rebuilt from
    tests/golden/checkpoint_layout.npz."""
    from make_golden_checkpoints import CHECKPOINT_S, rebuild_checkpoint
    from maskflownet_b200 import params as mparams, pipeline
    ck = rebuild_checkpoint(CHECKPOINT_S, tmp_path)
    pipe = pipeline.PipelineFlownet(device="cpu", network_class="MaskFlownet")
    pipe.load_head(ck)
    raw = mparams.read_params(ck)
    name = next(k for k in raw if k.endswith("conv3bweight"))
    assert np.array_equal(pipe.network.MaskFlownet_S.conv3b.weight.detach().numpy(), raw[name])
    n_all = sum(p.numel() for p in pipe.network.parameters())
    pipe.fix_head()
    n_train = sum(p.numel() for g in pipe.trainer.param_groups for p in g["params"])
    assert n_all == 20_655_716 and n_all - n_train == 10_514_256          # the S head's parameters are out of the optimizer
    assert all(not p.requires_grad for p in pipe.network.MaskFlownet_S.parameters())
    with pytest.raises(Exception):
        pipeline.PipelineFlownet(device="cpu").load_head(ck)               # MaskFlownet_S alone has no head to load


@pytest.mark.gpu
def test_pipeline_train_validate_predict_on_gpu():
    from maskflownet_b200 import augment, pipeline
    rng = np.random.default_rng(1)
    n, orig, target = 2, (160, 224), (128, 192)
    pipe = pipeline.PipelineFlownet(lr_schedule=[(10, 1e-4)])
    geo = augment.GeometryAugmentation(angle_range=(-17, 17), zoom_range=(0.5, 1 / 0.9), aspect_range=(0.9, 1 / 0.9),
                                       translation_range=0.1, target_shape=target, orig_shape=orig, batch_size=n,
                                       relative_angle=0.25, relative_scale=(0.96, 1 / 0.96), relative_translation=0.25, seed=3)
    col = augment.ColorAugmentation(contrast_range=(-0.4, 0.8), brightness_sigma=0.1, channel_range=(0.8, 1.4), batch_size=n,
                                    shape=target, noise_range=(0, 0.04), saturation=0.5, hue=0.5, seed=4)
    img1 = rng.integers(0, 256, (n, 3) + orig, dtype=np.uint8)
    img2 = rng.integers(0, 256, (n, 3) + orig, dtype=np.uint8)
    label = (rng.standard_normal((n, 2) + orig) * 2).astype(np.float32)
    w0 = pipe.network.conv2_0.weight.detach().clone()
    out = pipe.train_batch(img1, img2, label, geo, col)
    assert np.isfinite(out["epe"]) and not torch.equal(pipe.network.conv2_0.weight, w0)
    s1 = [rng.integers(0, 256, (100, 150, 3), dtype=np.uint8) for _ in range(2)]
    s2 = [rng.integers(0, 256, (100, 150, 3), dtype=np.uint8) for _ in range(2)]
    lab = [(rng.standard_normal((100, 150, 2)) * 3).astype(np.float32) for _ in range(2)]
    assert np.isfinite(pipe.validate(s1, s2, lab, batch_size=2))
    res = list(pipe.predict(s1, s2, batch_size=2))
    assert len(res) == 2 and res[0][0].shape == (100, 150, 2) and np.isfinite(res[0][0]).all() and res[0][2].shape == (100, 150, 3)
