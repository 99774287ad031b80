"""Widening rows of SURVEY §8(f): fused losses, fused Adam, GaussianModel (accessors, densify / prune in one
gather) -- each against a plain PyTorch statement of the reference's formula / sequence of operations."""
import copy
import json
import os
import math
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- plain torch statements (reference formulas)
def _window(dtype, device):
    g = torch.tensor([math.exp(-((x - 5) ** 2) / float(2 * 1.5 ** 2)) for x in range(11)])   # loss_utils.py:45-52
    g = (g / g.sum()).unsqueeze(1)
    return g.mm(g.t()).float().unsqueeze(0).unsqueeze(0).to(device=device, dtype=dtype)


def torch_ssim(a, b):
    """loss_utils.py:75-104, single channel, zero padding."""
    w = _window(a.dtype, a.device)
    a, b = a[None], b[None]
    mu1, mu2 = F.conv2d(a, w, padding=5), F.conv2d(b, w, padding=5)
    s11 = F.conv2d(a * a, w, padding=5) - mu1 * mu1
    s22 = F.conv2d(b * b, w, padding=5) - mu2 * mu2
    s12 = F.conv2d(a * b, w, padding=5) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    m = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s11 + s22 + C2))
    return m.mean()


def torch_tv(vol, mean):
    tv = vol.diff(dim=0).abs().sum() + vol.diff(dim=1).abs().sum() + vol.diff(dim=2).abs().sum()
    if mean:
        nx, ny, nz = vol.shape
        tv = tv / ((nx - 1) * ny * nz + nx * (ny - 1) * nz + nx * ny * (nz - 1))
    return tv


def _images(H, W, seed):
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, W), indexing="ij")
    base = torch.exp(-(xx ** 2 + yy ** 2) * 3) * 2.0
    a = (base + 0.15 * torch.rand(H, W, generator=g)).unsqueeze(0)
    b = (base * 0.9 + 0.1 * torch.rand(H, W, generator=g)).unsqueeze(0)
    return a.cuda(), b.cuda()


@pytest.mark.parametrize("H,W", [(64, 64), (50, 77), (11, 5), (512, 512)])
@pytest.mark.parametrize("lam", [0.25, 0.0])
def test_image_loss_matches_torch(H, W, lam):
    from r2_gaussian_b200 import losses
    a, b = _images(H, W, 1)
    a64 = a.double().requires_grad_(True)
    ref = (a64 - b.double()).abs().mean() + lam * (1.0 - torch_ssim(a64, b.double()))
    ref.backward()
    a32 = a.clone().requires_grad_(True)
    out = losses.image_loss(a32, b, lambda_dssim=lam)
    out["total"].backward()
    # float32 SSIM is limited by the cancellation in E[x^2] - mu^2 (the reference's too): the bar is the error of
    # the same formula evaluated by torch in float32 (TF32 off), with a floor of 5e-6
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    a_t = a.clone().requires_grad_(True)
    t32 = (a_t - b).abs().mean() + lam * (1.0 - torch_ssim(a_t, b))
    t32.backward()
    s32 = torch_ssim(a, b).item()
    torch.backends.cudnn.allow_tf32 = tf32
    s64 = torch_ssim(a.double(), b.double()).item()
    bar = max(5e-6, 3.0 * abs(s32 - s64))
    assert abs((1 - out["dssim"]).item() - s64) <= bar
    assert abs(out["total"].item() - ref.item()) <= 2e-6 * max(1.0, abs(ref.item())) + lam * bar
    assert abs(out["render"].item() - (a - b).abs().mean().item()) <= 1e-6
    gref = a64.grad.float()
    scale = gref.abs().max().item()
    gbar = max(2e-4 * scale, 3.0 * (a_t.grad - gref).abs().max().item())
    assert (a32.grad - gref).abs().max().item() <= gbar + 1e-9
    # reference-named entry points
    assert abs(losses.l1_loss(a, b).item() - (a - b).abs().mean().item()) <= 1e-6
    assert abs(losses.ssim(a, b).item() - s64) <= bar
    # bitwise reproducible
    out2 = losses.image_loss(a, b, lambda_dssim=lam)
    out3 = losses.image_loss(a, b, lambda_dssim=lam)
    assert torch.equal(out2["total"], out3["total"])


@pytest.mark.parametrize("shape", [(32, 32, 32), (7, 9, 5), (1, 4, 4), (64, 48, 40)])
@pytest.mark.parametrize("mean", [True, False])
def test_tv3d_matches_torch(shape, mean):
    from r2_gaussian_b200 import losses
    g = torch.Generator().manual_seed(3)
    v = torch.rand(*shape, generator=g).cuda()
    v[v < 0.2] = 0.0                       # plateaus: sign(0) = 0 like torch.abs' backward
    v64 = v.double().requires_grad_(True)
    ref = torch_tv(v64, mean)
    ref.backward()
    v32 = v.clone().requires_grad_(True)
    got = losses.tv_3d_loss(v32, reduction="mean" if mean else "sum")
    got.backward()
    assert abs(got.item() - ref.item()) <= 2e-6 * max(1.0, abs(ref.item()))
    assert (v32.grad - v64.grad.float()).abs().max().item() <= 1e-6 * max(1.0, v64.grad.abs().max().item())


def test_fused_adam_matches_torch_adam():
    from r2_gaussian_b200.optim import FusedAdam
    torch.manual_seed(0)
    shapes = [(1000, 3), (1000, 1), (1000, 3), (1000, 4)]
    lrs = [2e-4, 1e-2, 5e-3, 1e-3]
    p_ref = [torch.nn.Parameter(torch.randn(*s, device="cuda")) for s in shapes]
    p_our = [torch.nn.Parameter(p.detach().clone()) for p in p_ref]
    o_ref = torch.optim.Adam([{"params": [p], "lr": lr, "name": str(i)} for i, (p, lr) in enumerate(zip(p_ref, lrs))],
                             lr=0.0, eps=1e-15)
    o_our = FusedAdam([{"params": [p], "lr": lr, "name": str(i)} for i, (p, lr) in enumerate(zip(p_our, lrs))],
                      lr=0.0, eps=1e-15)
    for it in range(25):
        for pr, po in zip(p_ref, p_our):
            g = torch.randn_like(pr) * (0.1 + it)
            g[::7] = 0.0
            pr.grad, po.grad = g.clone(), g.clone()
        if it == 10:                               # schedules change the learning rates between steps
            for gr, go in zip(o_ref.param_groups, o_our.param_groups):
                gr["lr"] *= 0.5
                go["lr"] *= 0.5
        o_ref.step()
        o_our.step()
    for pr, po in zip(p_ref, p_our):
        assert (pr - po).abs().max().item() <= 2e-6 * pr.abs().max().item()
        sr, so = o_ref.state[pr], o_our.state[po]
        for k in ("exp_avg", "exp_avg_sq"):
            assert (sr[k] - so[k]).abs().max().item() <= 2e-6 * sr[k].abs().max().item(), k
        assert float(sr["step"]) == float(so["step"]) == 25
    # the state dict is interchangeable with torch's Adam
    o_ref.load_state_dict(o_our.state_dict())


# ---------------------------------------------------------------- GaussianModel
def _opt_args():
    return types.SimpleNamespace(
        position_lr_init=2e-4, position_lr_final=2e-5, position_lr_max_steps=30000,
        density_lr_init=1e-2, density_lr_final=1e-3, density_lr_max_steps=30000,
        scaling_lr_init=5e-3, scaling_lr_final=5e-4, scaling_lr_max_steps=30000,
        rotation_lr_init=1e-3, rotation_lr_final=1e-4, rotation_lr_max_steps=30000)


def _make_model(n=4000, seed=0, scale_bound=(0.0005, 0.5)):
    from r2_gaussian_b200.gaussian_model import GaussianModel
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(-0.8, 0.8, size=(n, 3)).astype(np.float32)
    dens = rng.uniform(0.05, 0.9, size=(n, 1)).astype(np.float32)
    gm = GaussianModel(scale_bound)
    gm.create_from_pcd(xyz, dens, 1.0)
    gm.training_setup(_opt_args())
    return gm, xyz, dens


def test_model_accessors_and_init():
    from oracle import r2_oracle as orc
    gm, xyz, dens = _make_model()
    assert torch.allclose(gm.get_density, torch.from_numpy(dens).cuda(), rtol=1e-5, atol=1e-6)   # softplus(inverse) = id
    d2 = np.maximum(orc.knn3_mean_dist2(xyz), 0.001 ** 2)
    want = np.clip(np.sqrt(d2), 0.0005 + 1e-5, 0.5 - 1e-5)
    assert np.allclose(gm.get_scaling.detach().cpu().numpy(), np.repeat(want[:, None], 3, 1), rtol=2e-4, atol=1e-7)
    q = gm.get_rotation
    assert torch.allclose(q.norm(dim=1), torch.ones_like(q[:, 0]))
    cov = gm.get_covariance(1.5)
    s = (1.5 * gm.get_scaling) ** 2
    assert torch.allclose(cov[:, [0, 3, 5]], s, rtol=1e-5, atol=1e-9)            # identity rotation: diag(s^2)
    assert gm.construct_list_of_attributes()[:7] == ["x", "y", "z", "nx", "ny", "nz", "density"]
    gm.update_learning_rate(15000)
    lr = {g["name"]: g["lr"] for g in gm.optimizer.param_groups}
    assert abs(lr["xyz"] - math.sqrt(2e-4 * 2e-5)) < 1e-12                       # log-linear midpoint


class _Sequential:
    """The reference's order of operations (gaussian_model.py:320-550: cat -> mask per step, torch Adam), written
    straightforwardly, as the yardstick for the one-gather implementation."""

    def __init__(self, gm):
        self.gm = gm
        self.p = {n: getattr(gm, a).detach().clone() for n, a in (("xyz", "_xyz"), ("density", "_density"),
                                                                   ("scaling", "_scaling"), ("rotation", "_rotation"))}
        self.m = {n: gm.optimizer.state[getattr(gm, a)]["exp_avg"].clone() for n, a in
                  (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation"))}
        self.v = {n: gm.optimizer.state[getattr(gm, a)]["exp_avg_sq"].clone() for n, a in
                  (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation"))}
        self.radii = gm.max_radii2D.clone()

    def _cat(self, new, radii):
        for k in self.p:
            self.p[k] = torch.cat((self.p[k], new[k]))
            self.m[k] = torch.cat((self.m[k], torch.zeros_like(new[k])))
            self.v[k] = torch.cat((self.v[k], torch.zeros_like(new[k])))
        self.radii = torch.cat((self.radii, radii))

    def _mask(self, keep):
        for k in self.p:
            self.p[k], self.m[k], self.v[k] = self.p[k][keep], self.m[k][keep], self.v[k][keep]
        self.radii = self.radii[keep]

    def run(self, grads, max_grad, min_density, max_screen_size, max_scale, thr, bbox):
        from r2_gaussian_b200.gaussian_utils import build_rotation
        gm = self.gm
        act_s, inv_s, act_d, inv_d = gm.scaling_activation, gm.scaling_inverse_activation, gm.density_activation, gm.density_inverse_activation
        # clone (:474-501)
        sel = (torch.norm(grads, dim=-1) >= max_grad) & (act_s(self.p["scaling"]).max(dim=1).values <= thr)
        half = inv_d(act_d(self.p["density"][sel]) * 0.5)
        new = {"xyz": self.p["xyz"][sel], "density": half, "scaling": self.p["scaling"][sel], "rotation": self.p["rotation"][sel]}
        r = self.radii[sel]
        self.p["density"][sel] = half
        self._cat(new, r)
        # split (:430-472)
        n = self.p["xyz"].shape[0]
        pad = torch.zeros(n, device="cuda")
        pad[: grads.shape[0]] = grads.squeeze()
        sel = (pad >= max_grad) & (act_s(self.p["scaling"]).max(dim=1).values > thr)
        stds = act_s(self.p["scaling"])[sel].repeat(2, 1)
        samples = torch.normal(mean=torch.zeros((stds.size(0), 3), device="cuda"), std=stds)
        rots = build_rotation(self.p["rotation"][sel]).repeat(2, 1, 1)
        new = {"xyz": torch.bmm(rots, samples.unsqueeze(-1)).squeeze(-1) + self.p["xyz"][sel].repeat(2, 1),
               "scaling": inv_s(act_s(self.p["scaling"])[sel].repeat(2, 1) / (0.8 * 2)),
               "rotation": self.p["rotation"][sel].repeat(2, 1),
               "density": inv_d(act_d(self.p["density"])[sel].repeat(2, 1) * 0.5)}
        r = self.radii[sel].repeat(2)
        self._cat(new, r)
        self._mask(~torch.cat((sel, torch.zeros(2 * int(sel.sum()), device="cuda", dtype=bool))))
        # prune (:528-548)
        xyz = self.p["xyz"]
        drop = (act_d(self.p["density"]) < min_density).squeeze()
        drop |= ((xyz[:, 0] < bbox[0, 0]) | (xyz[:, 0] > bbox[1, 0]) | (xyz[:, 1] < bbox[0, 1]) | (xyz[:, 1] > bbox[1, 1])
                 | (xyz[:, 2] < bbox[0, 2]) | (xyz[:, 2] > bbox[1, 2]))
        drop |= self.radii > max_screen_size
        drop |= act_s(self.p["scaling"]).max(dim=1).values > max_scale
        self._mask(~drop)


def test_densify_and_prune_equals_the_sequential_procedure():
    gm, _, _ = _make_model(n=6000, seed=5)
    torch.manual_seed(1)
    # a few optimizer steps so that the Adam moments are non-trivial
    for _ in range(3):
        for _, attr in (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation")):
            p = getattr(gm, attr)
            p.grad = torch.randn_like(p) * 1e-2
        gm.optimizer.step()
    n = gm.get_xyz.shape[0]
    gm.max_radii2D = torch.rand(n, device="cuda") * 40
    gm.xyz_gradient_accum = torch.rand(n, 1, device="cuda") * 3e-3
    gm.denom = torch.randint(0, 4, (n, 1), device="cuda").float()          # zeros -> NaN -> 0 like the reference
    with torch.no_grad():
        gm._scaling[: n // 2] += 2.0                                        # some large Gaussians -> split candidates
        gm._density[::17] = -9.0                                            # some nearly empty ones -> pruned
    bbox = torch.tensor([[-0.75, -0.75, -0.75], [0.75, 0.75, 0.75]], device="cuda")
    args = dict(max_grad=5e-4, min_density=1e-3, max_screen_size=35.0, max_scale=0.3)
    thr = 0.01
    seq = _Sequential(gm)
    grads = gm.xyz_gradient_accum / gm.denom
    grads[grads.isnan()] = 0.0
    torch.manual_seed(123)
    seq.run(grads, args["max_grad"], args["min_density"], args["max_screen_size"], args["max_scale"], thr, bbox)
    torch.manual_seed(123)
    with torch.no_grad():
        out = gm.densify_and_prune(args["max_grad"], args["min_density"], args["max_screen_size"], args["max_scale"],
                                   None, thr, bbox)
    assert torch.equal(out, grads)
    assert gm.get_xyz.shape[0] == seq.p["xyz"].shape[0] and gm.get_xyz.shape[0] != n
    for name, attr in (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation")):
        p = getattr(gm, attr)
        assert isinstance(p, torch.nn.Parameter) and p.requires_grad
        assert torch.equal(p.detach(), seq.p[name]), name
        st = gm.optimizer.state[p]
        assert torch.equal(st["exp_avg"], seq.m[name]) and torch.equal(st["exp_avg_sq"], seq.v[name]), name
        assert any(g["params"][0] is p for g in gm.optimizer.param_groups)
    assert torch.equal(gm.max_radii2D, seq.radii)
    assert gm.xyz_gradient_accum.shape == (gm.get_xyz.shape[0], 1) and float(gm.xyz_gradient_accum.abs().sum()) == 0.0
    # the model still trains after the surgery
    for _, attr in (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation")):
        p = getattr(gm, attr)
        p.grad = torch.ones_like(p)
    gm.optimizer.step()


def test_prune_reset_capture_restore_and_pickle(tmp_path):
    from r2_gaussian_b200.gaussian_model import GaussianModel
    gm, _, _ = _make_model(n=500, seed=2)
    for _, attr in (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation")):
        p = getattr(gm, attr)
        p.grad = torch.randn_like(p)
    gm.optimizer.step()
    mask = torch.zeros(500, dtype=torch.bool, device="cuda")
    mask[::5] = True
    before = gm._xyz.detach().clone()
    gm.prune_points(mask)
    assert gm.get_xyz.shape[0] == 400 and torch.equal(gm._xyz.detach(), before[~mask])
    assert gm.optimizer.state[gm._xyz]["exp_avg"].shape[0] == 400 and gm.max_radii2D.shape[0] == 400
    gm.reset_density(0.1)
    assert float(gm.get_density.detach().max()) <= 0.1 + 1e-6
    assert float(gm.optimizer.state[gm._density]["exp_avg"].abs().sum()) == 0.0
    snap = copy.deepcopy(gm.capture())
    gm2 = GaussianModel(None)
    gm2.restore(snap, _opt_args())
    assert torch.equal(gm2._xyz, gm._xyz) and gm2.scale_bound == gm.scale_bound
    assert torch.equal(gm2.optimizer.state[gm2._xyz]["exp_avg"], gm.optimizer.state[gm._xyz]["exp_avg"])
    path = tmp_path / "point_cloud" / "point_cloud.pickle"
    gm.save_ply(str(path))
    gm3 = GaussianModel(None)
    gm3.load_ply(str(path))
    assert torch.equal(gm3._scaling, gm._scaling) and tuple(gm3.scale_bound) == tuple(gm.scale_bound)
    assert torch.allclose(gm3.get_scaling, gm.get_scaling)


def test_short_training_run_reduces_the_loss():
    """render() + fused image loss + fused Adam on a small scene: the projection error of a perturbed cloud
    goes down (end-to-end smoke of the training step around the hot path)."""
    from r2_gaussian_b200 import losses, scene
    from r2_gaussian_b200.render_query import render
    from r2_gaussian_b200.gaussian_model import GaussianModel
    scanner = scene.cone_beam_scanner(n_detector=128)
    views = [scene.camera_from_view(v) for v in scene.make_views(scanner, 4)]
    cloud = scene.make_cloud(3000, seed=4)
    pipe = types.SimpleNamespace(compute_cov3D_python=False, debug=False)

    def model_from(xyz, dens):
        gm = GaussianModel((0.0005, 0.5))
        gm.create_from_pcd(xyz, dens, 1.0)
        gm.training_setup(_opt_args())
        return gm

    truth = model_from(cloud.means, cloud.density)
    with torch.no_grad():
        targets = [render(v, truth, pipe)["render"].clone() for v in views]
    rng = np.random.default_rng(0)
    start = model_from(cloud.means + rng.normal(scale=0.01, size=cloud.means.shape).astype(np.float32),
                       cloud.density * 0.6 + 0.02)
    history = []
    for it in range(40):
        v = it % len(views)
        start.update_learning_rate(it + 1)
        img = render(views[v], start, pipe)["render"]
        loss = losses.image_loss(img, targets[v], lambda_dssim=0.25)
        loss["total"].backward()
        start.optimizer.step()
        start.optimizer.zero_grad(set_to_none=True)
        history.append(float(loss["total"]))
    assert history[-1] < 0.7 * history[0], history[::8]


def test_densification_stats_without_mask_indexing():
    gm, _, _ = _make_model(n=300, seed=9)
    vsp = torch.zeros(300, 3, device="cuda", requires_grad=True)
    vsp.grad = torch.randn(300, 3, device="cuda")
    vsp.grad[5] = float("nan")                         # an invisible row may hold anything
    vis = torch.rand(300, device="cuda") > 0.4
    vis[5] = False
    acc0, den0 = gm.xyz_gradient_accum.clone(), gm.denom.clone()
    gm.add_densification_stats(vsp, vis)
    want = acc0.clone()
    want[vis] += torch.norm(vsp.grad[vis, :2], dim=-1, keepdim=True)      # the reference's statement (:552-556)
    den = den0.clone()
    den[vis] += 1
    assert torch.equal(gm.xyz_gradient_accum, want) and torch.equal(gm.denom, den)
    radii = torch.randint(0, 50, (300,), device="cuda", dtype=torch.int32)
    before = gm.max_radii2D.clone()
    gm.update_max_radii(radii, vis)
    ref = before.clone()
    ref[vis] = torch.max(ref[vis], radii[vis].float())
    assert torch.equal(gm.max_radii2D, ref)


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_fused_losses_against_reference_golden_vectors(tag):
    """The fused L1 + D-SSIM kernel and the TV kernel against outputs of the reference's own loss_utils.py
    (float64 evaluation; tests/golden/make_golden_host.py)."""
    import os
    from r2_gaussian_b200 import losses
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_golden.npz"))
    img = torch.from_numpy(G[f"loss_{tag}_img"]).cuda().requires_grad_(True)
    gt = torch.from_numpy(G[f"loss_{tag}_gt"]).cuda()
    l1_64, ssim_64, total_64 = G[f"loss_{tag}_f64"]
    ssim_32 = G[f"loss_{tag}_f32"][1]
    out = losses.image_loss(img, gt, lambda_dssim=0.25)
    out["total"].backward()
    bar = max(5e-6, 3.0 * abs(ssim_32 - ssim_64))               # the reference's own float32 error sets the scale
    assert abs(out["render"].item() - l1_64) <= 1e-6
    assert abs((1.0 - out["dssim"].item()) - ssim_64) <= bar
    assert abs(out["total"].item() - total_64) <= 2e-6 + 0.25 * bar
    g64, g32 = G[f"loss_{tag}_grad_f64"], G[f"loss_{tag}_grad_f32"]
    gbar = max(2e-4 * np.abs(g64).max(), 3.0 * np.abs(g32 - g64).max())
    assert np.abs(img.grad.cpu().numpy() - g64).max() <= gbar
    if tag in ("a", "b"):
        for red in ("sum", "mean"):
            v = torch.from_numpy(G[f"tv_{tag}_vol"]).cuda().requires_grad_(True)
            t = losses.tv_3d_loss(v, reduction=red)
            t.backward()
            want = float(G[f"tv_{tag}_{red}"][0])
            assert abs(t.item() - want) <= 2e-6 * max(1.0, abs(want))
            gw = G[f"tv_{tag}_{red}_grad"]
            assert np.abs(v.grad.cpu().numpy() - gw).max() <= 1e-6 * max(1.0, np.abs(gw).max())


DENSIFY_GROUPS = (("xyz", "_xyz"), ("density", "_density"), ("scaling", "_scaling"), ("rotation", "_rotation"))
DENSIFY_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "densify_prune_reference.json")


def tensor_digest(t):
    """shape, dtype and SHA-256 of the raw bytes: equal digests mean bit-identical tensors."""
    import hashlib
    a = t.detach().contiguous().cpu().numpy()
    return {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}


def densify_state_digests(model):
    """Digests of everything densify_and_prune reads or writes on a model (ours or the reference's class): the four
    parameters with both Adam moments, max_radii2D and the gradient statistics, in row order."""
    out = {}
    for name, attr in DENSIFY_GROUPS:
        p = getattr(model, attr)
        st = model.optimizer.state[p]
        out[name] = tensor_digest(p)
        out[name + ".exp_avg"] = tensor_digest(st["exp_avg"])
        out[name + ".exp_avg_sq"] = tensor_digest(st["exp_avg_sq"])
    for attr in ("max_radii2D", "xyz_gradient_accum", "denom"):
        out[attr] = tensor_digest(getattr(model, attr))
    return out


def densify_case(max_num):
    """The model state densify_and_prune starts from, and its arguments (tests/golden/make_golden_densify.py builds
    the reference's class in exactly this state)."""
    gm, xyz, dens = _make_model(n=6000, seed=5)
    torch.manual_seed(1)
    for _ in range(3):      # a few optimizer steps so that the Adam moments are non-trivial
        for _, attr in DENSIFY_GROUPS:
            p = getattr(gm, attr)
            p.grad = torch.randn_like(p) * 1e-2
        gm.optimizer.step()
    n = gm.get_xyz.shape[0]
    gm.max_radii2D = torch.rand(n, device="cuda") * 40
    gm.xyz_gradient_accum = torch.rand(n, 1, device="cuda") * 3e-3
    gm.denom = torch.randint(0, 4, (n, 1), device="cuda").float()
    with torch.no_grad():
        gm._scaling[: n // 2] += 2.0
        gm._density[::17] = -9.0
    bbox = torch.tensor([[-0.75, -0.75, -0.75], [0.75, 0.75, 0.75]], device="cuda")
    args = (5e-4, 1e-3, 35.0, 0.3, max_num, 0.01, bbox)
    return gm, xyz, dens, args


@pytest.mark.parametrize("max_num", [None, 10])
def test_densify_and_prune_bit_equal_to_the_reference_class(max_num):
    """Device-side compaction (r2x_mask_select + r2x_gather_rows) against the reference's cat / boolean-mask sequence:
    the reference's own GaussianModel.densify_and_prune was run from the same state and its result is stored as
    digests (tests/golden/make_golden_densify.py).  Parameters, both Adam moments, max_radii2D, statistics, row order,
    the returned tensor and the CUDA RNG stream are bit-identical (max_num=10: the densification branch is skipped,
    prune only)."""
    with open(DENSIFY_GOLDEN) as f:
        golden = json.load(f)[str(max_num)]
    gm, _, _, args = densify_case(max_num)
    n = gm.get_xyz.shape[0]
    # the digests only speak for this test if it starts where the reference started
    assert densify_state_digests(gm) == golden["before"], "the starting state differs from the recorded one"
    torch.manual_seed(123)
    with torch.no_grad():
        g_our = gm.densify_and_prune(*args)
    # the same stream of random numbers has been consumed
    assert torch.cuda.get_rng_state().numpy().tobytes().hex() == golden["cuda_rng_state_after"]
    assert tensor_digest(g_our) == golden["returned"]
    assert gm.get_xyz.shape[0] == golden["after"]["xyz"]["shape"][0] and gm.get_xyz.shape[0] != n
    ours = densify_state_digests(gm)
    for k, want in golden["after"].items():
        assert ours[k] == want, k


def test_select_and_gather_rows_against_torch_indexing():
    from r2_gaussian_b200 import compact
    g = torch.Generator("cuda").manual_seed(3)
    for n in (0, 1, 5, 1000, 70001):
        mask = torch.rand(n, device="cuda", generator=g) < 0.37
        idx, cnt = compact.select_rows(mask)
        k = compact.read_counts(cnt)[0]
        want = torch.nonzero(mask).squeeze(-1)
        assert k == want.numel() and torch.equal(idx[:k].long(), want)
        a = torch.randn(n, 3, device="cuda", generator=g); b = torch.randn(n, device="cuda", generator=g)
        extra = torch.randn(7, 3, device="cuda", generator=g)
        sel = torch.cat((idx[:k], torch.arange(n, n + 7, device="cuda", dtype=torch.int32)))
        out = compact.gather_rows([(a, extra), (b, None), (a, None)], sel, k + 7)
        assert torch.equal(out[0], torch.cat((a, extra))[sel.long()])
        assert torch.equal(out[1], torch.cat((b, torch.zeros(7, device="cuda")))[sel.long()])
        assert torch.equal(out[2], torch.cat((a, torch.zeros(7, 3, device="cuda")))[sel.long()])


@pytest.mark.parametrize("bounded", [True, False])
def test_folded_activations_match_the_torch_activations(bounded, monkeypatch):
    """render() / query() on raw parameters (activations inside the preprocess kernels, gradients w.r.t. the raw
    parameters from the per-Gaussian backward kernels) against the plain path (torch softplus / sigmoid / normalize +
    autograd), image, volume and every parameter gradient."""
    from r2_gaussian_b200 import scene
    from r2_gaussian_b200.render_query import query, render
    pipe = types.SimpleNamespace(compute_cov3D_python=False, debug=False)
    cam = scene.camera_from_view(scene.make_view(scene.cone_beam_scanner(128, 64), 0.6))
    rng = np.random.default_rng(3)
    groups = ("_xyz", "_density", "_scaling", "_rotation")

    def run(fused_on):
        monkeypatch.setenv("R2X_FUSED_ACTIVATIONS", "1" if fused_on else "0")
        gm, _, _ = _make_model(n=3000, seed=7, scale_bound=(0.0005, 0.5) if bounded else None)
        with torch.no_grad():
            gm._rotation += torch.tensor(rng.normal(scale=0.3, size=(3000, 4)).astype(np.float32), device="cuda")
            gm._scaling += torch.tensor(rng.normal(scale=0.2, size=(3000, 3)).astype(np.float32), device="cuda")
        pkg = render(cam, gm, pipe)
        vol = query(gm, [0.1, 0.0, -0.1], [32, 32, 32], [0.5, 0.5, 0.5], pipe)["vol"]
        g = torch.Generator("cuda").manual_seed(5)
        loss = (pkg["render"] * torch.randn(pkg["render"].shape, device="cuda", generator=g)).sum() + \
               (vol * torch.randn(vol.shape, device="cuda", generator=g)).sum()
        loss.backward()
        return (pkg["render"].detach(), vol.detach(), [getattr(gm, a).grad.clone() for a in groups],
                pkg["viewspace_points"].grad.clone(), pkg["radii"].clone())

    rng = np.random.default_rng(3); plain = run(False)
    rng = np.random.default_rng(3); fused = run(True)
    assert torch.equal(plain[4], fused[4])
    for a, b, what in ((plain[0], fused[0], "image"), (plain[1], fused[1], "volume")):
        assert float((a - b).abs().max()) <= 2e-6 * float(a.abs().max()) + 1e-9, what
    for ga, gb, name in zip(plain[2], fused[2], groups):
        assert float((ga - gb).abs().max()) <= 2e-5 * float(ga.abs().max()) + 1e-9, name
    assert float((plain[3] - fused[3]).abs().max()) <= 2e-5 * float(plain[3].abs().max()) + 1e-9


def _train_inputs(n_cams=4, det=128):
    from r2_gaussian_b200 import scene
    scanner = scene.cone_beam_scanner(det, 64)
    cams = [scene.camera_from_view(scene.make_view(scanner, 0.3 + 0.9 * k)) for k in range(n_cams)]
    g = torch.Generator("cuda").manual_seed(9)
    gts = [torch.rand((1, det, det), device="cuda", generator=g) * 0.5 for _ in cams]
    centres = [(0.1 * k - 0.15, 0.05 * k, -0.1 + 0.07 * k) for k in range(n_cams)]
    return cams, gts, centres


@pytest.mark.parametrize("use_tv", [True, False])
def test_native_train_step_is_the_autograd_iteration(use_tv):
    """NativeTrainStep (fixed launch sequence, guarded Adam / statistics, no autograd) against the same iteration through
    render() / query() / the fused losses / autograd / FusedAdam: parameters and Adam moments bit for bit."""
    from r2_gaussian_b200 import losses
    from r2_gaussian_b200.render_query import query, render
    from r2_gaussian_b200.train_step import NativeTrainStep
    pipe = types.SimpleNamespace(compute_cov3D_python=False, debug=False)
    cams, gts, centres = _train_inputs()
    lam_d, lam_tv, n_it = 0.25, 0.05, 7
    tv_n, tv_s = [32, 32, 32], [0.5, 0.5, 0.5]
    a, _, _ = _make_model(n=5000, seed=11)
    b, _, _ = _make_model(n=5000, seed=11)
    step = NativeTrainStep(b, lam_d, lam_tv if use_tv else 0.0, tv_n, tv_s)
    for i in range(1, n_it + 1):
        k = i % len(cams)
        a.update_learning_rate(i); b.update_learning_rate(i)
        pkg = render(cams[k], a, pipe)
        total = losses.image_loss(pkg["render"], gts[k], lam_d)["total"]
        if use_tv:
            total = total + lam_tv * losses.tv_3d_loss(query(a, centres[k], tv_n, tv_s, pipe)["vol"], "mean")
        total.backward()
        with torch.no_grad():
            a.update_max_radii(pkg["radii"], pkg["visibility_filter"])
            a.add_densification_stats(pkg["viewspace_points"], pkg["visibility_filter"])
        a.optimizer.step()
        a.optimizer.zero_grad(set_to_none=True)
        res = step(cams[k], gts[k], centres[k])
        if i == n_it:
            assert abs(step.total_loss() - float(total)) <= 1e-6 * abs(float(total))
            assert torch.equal(res["radii"], pkg["radii"])
    step.flush()
    assert step.repeats == 0
    for name in ("_xyz", "_density", "_scaling", "_rotation"):
        pa, pb = getattr(a, name), getattr(b, name)
        assert torch.equal(pa, pb), name
        sa, sb = a.optimizer.state[pa], b.optimizer.state[pb]
        assert torch.equal(sa["exp_avg"], sb["exp_avg"]) and torch.equal(sa["exp_avg_sq"], sb["exp_avg_sq"]), name
        assert float(sa["step"]) == float(sb["step"]) == n_it
    assert torch.equal(a.max_radii2D, b.max_radii2D)
    assert torch.equal(a.denom, b.denom)
    assert float((a.xyz_gradient_accum - b.xyz_gradient_accum).abs().max()) <= 1e-6 * float(a.xyz_gradient_accum.abs().max())


def test_native_train_step_repeats_an_overflowed_iteration():
    """A speculative forward that runs out of instance capacity changes nothing on the device (guarded launches); the
    step notices one call late, raises the capacity and repeats the iteration: same result as without the overflow."""
    from r2_gaussian_b200 import _C
    from r2_gaussian_b200.train_step import NativeTrainStep
    cams, gts, centres = _train_inputs(n_cams=2)
    a, _, _ = _make_model(n=5000, seed=13)
    b, _, _ = _make_model(n=5000, seed=13)
    sa = NativeTrainStep(a, 0.25, 0.05, [32, 32, 32], [0.5, 0.5, 0.5])
    sb = NativeTrainStep(b, 0.25, 0.05, [32, 32, 32], [0.5, 0.5, 0.5])
    for i in (1, 2):
        a.update_learning_rate(i); sa(cams[i % 2], gts[i % 2], centres[i % 2])
    sa.flush()
    b.update_learning_rate(1); sb(cams[1], gts[1], centres[1]); sb.flush()
    # starve b's second iteration: a capacity of one page of instances for both forwards
    sb.cap_r, sb.cap_v = 4096, 4096
    lib = sb.lib
    sb.binning_r = torch.empty(lib.r2x_binning_bytes(4096), dtype=torch.uint8, device="cuda")
    sb.scratch_r = torch.empty(lib.r2x_raster_bwd_scratch_bytes(4096), dtype=torch.uint8, device="cuda")
    sb.binning_v = torch.empty(lib.r2x_binning_bytes(4096), dtype=torch.uint8, device="cuda")
    sb.scratch_v = torch.empty(lib.r2x_voxel_bwd_scratch_bytes(4096), dtype=torch.uint8, device="cuda")
    saved = dict(_C._Workspace.hints)
    _C._Workspace.hints[sb.key_r] = 1; _C._Workspace.hints[sb.key_v] = 1
    sb._provision = lambda: None                       # keep the starved buffers for the next call
    b.update_learning_rate(2)
    before = b._xyz.clone()
    sb(cams[0], gts[0], centres[0])
    torch.cuda.synchronize()
    assert torch.equal(before, b._xyz)                  # guarded: the overflowed iteration changed nothing
    del sb._provision                                   # normal provisioning again
    sb.cap_r = sb.cap_v = 0
    sb.flush()                                          # notices the overflow, repeats the iteration
    assert sb.repeats == 1
    _C._Workspace.hints.update({k: v for k, v in saved.items() if k in (sb.key_r, sb.key_v)})
    for name in ("_xyz", "_density", "_scaling", "_rotation"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert float(a.optimizer.state[a._xyz]["step"]) == float(b.optimizer.state[b._xyz]["step"]) == 2
