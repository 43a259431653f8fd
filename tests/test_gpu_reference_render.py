"""-m gpu: the drop-in module and the fused expansion on the GPU against what the REFERENCE's own, unmodified Python computes.

tests/golden/make_reference_render_golden.py ran the reference's code on the CPU and stored in tests/golden/reference_*.npz
  * the raster settings and Gaussians that renderer.gaussian_renderer.render (renderer/gaussian_renderer/__init__.py:25-111)
    and renderer.gaussian_animated_renderer.render (:21-121) hand the rasterizer for a stock GaussianMeshModel
    (create_from_pcd, update_alpha, prepare_scaling_rot),
  * the gradients of the raw parameters its autograd returns when fed the rasterizer gradients of the CPU oracle,
  * the stock update_alpha / prepare_scaling_rot values,
  * which PLY property GaussianModel._load_ply puts at each tensor position, and the model_params.pt keys load_ply reads.
Here the same inputs go through `diff_gaussian_rasterization` (this repo's shim) on the GPU, with the Gaussians either as the
stock expansion made them or from the fused kernels swapped into a GaussianMeshModel-like instance by
expansion.patch_mesh_model(); images and radii are compared with the oracle (oracle/gms_oracle.c) rasterizing the same
Gaussians, gradients with the reference's.  The fixtures keep a fixed sample of each array's rows (`rows<n>` for a leading dimension n):
everything is computed on the full scene and compared on those rows."""
import hashlib
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

import diff_gaussian_rasterization as dgr
from gms_b200 import expansion, scenes
from oracle import expansion as oexp
from oracle import raster

pytestmark = pytest.mark.gpu

GRAD_TOL = {"vertices": 5e-3, "_scale": 5e-3, "_alpha": 1e-3}     # through the near-singular 2D covariance (DESIGN.md 2.2)
SETTINGS = ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix", "sh_degree",
            "campos", "prefiltered", "debug", "antialiasing")


def _golden(golden_dir, name, p):
    """The stored reference outputs, after checking that they were made from the same raw parameters as `p`."""
    z = dict(np.load(os.path.join(golden_dir, name)))
    for k in ("vertices", "faces", "_alpha", "_scale", "_opacity"):
        assert hashlib.sha256(getattr(p, k).numpy().tobytes()).hexdigest() == str(z["digest" + k]), k
    return z


def _rows(z, x):
    """The rows of `x` (a tensor or array over the full scene) that the fixtures keep."""
    x = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return x[z[f"rows{x.shape[0]}"]]


def _settings(z):
    """The settings render() built (tanfov from the camera's FoV, campos from MiniCam's inverse view matrix)."""
    v = {k: z[k] for k in SETTINGS}
    S = raster.Settings(int(v["image_height"]), int(v["image_width"]), float(v["tanfovx"]), float(v["tanfovy"]), v["bg"],
                        float(v["scale_modifier"]), v["viewmatrix"], v["projmatrix"], int(v["sh_degree"]), v["campos"],
                        bool(v["prefiltered"]), bool(v["debug"]), bool(v["antialiasing"]))
    t = lambda a: torch.tensor(a, device="cuda")
    rs = dgr.GaussianRasterizationSettings(
        image_height=S.image_height, image_width=S.image_width, tanfovx=S.tanfovx, tanfovy=S.tanfovy, bg=t(S.bg),
        scale_modifier=S.scale_modifier, viewmatrix=t(S.viewmatrix), projmatrix=t(S.projmatrix), sh_degree=S.sh_degree,
        campos=t(S.campos), prefiltered=S.prefiltered, debug=S.debug, antialiasing=S.antialiasing)
    return S, rs


class _MeshModel:
    """The attributes and getters of a GaussianMeshModel instance (scene/gaussian_model.py:95-115) that the renderers use;
    expansion.patch_mesh_model() supplies update_alpha / prepare_scaling_rot."""

    def __init__(self, p):
        mk = lambda t: nn.Parameter(t.cuda().float().contiguous().requires_grad_(True))
        self.vertices, self._alpha, self._scale, self._opacity = (mk(t) for t in (p.vertices, p._alpha, p._scale, p._opacity))
        self._features_dc, self._features_rest = mk(p._features_dc), mk(p._features_rest)
        self.faces = p.faces.cuda()
        self.eps_s0 = 1e-8
        expansion.patch_mesh_model(self)

    get_xyz = property(lambda self: self._xyz)
    get_scaling = property(lambda self: torch.exp(self._scaling))
    get_rotation = property(lambda self: torch.nn.functional.normalize(self._rotation))
    get_opacity = property(lambda self: torch.sigmoid(self._opacity))
    get_features = property(lambda self: torch.cat((self._features_dc, self._features_rest), dim=1))


def _dC(seed, S):
    rs = np.random.RandomState(seed)
    return (rs.randn(3, S.image_height, S.image_width) / (S.image_width * S.image_height)).astype(np.float32)


def _render(rs, means3D, scales, rotations, opacities, shs, dC):
    """The rasterizer call of render() (:94-102), then backward of sum(image * dC)."""
    means2D = torch.zeros_like(means3D, requires_grad=True)
    img, radii, _ = dgr.GaussianRasterizer(raster_settings=rs)(means3D=means3D, means2D=means2D, shs=shs, colors_precomp=None,
                                                               opacities=opacities, scales=scales, rotations=rotations,
                                                               cov3D_precomp=None)
    (img * torch.tensor(dC, device="cuda")).sum().backward()
    assert means2D.grad is not None and (radii > 0).dtype == torch.bool
    return img, radii


def _check_against_oracle(img, radii, S, gauss, tag):
    """Image and radii against the oracle rasterizing the Gaussians the GPU run rasterized."""
    xyz, sc, rot, op, shs = (t.detach().cpu() for t in gauss)
    st = raster.forward(S, xyz, op, shs=shs.contiguous(), scales=sc, rotations=rot)
    ok = st.ambiguous == 0
    nb = int((~ok).sum())
    err = float(np.abs(img.detach().cpu().numpy() - st.color)[:, ok].max())
    print(f"[{tag}] P={st.radii.shape[0]} N={st.N} threshold-ambiguous pixels={nb} max|image-oracle| (others)={err:.2e}")
    np.testing.assert_array_equal(radii.cpu().numpy(), st.radii)
    assert err <= 1e-5, err
    assert nb <= 1e-3 * ok.size
    return st


def _check_gaussians(z, prefix, xyz, sc, rot):
    """The GPU expansion reproduces the Gaussians the reference's stock expansion handed the rasterizer."""
    gx, gs, gr = (_rows(z, t) for t in (xyz, sc, rot))
    assert float(np.abs(gx - z[prefix + "means3D"]).max()) <= 2e-6 and float(np.abs(gr - z[prefix + "rotations"]).max()) <= 4e-6
    assert float((np.abs(gs - z[prefix + "scales"]) / z[prefix + "scales"]).max()) <= 1e-5


def _check_grads(got, z, prefix, tag):
    for k, g in got.items():
        ref_g = z[prefix + "grad" + k]
        assert g is not None, k
        scale = max(float(np.abs(ref_g).max()), 1e-20)
        e = float(np.abs(_rows(z, g).reshape(ref_g.shape) - ref_g).max()) / scale
        print(f"[{tag}] grad {k}: max err / max|reference| = {e:.2e}")
        assert e <= GRAD_TOL.get(k, 2e-4), (k, e)


def _check_sh_grads(st, dC, m, tag):
    """Colour gradients pass the reference's get_features unchanged: compare with the oracle's dL/dsh."""
    g = raster.backward(st, dC)["dL_dsh"]
    for k, ref_g in (("_features_dc", g[:, :1]), ("_features_rest", g[:, 1:])):
        ref_g = torch.tensor(ref_g)
        e = float((getattr(m, k).grad.detach().cpu() - ref_g).abs().max()) / max(float(ref_g.abs().max()), 1e-20)
        print(f"[{tag}] grad {k}: max err / max|oracle| = {e:.2e}")
        assert e <= 2e-4, (k, e)


@pytest.mark.parametrize("patched", [False, True])
def test_reference_render_on_stock_mesh_model_matches_oracle(golden_dir, patched):
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=3, seed=11, trained_like=True)
    z = _golden(golden_dir, "reference_render_static.npz", p)
    S, rs = _settings(z)
    dC = _dC(3, S)
    m = _MeshModel(p)
    tag = f"render/{'patched' if patched else 'stock'}-expansion"
    if patched:
        m.update_alpha(); m.prepare_scaling_rot()      # train.py:154-157
        gauss = (m.get_xyz, m.get_scaling, m.get_rotation, m.get_opacity)
        _check_gaussians(z, "", *gauss[:3])
    else:
        # the stock expansion's Gaussians: the oracle's restatement of it, which must give the reference's values
        xyz, sl, rr, _, _ = oexp.expand(p.vertices, p.faces, p._alpha, p._scale)
        sc, rot, op, _ = oexp.activate(sl, rr, p._opacity, p._features_dc, p._features_rest)
        _check_gaussians(z, "", xyz, sc, rot)
        assert float(np.abs(_rows(z, op) - z["opacities"]).max()) <= 1e-7
        gauss = tuple(t.detach().cuda().requires_grad_(True) for t in (xyz, sc, rot, op))
    gauss = gauss + (m.get_features,)
    img, radii = _render(rs, *gauss, dC)
    st = _check_against_oracle(img, radii, S, gauss, tag)
    _check_sh_grads(st, dC, m, tag)
    if patched:
        got = {k: getattr(m, k).grad for k in ("vertices", "_alpha", "_scale", "_opacity")}
    else:
        # the GPU's rasterizer gradients through the oracle's restatement of the stock expansion (tests/test_oracle_golden.py)
        tv, ta, ts, top = (x.clone().requires_grad_(True) for x in (p.vertices, p._alpha, p._scale, p._opacity))
        xyz, sl, rr, _, _ = oexp.expand(tv, p.faces, ta, ts)
        sc, rot, op, _ = oexp.activate(sl, rr, top, p._features_dc, p._features_rest)
        torch.autograd.backward([xyz, sc, rot, op], [t.grad.cpu() for t in gauss[:4]])
        got = dict(vertices=tv.grad, _alpha=ta.grad, _scale=ts.grad, _opacity=top.grad)
    _check_grads(got, z, "", tag)


def test_patched_and_stock_expansion_agree_on_the_gpu(golden_dir):
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=5, seed=12, trained_like=True)
    z = _golden(golden_dir, "reference_expansion_k5.npz", p)
    b = _MeshModel(p)
    b.update_alpha(); b.prepare_scaling_rot()
    for k, tol in (("alpha", 1e-6), ("triangles", 0.0), ("_xyz", 1e-6), ("_scaling", 1e-5), ("_rotation", 2e-6)):
        x, y = z[k], _rows(z, getattr(b, k))
        assert x.shape == y.shape and float(np.abs(x - y).max()) <= tol, k
    # alpha stays differentiable on the patched model (renderer/gaussian_animated_renderer/__init__.py:61-64 consumes it)
    g = np.random.RandomState(12).randn(*b.alpha.shape).astype(np.float32)
    (b.alpha * torch.tensor(g, device="cuda")).sum().backward()
    ref_g = z["grad_alpha"]
    assert float(np.abs(_rows(z, b._alpha.grad) - ref_g).max()) <= 1e-5 * float(np.abs(ref_g).max())


@pytest.mark.parametrize("t", [0.0, 2.1, 5.7])
def test_reference_animated_renderer_matches_oracle(golden_dir, t):
    """scripts/render_time_animated.py:68-87: vertices moved by transform_hotdog_fly(t), triangles gathered, and
    gaussian_animated_renderer.render(idxs, triangles, ...) re-expanding from them -- here with gradients as well."""
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=3, seed=13, trained_like=True)
    z = _golden(golden_dir, "reference_render_animated.npz", p)
    i = [float(x) for x in z["times"]].index(t)
    S, rs = _settings(z)
    m = _MeshModel(p)
    m.update_alpha(); m.prepare_scaling_rot()
    tri = scenes.transform_hotdog_fly(p.vertices, t)[p.faces].cuda()
    # what the animated renderer does with the triangles (:61-73)
    means3D = torch.matmul(m.alpha, tri).reshape(-1, 3)
    m.triangles = tri
    m.prepare_scaling_rot()
    gauss = (means3D, m.get_scaling, m.get_rotation, m.get_opacity)
    _check_gaussians(z, f"t{i}_", *gauss[:3])
    gauss = gauss + (m.get_features,)
    dC = _dC(4, S)
    img, radii = _render(rs, *gauss, dC)
    st = _check_against_oracle(img, radii, S, gauss, f"animated t={t}")
    _check_sh_grads(st, dC, m, f"animated t={t}")
    _check_grads({k: getattr(m, k).grad for k in ("_alpha", "_scale", "_opacity")}, z, f"t{i}_", f"animated t={t}")
    # the animated path feeds triangles directly: no gradient reaches pc.vertices
    assert m.vertices.grad is None or not m.vertices.grad.any()


def test_checkpoint_written_here_loads_in_the_reference(golden_dir, tmp_path):
    """io_ply.save_mesh_model -> the tensors the reference's GaussianMeshModel.load_ply (gaussian_mesh_model.py:211-225 ->
    scene/gaussian_model.py:226-262) builds from it, assembled with the property layout its loader was seen to use ->
    the same image as the model that was saved."""
    from gms_b200 import io_ply
    from gms_b200.model import MeshGaussianModel
    from gms_b200.trainer import render_frame
    lay = np.load(os.path.join(golden_dir, "reference_ply_layout.npz"))
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=3, seed=31, trained_like=True)
    ours = MeshGaussianModel.from_params(p, "cuda")
    ply = str(tmp_path / "point_cloud" / "iteration_30000" / "point_cloud.ply")
    io_ply.save_mesh_model(ply, ours)
    data, names = io_ply.read_ply_vertices(ply)
    loaded = {}
    for k in ("_xyz", "_features_dc", "_features_rest", "_opacity", "_scaling", "_rotation"):
        props = lay["property_names"][lay[k]]
        assert all(n in names for n in props.ravel()), (k, props)
        loaded[k] = torch.tensor(np.stack([np.asarray(data[n], np.float32) for n in props.ravel()], -1).reshape(len(data), *props.shape))
    params = torch.load(ply.replace("point_cloud.ply", "model_params.pt"))
    for k in lay["model_params_keys"]:
        assert k in params, k
    assert params["vertices"].is_cuda and params["_alpha"].is_cuda and params["faces"].is_cuda   # used where they are: no .cuda() in the reference
    d = lambda t: t.detach().cpu()
    q = scenes.MeshGaussianParams(d(params["vertices"]), d(params["faces"]), d(params["_alpha"]), d(params["_scale"]),
                                  loaded["_features_dc"], loaded["_features_rest"], loaded["_opacity"])
    m = MeshGaussianModel.from_params(q, "cuda")
    cam = scenes.look_at_camera((2.3, 0.9, 1.1), (0, 0, 0), 320, 240)
    bg = torch.ones(3, device="cuda")
    with torch.no_grad():
        a = render_frame(m, cam.to("cuda"), bg, fused=False)[0]
        b = render_frame(ours, cam.to("cuda"), bg, fused=False)[0]
    # a 1/255 blending threshold may flip on a handful of pixels, each by at most one splat's contribution
    err = (a - b).abs().amax(dim=0)
    assert float((err > 1e-5).float().mean()) <= 1e-3 and float(err.max()) <= 2e-2, (float((err > 1e-5).float().mean()), float(err.max()))
