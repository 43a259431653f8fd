"""Generate tests/golden/reference_render_*.npz by running the REFERENCE's own Python (its renderers, GaussianMeshModel and
GaussianModel._load_ply) on the CPU.  tests/test_gpu_reference_render.py compares the GPU path against these files, so the
reference is never needed at test time.

    python tests/golden/make_reference_render_golden.py <reference checkout>

The rasterizer the reference imports (`diff_gaussian_rasterization`) is replaced by a recorder: it keeps the settings and
tensors that render() hands it.  The rasterizer's own gradients come from the CPU oracle (oracle/gms_oracle.c, built by
__graft_entry__.build()) and are pushed back through the reference's autograd graph, so the stored gradients of the raw
parameters are the reference's expansion backward fed by an independent rasterizer backward.  The reference hard-codes
device="cuda" in a few places; those allocations are mapped to the CPU while it runs (the arithmetic is untouched).

The test recomputes everything on the full scene; to keep the fixtures small, each stored array holds a fixed sample of
its rows (`rows<n>` lists the rows kept of an array whose leading dimension is n), and the raw parameters the reference
started from are stored as SHA-256 digests of the arrays the scene generator returns.

What is stored (scene, camera and cotangent seeds are the ones the test uses):
  reference_render_static.npz    render() on a stock GaussianMeshModel (create_from_pcd + update_alpha +
                                 prepare_scaling_rot): raster settings, the Gaussians it rasterizes, raw-parameter gradients
  reference_expansion_k5.npz     stock update_alpha / prepare_scaling_rot values and the _alpha gradient through `alpha`
  reference_render_animated.npz  gaussian_animated_renderer.render at three times of transform_hotdog_fly
  reference_ply_layout.npz       which PLY property _load_ply puts at each position of each tensor, and which
                                 model_params.pt keys GaussianMeshModel.load_ply reads
  reference_rasterizer_imports.npz  the names each renderer module imports from diff_gaussian_rasterization
"""
import hashlib
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "gaussian-mesh-splatting_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

from gms_b200 import io_ply, scenes  # noqa: E402
from helpers import settings_from_camera  # noqa: E402
from oracle import raster  # noqa: E402

RECORDED = []


class _Settings(types.SimpleNamespace):
    pass


class _RecordingRasterizer:
    def __init__(self, raster_settings):
        self.s = raster_settings

    def __call__(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None):
        RECORDED.append(dict(settings=self.s, means3D=means3D, opacities=opacities, shs=shs, scales=scales, rotations=rotations))
        H, W = int(self.s.image_height), int(self.s.image_width)
        return torch.zeros(3, H, W), torch.zeros(means3D.shape[0], dtype=torch.int32), torch.zeros(1, H, W)


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m


def _cpu_device(k):
    if str(k.get("device", "")).startswith("cuda"):
        k["device"] = "cpu"
    return k


def _map_cuda_to_cpu():
    for name in ("zeros", "ones", "zeros_like", "tensor"):
        f = getattr(torch, name)
        setattr(torch, name, (lambda f: lambda *a, **k: f(*a, **_cpu_device(k)))(f))
    torch.Tensor.cuda = lambda self, *a, **k: self


def _import_reference(ref_root):
    _stub("plyfile", PlyData=object, PlyElement=object)
    _stub("simple_knn")
    _stub("simple_knn._C", distCUDA2=None)
    _stub("trimesh")
    _stub("smplx")
    _stub("smplx.lbs", lbs=None, batch_rodrigues=None, vertices2landmarks=None, find_dynamic_lmk_idx_and_bcoords=None)
    _stub("smplx.utils", Struct=object, to_tensor=None, to_np=None, rot_mat_to_euler=None)
    _stub("diff_gaussian_rasterization", GaussianRasterizationSettings=_Settings, GaussianRasterizer=_RecordingRasterizer)
    sys.path.insert(0, ref_root)
    from games.mesh_splatting.scene.gaussian_mesh_model import GaussianMeshModel
    from games.mesh_splatting.utils.graphics_utils import MeshPointCloud
    import renderer.gaussian_renderer as r_static
    import renderer.gaussian_animated_renderer as r_anim
    import scene.gaussian_model as sgm
    from scene.cameras import MiniCam
    return types.SimpleNamespace(GaussianMeshModel=GaussianMeshModel, MeshPointCloud=MeshPointCloud, render=r_static.render,
                                 render_animated=r_anim.render, MiniCam=MiniCam, sgm=sgm)


PIPE = types.SimpleNamespace(debug=False, antialiasing=False, compute_cov3D_python=False, convert_SHs_python=False)


def _reference_model(ref, p):
    """Stock GaussianMeshModel through its own create_from_pcd, then given the appearance of `p` (as the test did)."""
    F, K = p._alpha.shape[:2]
    tri = p.vertices[p.faces]
    alpha_n = torch.relu(p._alpha) + 1e-8
    alpha_n = alpha_n / alpha_n.sum(-1, keepdim=True)
    pts = torch.matmul(alpha_n, tri).reshape(-1, 3)
    pcd = ref.MeshPointCloud(alpha=p._alpha.clone(), points=pts, colors=np.full((F * K, 3), 0.5, np.float32),
                             normals=np.zeros((F * K, 3), np.float32), vertices=p.vertices.clone(), faces=p.faces.numpy(),
                             transform_vertices_function=None, triangles=tri)
    m = ref.GaussianMeshModel(3)
    m.create_from_pcd(pcd, 1.0)
    with torch.no_grad():
        m._opacity.copy_(p._opacity); m._features_dc.copy_(p._features_dc); m._features_rest.copy_(p._features_rest)
        m._scale.copy_(p._scale)
    m.active_sh_degree = 3
    m.update_alpha(); m.prepare_scaling_rot()
    return m


def _minicam(ref, cam):
    return ref.MiniCam(cam.image_width, cam.image_height, cam.FoVy, cam.FoVx, scenes.ZNEAR, scenes.ZFAR,
                       cam.world_view_transform, cam.full_proj_transform)


def _f32(t):
    return np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)


def _settings_arrays(s, prefix=""):
    return {prefix + "image_height": np.int64(s.image_height), prefix + "image_width": np.int64(s.image_width),
            prefix + "tanfovx": np.float64(s.tanfovx), prefix + "tanfovy": np.float64(s.tanfovy), prefix + "bg": _f32(s.bg),
            prefix + "scale_modifier": np.float64(s.scale_modifier), prefix + "viewmatrix": _f32(s.viewmatrix),
            prefix + "projmatrix": _f32(s.projmatrix), prefix + "sh_degree": np.int64(s.sh_degree), prefix + "campos": _f32(s.campos),
            prefix + "prefiltered": np.bool_(s.prefiltered), prefix + "debug": np.bool_(s.debug),
            prefix + "antialiasing": np.bool_(s.antialiasing)}


def _oracle_cotangents(rec, cam, dC):
    """Rasterizer gradients of sum(image * dC) at the recorded inputs, from the CPU oracle."""
    S = settings_from_camera(cam, bg=(1, 1, 1))
    st = raster.forward(S, rec["means3D"].detach(), rec["opacities"].detach(), shs=rec["shs"].detach().contiguous(),
                        scales=rec["scales"].detach(), rotations=rec["rotations"].detach())
    g = raster.backward(st, dC)
    return [torch.tensor(g[k]).reshape(rec[n].shape) for k, n in (("dL_dmeans3D", "means3D"), ("dL_dscales", "scales"),
                                                                   ("dL_drotations", "rotations"), ("dL_dopacity", "opacities"))]


def _dC(seed, cam):
    rs = np.random.RandomState(seed)
    return (rs.randn(3, cam.image_height, cam.image_width) / (cam.image_width * cam.image_height)).astype(np.float32)


N_ROWS = 256


def _raw(p):
    return {f"digest{k}": np.array(hashlib.sha256(getattr(p, k).numpy().tobytes()).hexdigest())
            for k in ("vertices", "faces", "_alpha", "_scale", "_opacity")}


def _sampled(**arrays):
    """A fixed, seeded sample of each array's rows, and the rows kept (rows<n> for a leading dimension n)."""
    out = {}
    for name, a in arrays.items():
        n = a.shape[0]
        rows = np.sort(np.random.RandomState(n).choice(n, min(n, N_ROWS), replace=False)).astype(np.int32)
        out[f"rows{n}"], out[name] = rows, np.ascontiguousarray(a[rows])
    return out


def static(ref):
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=3, seed=11, trained_like=True)
    cam = scenes.look_at_camera((2.3, 0.9, 1.1), (0, 0, 0), 400, 304)
    m = _reference_model(ref, p)
    RECORDED.clear()
    ref.render(_minicam(ref, cam), m, PIPE, torch.ones(3))
    rec = RECORDED[0]
    assert torch.equal(rec["shs"], torch.cat([p._features_dc, p._features_rest], 1))
    outs = [rec[n] for n in ("means3D", "scales", "rotations", "opacities")]
    torch.autograd.backward(outs, _oracle_cotangents(rec, cam, _dC(3, cam)))
    out = dict(_raw(p), **_settings_arrays(rec["settings"]),
               **_sampled(means3D=_f32(rec["means3D"]), scales=_f32(rec["scales"]), rotations=_f32(rec["rotations"]),
                          opacities=_f32(rec["opacities"]), **{f"grad{k}": _f32(getattr(m, k).grad) for k in ("vertices", "_alpha", "_scale", "_opacity")}))
    np.savez_compressed(os.path.join(HERE, "reference_render_static.npz"), **out)


def expansion_k5(ref):
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=5, seed=12, trained_like=True)
    m = _reference_model(ref, p)
    g = torch.tensor(np.random.RandomState(12).randn(*m.alpha.shape).astype(np.float32))
    (m.alpha * g).sum().backward()
    out = dict(_raw(p), **_sampled(alpha=_f32(m.alpha), triangles=_f32(m.triangles), _xyz=_f32(m._xyz), _scaling=_f32(m._scaling),
                                   _rotation=_f32(m._rotation), grad_alpha=_f32(m._alpha.grad)))
    np.savez_compressed(os.path.join(HERE, "reference_expansion_k5.npz"), **out)


ANIMATED_TIMES = (0.0, 2.1, 5.7)


def animated(ref):
    p = scenes.init_mesh_gaussians(*scenes.icosphere(3), K=3, seed=13, trained_like=True)
    cam = scenes.look_at_camera((2.6, -0.7, 0.8), (0, 0, 0), 368, 272)
    out = _raw(p)
    for i, t in enumerate(ANIMATED_TIMES):
        m = _reference_model(ref, p)
        tri = scenes.transform_hotdog_fly(p.vertices, t)[p.faces]
        RECORDED.clear()
        ref.render_animated(None, tri, _minicam(ref, cam), m, PIPE, torch.ones(3))
        rec = RECORDED[0]
        outs = [rec[n] for n in ("means3D", "scales", "rotations", "opacities")]
        cot = _oracle_cotangents(rec, cam, _dC(4, cam))
        keep = [(o, c) for o, c in zip(outs, cot) if o.requires_grad]     # rotation is a constant of the triangles here
        torch.autograd.backward([o for o, _ in keep], [c for _, c in keep])
        if i == 0:
            out.update(_settings_arrays(rec["settings"]))
        out.update(_sampled(**{f"t{i}_means3D": _f32(rec["means3D"]), f"t{i}_scales": _f32(rec["scales"]),
                               f"t{i}_rotations": _f32(rec["rotations"]),
                               **{f"t{i}_grad{k}": _f32(getattr(m, k).grad) for k in ("_alpha", "_scale", "_opacity")}}))
        assert m.vertices.grad is None
    out["times"] = np.float64(ANIMATED_TIMES)
    np.savez_compressed(os.path.join(HERE, "reference_render_animated.npz"), **out)


def ply_layout(ref):
    """Write a checkpoint with this project's writer, replace every PLY value by the index of its column, and load it with
    the reference's GaussianMeshModel.load_ply: each loaded element then names the PLY property it was read from."""
    p = scenes.init_mesh_gaussians(*scenes.icosphere(1), K=3, seed=31, trained_like=True)
    m = _reference_model(ref, p)
    with tempfile.TemporaryDirectory() as tmp:
        ply = os.path.join(tmp, "point_cloud", "iteration_30000", "point_cloud.ply")
        io_ply.save_mesh_model(ply, m)
        data, names = io_ply.read_ply_vertices(ply)
        with open(ply, "rb") as f:
            raw = f.read()
        header = raw[:raw.index(b"end_header\n") + len(b"end_header\n")]
        codes = np.tile(np.arange(len(names), dtype="<f4"), (len(data), 1))
        with open(ply, "wb") as f:
            f.write(header)
            codes.tofile(f)

        class _El:
            def __init__(self, data, names):
                self.data, self.properties = data, [types.SimpleNamespace(name=n) for n in names]

            def __getitem__(self, k):
                return self.data[k]

        class _PlyData:
            def __init__(self, elements):
                self.elements = elements

            @staticmethod
            def read(path):
                d, n = io_ply.read_ply_vertices(path)
                return _PlyData([_El(d, n)])

        read_keys = []

        class _LoggedDict(dict):
            def __getitem__(self, k):
                read_keys.append(k)
                return dict.__getitem__(self, k)

        ref.sgm.PlyData = _PlyData
        load = torch.load
        ref_torch = sys.modules["games.mesh_splatting.scene.gaussian_mesh_model"].torch
        ref_torch.load = lambda *a, **k: _LoggedDict(load(*a, **k))
        try:
            r = ref.GaussianMeshModel(3)
            r.load_ply(ply)
        finally:
            ref_torch.load = load
    out = {"property_names": np.array(names)}
    for k in ("_xyz", "_features_dc", "_features_rest", "_opacity", "_scaling", "_rotation"):
        col = getattr(r, k).detach().numpy()
        assert (col == col[:1]).all()
        out[k] = np.asarray(col[0], dtype=np.int64)        # per-Gaussian layout: PLY column index at each position
    out["model_params_keys"] = np.array(sorted(set(read_keys)))
    np.savez_compressed(os.path.join(HERE, "reference_ply_layout.npz"), **out)


def rasterizer_imports(ref):
    """The names each renderer module binds from `diff_gaussian_rasterization`."""
    stub = sys.modules["diff_gaussian_rasterization"]
    out = {}
    for mod in ("renderer.gaussian_renderer", "renderer.gaussian_animated_renderer"):
        m = sys.modules[mod]
        out[mod] = np.array(sorted(n for n in dir(stub) if not n.startswith("_") and getattr(m, n, None) is getattr(stub, n)))
    np.savez_compressed(os.path.join(HERE, "reference_rasterizer_imports.npz"), **out)


if __name__ == "__main__":
    ref = _import_reference(os.path.abspath(sys.argv[1]))
    rasterizer_imports(ref)
    _map_cuda_to_cpu()
    static(ref); expansion_k5(ref); animated(ref); ply_layout(ref)
    for f in sorted(os.listdir(HERE)):
        if f.startswith("reference_") and f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
