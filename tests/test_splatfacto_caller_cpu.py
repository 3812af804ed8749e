"""CPU: the calls the UNMODIFIED caller makes reach this package's operators and come back right.

The reference's SplatfactoModel (nerfstudio/models/splatfacto.py:28-31 imports `gsplat.project_gaussians / rasterize /
sh / _torch_impl`; :682-899 `get_outputs`) was run with `gsplat` resolving to 3dgs-deblur_b200/gsplat -- nothing of the
caller edited -- in training mode (motion blur + rolling shutter + velocity optimisation, "antialiased" opacities), in
eval mode (its second, depth-coloured rasterize_gaussians call) and in eval mode with motion blur.  Every call it made to
project_gaussians / spherical_harmonics / rasterize_gaussians is stored in tests/golden/caller_calls.npz
(tests/golden/make_golden_caller.py): the arguments, and which of them are outputs of an earlier call passed on
unchanged.  The tests replay those calls through this package, outputs linked as the caller linked them.

What runs under the operators: the C-ABI layer (`gsplat.cuda`, the 1:1 wrappers of libb200splat) is swapped for the CPU
ORACLE (oracle/splat_oracle.c, the checker the GPU parity tests hold the kernels to), so the tests run without a GPU.
Everything between the caller and the C ABI is the product's own code: the three operators' argument handling, autograd
Functions, gradient routing to velocities, the `xys.absgrad` side channel, the (rgb, alpha) return convention, the reuse
of one call's tile lists by the next.  Images are checked against the oracle chain driven directly from the recorded
arguments, gradients against central differences.

Packages the reference's import chain needs and this image lacks (viser, torchmetrics, pytorch_msssim, nerfacc) are
stubbed by _StubFinder (used by the fixture generators under tests/golden/)."""
import importlib.abc
import importlib.machinery
import inspect
import json
import os
import types

import numpy as np
import pytest
import torch

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _StubMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub


class _Stub(metaclass=_StubMeta):
    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Stub()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub()


class _StubModule(types.ModuleType):
    __path__ = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    NAMES = ("viser", "torchmetrics", "pytorch_msssim", "nerfacc")

    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in self.NAMES:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


# ---- gsplat.cuda on the oracle -------------------------------------------------------------------------------------

def _n(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else t


def _unpack(packed):
    """The stand-in "packed records": one (N, 11) float tensor xy | pix_vel | conic | colour | opacity."""
    a = packed.detach().numpy()
    return types.SimpleNamespace(xys=np.ascontiguousarray(a[:, 0:2]), pix_vels=np.ascontiguousarray(a[:, 2:4]),
                                 conics=np.ascontiguousarray(a[:, 4:7]), colors=np.ascontiguousarray(a[:, 7:10]),
                                 opac=np.ascontiguousarray(a[:, 10:11]))


def install_oracle_C(monkeypatch):
    """Every `gsplat.cuda` entry the three operators reach, computed by the CPU oracle (same signatures); returns the
    list the stand-ins log their calls to."""
    import gsplat.cuda as _C
    import gsplat._lib as L
    calls = []
    monkeypatch.setattr(L, "SYNC_CHECKS", True)  # the quaternion assert runs in Python (no device flag on the CPU)

    def project_gaussians_forward(n, means3d, scales, glob_scale, quats, lin, ang, rs, ex, viewmat, fx, fy, cx, cy, H, W, bw,
                                  clip, _vel_tensors=None, _quat_flag=None):
        lin, ang = _vel_tensors
        calls.append(("project_fwd", n, H, W, bw, float(rs), float(ex)))
        o = O.project_forward(_n(means3d), _n(scales), glob_scale, _n(quats), _n(lin), _n(ang), rs, ex, _n(viewmat), fx, fy, cx, cy, H, W, bw)
        return tuple(torch.from_numpy(o[k]) for k in ("cov3d", "xys", "depths", "pix_vels", "radii", "conics", "compensation", "num_tiles_hit"))

    def project_gaussians_backward(n, means3d, scales, glob_scale, quats, lin, ang, rs, ex, viewmat, fx, fy, cx, cy, H, W, cov3d, radii,
                                   conics, comp, v_xy, v_depth, v_pix_vel, v_conic, v_comp, _vel_tensors=None, _exact=False,
                                   _want_vel=False, _want_viewmat=False, _want_cov=True):
        """Exact mode = float64 autograd through oracle/torch_oracle.py (the reference's torch-path semantics)."""
        from oracle import torch_oracle as TO

        lin, ang = _vel_tensors
        calls.append(("project_bwd", bool(_exact), bool(_want_vel), bool(_want_viewmat)))
        t64 = lambda a: a.detach().double()
        vm4 = torch.cat([t64(viewmat).reshape(-1)[:12].view(3, 4), torch.tensor([[0, 0, 0, 1.0]], dtype=torch.float64)], 0)
        inputs = dict(means=t64(means3d), scales=t64(scales), quats=t64(quats), lin_vel=t64(lin), ang_vel=t64(ang), viewmat=vm4)
        ct = dict(v_xys=t64(v_xy), v_depths=t64(v_depth), v_pix_vels=t64(v_pix_vel), v_conics=t64(v_conic), v_compensation=t64(v_comp))
        with torch.enable_grad():  # (autograd is off inside a Function's backward)
            g, _ = TO.project_vjp(inputs, ct, glob_scale=glob_scale, rs_time=rs, exposure=ex, fx=fx, fy=fy, cx=cx, cy=cy, H=H, W=W, block_width=16)
        # (rows of Gaussians the projection culled: their cotangents are zero, but autograd through the masked-out branch
        # of the restatement yields 0 * inf there; the kernels write plain zeros)
        g = {k: torch.nan_to_num(v, nan=0.0, posinf=0.0, neginf=0.0) for k, v in g.items()}
        out = (None, None, g["v_means"].float(), g["v_scales"].float(), g["v_quats"].float())
        if _want_vel:
            out += (g["v_lin_vel"].float().reshape(3), g["v_ang_vel"].float().reshape(3))
        if _want_viewmat:
            out += (g["v_viewmat"].float()[:3],)
        return out

    def compute_sh_forward(method, n, degree, deg_use, viewdirs, coeffs):
        calls.append(("sh_fwd", method, degree, deg_use))
        return torch.from_numpy(O.sh_forward(method, deg_use, _n(viewdirs), _n(coeffs)))

    def compute_sh_backward(method, n, degree, deg_use, viewdirs, v_colors, *, out=None):
        calls.append(("sh_bwd", method, degree, deg_use))
        return torch.from_numpy(O.sh_backward(method, degree, deg_use, _n(viewdirs), _n(v_colors)))

    def pack_records(xys, pix_vels, conics, colors, opacity):
        return torch.cat([xys.detach(), pix_vels.detach(), conics.detach(), colors.detach(), opacity.detach().reshape(-1, 1)], 1).float().contiguous()

    def bin_cull(packed, depths, radii, nth, H, W, bw, S, rs, ex):
        calls.append(("bin", H, W, bw, S))
        b = O.bin_and_sort(_unpack(packed).xys, _n(depths), _n(radii), _n(nth), H, W, bw)
        return int(b["num_intersects"]), torch.from_numpy(b["gaussian_ids_sorted"]), torch.from_numpy(b["tile_bins"])

    def blend_forward_packed(H, W, bw, S, ids, bins, packed, rs, ex, bg, want_alpha=False, *, status=None):
        calls.append(("blend_fwd", S, float(rs), float(ex)))
        packed = _unpack(packed)
        img, Ts, fi = O.rasterize_forward(H, W, bw, S, _n(ids), _n(bins), packed.xys, packed.pix_vels, rs, ex, packed.conics,
                                          packed.colors, packed.opac, _n(bg))
        out = (torch.from_numpy(img), torch.from_numpy(Ts), torch.from_numpy(fi))
        return out + (torch.from_numpy(1 - Ts.mean(-1)),) if want_alpha else out

    def blend_backward_packed(n, H, W, bw, S, ids, bins, packed, rs, ex, bg, Ts, fi, v_out, v_alpha):
        calls.append(("blend_bwd", S))
        packed = _unpack(packed)
        va = np.zeros((H, W), np.float32) if v_alpha is None else _n(v_alpha)
        g = O.rasterize_backward(H, W, bw, S, _n(ids), _n(bins), packed.xys, packed.pix_vels, rs, ex, packed.conics, packed.colors,
                                 packed.opac, _n(bg), _n(Ts), _n(fi), _n(v_out), va)
        return tuple(torch.from_numpy(g[k]) for k in ("v_xy", "v_xy_abs", "v_pix_vels", "v_conic", "v_colors", "v_opacity"))

    for name, fn in list(locals().items()):
        if callable(fn) and hasattr(_C, name):
            monkeypatch.setattr(_C, name, fn)
    return calls


@pytest.fixture
def oracle_C(monkeypatch):
    return install_oracle_C(monkeypatch)


@pytest.fixture(scope="module")
def recorded(golden):
    g = golden("caller_calls.npz")
    return json.loads(str(g.pop("spec"))), g


def _replay(spec, arrays):
    """The recorded calls through this package: returns [(op, bound arguments, outputs)]."""
    import gsplat

    done, objects = [], {}

    def dec(e):
        if e["t"] == "out":
            return done[e["c"]][2][e["o"]]
        if e["t"] == "py":
            return e["v"]
        if e["id"] not in objects:  # (one tensor object where the caller passed one object twice: list reuse sees it)
            t = torch.from_numpy(arrays[e["k"]].copy())
            objects[e["id"]] = t.requires_grad_(True) if e["grad"] else t
        return objects[e["id"]]

    for c in spec["calls"]:
        fn = getattr(gsplat, c["op"])
        args, kwargs = [dec(e) for e in c["args"]], {k: dec(e) for k, e in c["kwargs"].items()}
        bound = inspect.signature(fn).bind(*args, **kwargs)
        bound.apply_defaults()
        out = fn(*args, **kwargs)
        done.append((c["op"], bound.arguments, list(out) if isinstance(out, (tuple, list)) else [out]))
    return done


def _oracle_blend(proj_args, ras_args):
    """The oracle chain on the recorded arguments: projection, binning and blend of the colours / opacities the caller
    passed."""
    p, r = {k: _n(v) for k, v in proj_args.items()}, {k: _n(v) for k, v in ras_args.items()}
    proj = O.project_forward(p["means3d"], p["scales"], p["glob_scale"], p["quats"], p["linear_velocity"], p["angular_velocity"],
                             p["rolling_shutter_time"], p["exposure_time"], p["viewmat"], p["fx"], p["fy"], p["cx"], p["cy"],
                             p["img_height"], p["img_width"], p["block_width"], p["clip_thresh"])
    H, W, bw = r["img_height"], r["img_width"], r["block_width"]
    b = O.bin_and_sort(proj["xys"], proj["depths"], proj["radii"], proj["num_tiles_hit"], H, W, bw)
    bg = np.ones(3, np.float32) if r["background"] is None else r["background"]
    img, Ts, _ = O.rasterize_forward(H, W, bw, r["blur_samples"], b["gaussian_ids_sorted"], b["tile_bins"], proj["xys"],
                                     proj["pix_vels"], r["rolling_shutter_time"], r["exposure_time"], proj["conics"],
                                     r["colors"], r["opacity"].reshape(-1, 1), bg)
    return img, 1 - Ts.mean(-1), proj


def test_unmodified_splatfacto_trains_through_this_package(recorded, oracle_C):
    spec, arrays = recorded
    spec = spec["train"]
    H, W, n = spec["H"], spec["W"], spec["n"]
    calls = _replay(spec, arrays)
    assert [c[0] for c in calls] == ["project_gaussians", "spherical_harmonics", "rasterize_gaussians"]
    (_, pa, pout), (_, sa, sout), (_, ra, rout) = calls
    img, alpha = rout
    assert img.shape == (H, W, 3) and alpha.shape == (H, W)
    # one projection (velocities carry gradients -> exact mode), one SH call at degree 3, one 5-sample blur + RS blend
    assert ("project_fwd", n, H, W, 16, 1 / 50, 1 / 60) in oracle_C and ("sh_fwd", "fast", 3, 3) in oracle_C
    assert ("blend_fwd", 5, 1 / 50, 1 / 60) in oracle_C
    ref_img, ref_alpha, proj = _oracle_blend(pa, ra)
    assert int((proj["num_tiles_hit"] > 0).sum()) > 50
    np.testing.assert_allclose(_n(img), ref_img, atol=1e-6)
    np.testing.assert_allclose(_n(alpha), ref_alpha, atol=1e-6)
    np.testing.assert_allclose(_n(sout[0]), O.sh_forward("fast", 3, _n(sa["viewdirs"]), _n(sa["coeffs"])), atol=1e-6)
    g = torch.Generator().manual_seed(1)
    v_img, v_alpha = torch.randn(H, W, 3, generator=g) / img.numel(), torch.randn(H, W, generator=g) / alpha.numel()
    torch.autograd.backward([img, alpha, sout[0]], [v_img, v_alpha, torch.randn(sout[0].shape, generator=g)])
    assert ("project_bwd", True, True, False) in oracle_C and ("blend_bwd", 5) in oracle_C and ("sh_bwd", "fast", 3, 3) in oracle_C
    leaves = {k: v for args in (pa, sa, ra) for k, v in args.items() if torch.is_tensor(v) and v.requires_grad and v.is_leaf}
    assert {"means3d", "scales", "quats", "linear_velocity", "angular_velocity", "coeffs", "colors", "opacity"} <= set(leaves)
    for k, v in leaves.items():
        assert v.grad is not None and torch.isfinite(v.grad).all() and float(v.grad.abs().sum()) > 0, k
    # the densification side channel the caller reads next (splatfacto.py:416-417)
    xys = pout[0]
    assert xys.absgrad.shape == (n, 2) and float(xys.absgrad.sum()) > 0 and (xys.absgrad >= 0).all()
    # d loss / d colour of the Gaussian with the largest gradient, by central differences of the oracle chain
    colors = ra["colors"]
    idx = int(np.argmax(np.abs(_n(colors.grad)).sum(-1)))
    vals = []
    for eps in (1e-2, -1e-2):
        c = dict(ra, colors=colors.detach().clone())
        c["colors"][idx, 0] += eps
        im, al, _ = _oracle_blend(pa, c)
        vals.append(float((im * _n(v_img)).sum() + (al * _n(v_alpha)).sum()))
    fd = (vals[0] - vals[1]) / 2e-2
    assert abs(fd - float(colors.grad[idx, 0])) < 0.05 * abs(fd) + 1e-6, (fd, float(colors.grad[idx, 0]))


def test_unmodified_splatfacto_eval_pass_renders_depth_through_this_package(recorded, oracle_C):
    """Eval mode: static camera (no velocity data, optimizer off), no blur -> S = 1, and the caller's second
    rasterize_gaussians call with depth-valued colours (splatfacto.py:881-897)."""
    spec, arrays = recorded
    spec = spec["eval"]
    H, W = spec["H"], spec["W"]
    with torch.no_grad():
        calls = _replay(spec, arrays)
    assert [c[0] for c in calls] == ["project_gaussians", "spherical_harmonics", "rasterize_gaussians", "rasterize_gaussians"]
    assert [c for c in oracle_C if c[0] == "blend_fwd"] == [("blend_fwd", 1, 0.0, 0.0)] * 2
    (_, pa, pout), _, (_, ra, (img, alpha)), (_, da, (depth_img,)) = calls
    ref_img, ref_alpha, proj = _oracle_blend(pa, ra)
    np.testing.assert_allclose(_n(img), ref_img, atol=1e-6)
    np.testing.assert_allclose(_n(alpha), ref_alpha, atol=1e-6)
    # the depth pass blends the projection's depths (what the caller coloured the Gaussians with) on a black background
    np.testing.assert_allclose(_n(da["colors"])[:, 0], proj["depths"], rtol=1e-3)
    ref_depth, _, _ = _oracle_blend(pa, da)
    np.testing.assert_allclose(_n(depth_img), ref_depth, atol=1e-5)
    covered = ref_alpha > 0.5
    d = _n(depth_img)[..., 0][covered] / ref_alpha[covered]
    assert covered.any() and np.all(d > 1.5) and np.all(d < 4.5)  # the cloud sits 2..4 units in front


@pytest.mark.parametrize("rolling_shutter", [False, True])
def test_eval_depth_pass_reuses_the_colour_pass_lists(recorded, oracle_C, monkeypatch, rolling_shutter):
    """Eval with motion blur: the caller's second (static, depth-coloured) rasterize_gaussians call (splatfacto.py:881-897)
    bins nothing when the colour pass had no rolling shutter and an odd sample count -- its lists contain the static
    lists (gsplat/rasterize.py) -- and bins again when it had.  Same depth image either way."""
    spec, arrays = recorded
    spec = spec["blur_eval_rs" if rolling_shutter else "blur_eval"]
    import gsplat.rasterize as R
    R._last_lists.clear()
    with torch.no_grad():
        calls = _replay(spec, arrays)
    blends = [c for c in oracle_C if c[0] == "blend_fwd"]
    assert blends[0][1] == 5 and blends[1] == ("blend_fwd", 1, 0.0, 0.0)
    assert len([c for c in oracle_C if c[0] == "bin"]) == (2 if rolling_shutter else 1)
    del oracle_C[:]
    monkeypatch.setenv("B200SPLAT_NO_LIST_REUSE", "1")
    R._last_lists.clear()
    with torch.no_grad():
        calls2 = _replay(spec, arrays)
    assert len([c for c in oracle_C if c[0] == "bin"]) == 2
    for (_, _, out), (_, _, out2) in zip(calls[2:], calls2[2:]):
        assert all(torch.equal(a, b) for a, b in zip(out, out2))
    _, ra, (img, alpha) = calls[2]
    d = calls[3][2][0][..., 0][alpha > 0.5]  # (blurred coverage can exceed the static one at the rim: depth 0 there)
    assert d.numel() > 0 and float((d / alpha[alpha > 0.5]).min()) > 1.0 and float((d / alpha[alpha > 0.5]).max()) < 4.5
