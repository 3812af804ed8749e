"""Generates tests/golden/caller_calls.npz: the calls the unmodified Splatfacto caller makes into this package.

The reference's SplatfactoModel (nerfstudio/models/splatfacto.py:682-899, `get_outputs`) is imported with `gsplat`
resolving to 3dgs-deblur_b200/gsplat and the C-ABI layer on the CPU oracle (tests/test_splatfacto_caller_cpu.py), and
run in training mode (motion blur + rolling shutter + velocity optimisation, "antialiased" opacities), in eval mode (its
second, depth-coloured rasterize_gaussians call) and in eval mode with motion blur, with and without rolling shutter.
Every call it makes to project_gaussians / spherical_harmonics / rasterize_gaussians is recorded: positional and keyword
arguments, each tensor either as "the i-th output of an earlier call" (what the caller passes on unchanged) or as a
value, with
its requires_grad flag and which argument tensors are one object.  tests/test_splatfacto_caller_cpu.py replays the calls.  viser / torchmetrics / pytorch_msssim /
nerfacc (not on the render path) are stubbed; populate_modules needs scikit-learn (k_nearest_sklearn).

    python tests/golden/make_golden_caller.py <nerfstudio source directory>   # the fixture it writes is committed
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "3dgs-deblur_b200"))
OPS = ("project_gaussians", "spherical_harmonics", "rasterize_gaussians")


def _make_model(sf, SceneBox, n, training, velocity_opt, seed=3):
    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed)
    pts = (torch.rand(n, 3, generator=g) - 0.5) * 2.0 + torch.tensor([0.0, 0.0, -3.0])  # in front of an OpenGL camera at the origin
    cols = torch.rand(n, 3, generator=g) * 255
    cfg = sf.SplatfactoModelConfig(rasterize_mode="antialiased", blur_samples=5, background_color="white", num_downscales=0,
                                   sh_degree=3, sh_degree_interval=1)
    cfg.camera_velocity_optimizer.enabled = velocity_opt
    box = SceneBox(aabb=torch.tensor([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]]))
    real_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self  # populate_modules moves the seed colours to "cuda" (splatfacto.py:223)
    try:
        model = sf.SplatfactoModel(cfg, scene_box=box, num_train_data=2, seed_points=(pts, cols))
    finally:
        torch.Tensor.cuda = real_cuda
    model.step = 10  # all SH degrees on (splatfacto.py:844)
    model.train(training)
    with torch.no_grad():  # something to render: visible sizes, mixed opacities, non-trivial higher SH bands
        model.gauss_params["scales"].copy_(torch.log(torch.full((n, 3), 0.05) * (0.5 + torch.rand(n, 3, generator=g))))
        model.gauss_params["opacities"].copy_(torch.randn(n, 1, generator=g))
        model.gauss_params["features_rest"].copy_(0.1 * torch.randn(n, 15, 3, generator=g))
    return model


def _camera(Cameras, H, W, meta, vel):
    return Cameras(camera_to_worlds=torch.eye(4)[:3].unsqueeze(0).clone(), fx=W / 2.0, fy=W / 2.0, cx=W / 2.0, cy=H / 2.0,
                   width=W, height=H, velocities=vel, metadata=meta)  # (cam_idx: camera_optimizers.py:248)


class Recorder:
    def __init__(self, arrays):
        self.arrays, self.calls, self.outputs, self.seen, self.seen_enc = arrays, [], [], [], []

    def _enc(self, x):
        if torch.is_tensor(x):
            for ci, outs in enumerate(self.outputs):
                for oi, o in enumerate(outs):
                    if o is x:
                        return {"t": "out", "c": ci, "o": oi}
            for i, o in enumerate(self.seen):  # the same tensor object as in an earlier call
                if o is x:
                    return dict(self.seen_enc[i])
            a = x.detach().cpu().numpy()
            a = a.astype(np.float32) if a.dtype.kind == "f" else a.astype(np.int32)
            key = hashlib.sha256(a.tobytes() + str(a.shape).encode()).hexdigest()[:16]
            self.arrays[key] = a
            self.seen.append(x)
            self.seen_enc.append({"t": "arr", "k": key, "grad": bool(x.requires_grad), "id": len(self.seen)})
            return dict(self.seen_enc[-1])
        if x is None or isinstance(x, (bool, int, float, str)):
            return {"t": "py", "v": x}
        raise TypeError(type(x))

    def wrap(self, name, fn):
        def call(*args, **kwargs):
            self.calls.append({"op": name, "args": [self._enc(a) for a in args],
                               "kwargs": {k: self._enc(v) for k, v in kwargs.items()}})
            out = fn(*args, **kwargs)
            self.outputs.append(list(out) if isinstance(out, (tuple, list)) else [out])
            return out
        return call


def main(nerfstudio_dir):
    sys.path.insert(0, nerfstudio_dir)
    from _pytest.monkeypatch import MonkeyPatch
    from test_splatfacto_caller_cpu import _StubFinder, install_oracle_C

    sys.meta_path.insert(0, _StubFinder())
    import nerfstudio.models.splatfacto as sf
    from nerfstudio.cameras.cameras import Cameras
    from nerfstudio.data.scene_box import SceneBox

    motion = torch.tensor([[0.3, -0.2, 0.1, 0.05, 0.4, -0.3]])
    scenarios = {  # name: (n, training, velocity optimiser, H, W, camera metadata, velocities)
        "train": (300, True, True, 48, 64, dict(exposure_time=1 / 60, rolling_shutter_time=1 / 50, cam_idx=0), motion),
        "eval": (300, False, False, 32, 48, None, None),
        "blur_eval": (300, False, False, 32, 48, dict(exposure_time=1 / 60, cam_idx=0), motion),
        "blur_eval_rs": (300, False, False, 32, 48, dict(exposure_time=1 / 60, rolling_shutter_time=1 / 50, cam_idx=0), motion),
    }
    arrays, spec = {}, {}
    for name, (n, training, vel_opt, H, W, meta, vel) in scenarios.items():
        mp = MonkeyPatch()
        try:
            install_oracle_C(mp)
            rec = Recorder(arrays)
            for op in OPS:
                mp.setattr(sf, op, rec.wrap(op, getattr(sf, op)))
            model = _make_model(sf, SceneBox, n, training=training, velocity_opt=vel_opt)
            with torch.set_grad_enabled(training):
                out = model.get_outputs(_camera(Cameras, H, W, meta, vel))
            assert out["rgb"].shape == (H, W, 3)
            spec[name] = {"n": n, "H": H, "W": W, "calls": rec.calls}
        finally:
            mp.undo()
    np.savez_compressed(os.path.join(HERE, "caller_calls.npz"), spec=np.asarray(json.dumps(spec)), **arrays)


if __name__ == "__main__":
    main(sys.argv[1])
