"""Generates tests/golden/densify_refinement.npz: the reference's adaptive density control on the inputs of
tests/test_densify_cpu.py.

The reference's SplatfactoModel (nerfstudio/models/splatfacto.py) is built on the CPU, given the test's parameters and
Adam optimizers (the test's own seed), fed the test's per-image statistics through `after_train` and refined by
`refinement_after` under the test's random seed.  Stored: its densification defaults, the statistics it accumulated, the
point count and, per Gaussian parameter, the digest of the refined values and of both Adam moments -- the refined means
in full where the refinement split Gaussians (the test compares them with a tolerance).  viser / torchmetrics /
pytorch_msssim / nerfacc (not on this path) are stubbed as in tests/test_splatfacto_caller_cpu.py; populate_modules needs
scikit-learn (k_nearest_sklearn).

    python tests/golden/make_golden_densify.py <nerfstudio source directory>   # the fixture it writes is committed
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "3dgs-deblur_b200"))


def main(nerfstudio_dir):
    sys.path.insert(0, nerfstudio_dir)
    from test_densify_cpu import H, IMAGES, N, NAMES, NUM_TRAIN_DATA, STEPS, W, digest, draw_image_stats, make_inputs
    from test_splatfacto_caller_cpu import _StubFinder

    sys.meta_path.insert(0, _StubFinder())
    import nerfstudio.models.splatfacto as sf
    from nerfstudio.data.scene_box import SceneBox

    from gsplat.densify import DensifyConfig

    out = {}
    for step in STEPS:
        params, opts, g = make_inputs(seed=step)
        real_cuda = torch.Tensor.cuda
        torch.Tensor.cuda = lambda self, *a, **k: self  # populate_modules moves the seed colours to "cuda"
        try:
            model = sf.SplatfactoModel(sf.SplatfactoModelConfig(sh_degree=3), num_train_data=NUM_TRAIN_DATA,
                                       scene_box=SceneBox(aabb=torch.tensor([[-1.0, -1, -1], [1.0, 1, 1]])),
                                       seed_points=(params["means"].detach().clone(), torch.zeros(N, 3)))
        finally:
            torch.Tensor.cuda = real_cuda
        with torch.no_grad():
            for k in NAMES:
                model.gauss_params[k].copy_(params[k])
        ref_opts = {}
        for k, v in model.get_gaussian_param_groups().items():
            ref_opts[k] = torch.optim.Adam(v, lr=1e-3, eps=1e-15)
            ref_opts[k].load_state_dict(opts[k].state_dict())
        model.step = step
        cfg = model.config
        if step == STEPS[0]:
            for f in DensifyConfig.__dataclass_fields__:
                out["config_" + f] = np.asarray(getattr(cfg, f))
        if step < cfg.stop_split_at:
            for _ in range(IMAGES):
                radii, absgrad = draw_image_stats(g)
                model.radii = radii
                model.xys = types.SimpleNamespace(absgrad=absgrad)
                model.last_size = (H, W)
                model.after_train(model.step)
            for k, v in (("grad_norm", model.xys_grad_norm), ("vis_counts", model.vis_counts), ("max_2d", model.max_2Dsize)):
                out[f"{step}_stats_{k}"] = np.asarray(digest(v))
        torch.manual_seed(77)
        model.refinement_after(types.SimpleNamespace(optimizers=ref_opts), step)
        assert model.xys_grad_norm is None and model.max_2Dsize is None
        out[f"{step}_num_points"] = np.asarray(model.num_points)
        means = model.gauss_params["means"].detach()
        # split children (the count grew): their means may differ in the last bits, the test compares them with a tolerance
        out[f"{step}_means"] = means.numpy().astype(np.float32) if model.num_points > N else np.asarray(digest(means))
        for k, o in ref_opts.items():
            st = o.state[o.param_groups[0]["params"][0]]
            if k != "means":
                out[f"{step}_{k}"] = np.asarray(digest(model.gauss_params[k]))
            out[f"{step}_{k}_exp_avg"] = np.asarray(digest(st["exp_avg"]))
            out[f"{step}_{k}_exp_avg_sq"] = np.asarray(digest(st["exp_avg_sq"]))
    np.savez_compressed(os.path.join(HERE, "densify_refinement.npz"), **out)


if __name__ == "__main__":
    main(sys.argv[1])
