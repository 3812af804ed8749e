"""CPU: oracle/densify_oracle.py (the restatement the GPU test holds gsplat.densify to) against the reference ITSELF --
the real SplatfactoModel.after_train / refinement_after (nerfstudio/models/splatfacto.py:408-531) with real
torch.optim.Adam optimizers, on the same parameters, statistics, step and random draw.

The inputs are generated here from a seed; what the reference computed from them is stored in
tests/golden/densify_refinement.npz (tests/golden/make_golden_densify.py, which runs the reference): the arrays the
test holds to exact equality as SHA-256 digests of their bytes; the means after a split, which it compares with a
tolerance, in full.  The digests assume that torch's CPU kernels give the oracle's float32 results bit for bit on every
x86-64 host the suite runs on, as exact equality with the reference did before."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import densify_oracle as DO

# the reference's parameter names, in the order of SplatfactoModel.get_gaussian_param_groups (splatfacto.py:638-644)
NAMES = {"means": "means", "scales": "log_scales", "quats": "quats", "features_dc": "features_dc",
         "features_rest": "features_rest", "opacities": "opacity_logit"}
N, H, W, NUM_TRAIN_DATA, IMAGES = 3000, 600, 800, 20, 3
# (step -> which branch): densify with every cull criterion; densify before the "too big" culls switch on; the step of an
# opacity reset; cull-only after stop_split_at; a step the schedule skips
STEPS = [3500, 2500, 3100, 15100, 3000 + 50]


def digest(t):
    """SHA-256 of a tensor's float32 / int bytes; + 0 makes -0.0 and 0.0 one value, as exact assert_close has them."""
    a = t.detach().cpu().numpy()
    if a.dtype.kind == "f":
        a = a.astype(np.float32) + np.float32(0)
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def make_inputs(seed):
    """Parameters (reference names) after one Adam step on a random gradient, that step's optimizers, and the generator
    the statistics are drawn from next.  A spread of sizes / opacities so that every branch (split, dup, three kinds of
    cull) is taken."""
    g = torch.Generator().manual_seed(seed)
    quats = torch.randn(N, 4, generator=g)
    params = {
        "means": (torch.rand(N, 3, generator=g) - 0.5) * 2.0,
        "scales": torch.log(10.0 ** (torch.rand(N, 3, generator=g) * 2.6 - 3.0)),
        "quats": quats / quats.norm(dim=-1, keepdim=True),
        "features_dc": torch.rand(N, 3, generator=g),
        "features_rest": 0.1 * torch.randn(N, 15, 3, generator=g),
        "opacities": 3.0 * torch.randn(N, 1, generator=g),
    }
    params = {k: torch.nn.Parameter(v) for k, v in params.items()}
    opts = {k: torch.optim.Adam([v], lr=1e-3, eps=1e-15) for k, v in params.items()}
    for k in NAMES:  # one real step so every optimizer carries non-trivial moments
        params[k].grad = torch.randn(params[k].shape, generator=g)
        opts[k].step()
    return params, opts, g


def draw_image_stats(g):
    """One image's radii and |d loss / d xy| (what after_train reads)."""
    radii = (torch.rand(N, generator=g) * 60).int() * (torch.rand(N, generator=g) < 0.6).int()
    absgrad = torch.rand(N, 2, generator=g) * 2e-3
    return radii, absgrad


def moments_of(opt):
    st = opt.state[opt.param_groups[0]["params"][0]]
    return st["exp_avg"], st["exp_avg_sq"]


@pytest.fixture(scope="module")
def gold(golden):
    return golden("densify_refinement.npz")


@pytest.mark.parametrize("step", STEPS)
def test_oracle_matches_the_reference_refinement(gold, step):
    from gsplat.densify import DensifyConfig

    params, opts, g = make_inputs(seed=step)
    dcfg = DensifyConfig()
    for f in dcfg.__dataclass_fields__:  # the port's defaults ARE the reference's
        assert getattr(dcfg, f) == gold["config_" + f].item(), f
    stats = {}
    if step < dcfg.stop_split_at:
        for _ in range(IMAGES):
            radii, absgrad = draw_image_stats(g)
            DO.accumulate(stats, absgrad, radii, H, W)
        for k in ("grad_norm", "vis_counts", "max_2d"):
            assert digest(stats[k]) == str(gold[f"{step}_stats_{k}"]), k
    p = {NAMES[k]: v.detach().clone() for k, v in params.items()}
    m = {NAMES[k]: tuple(x.clone() for x in moments_of(o)) for k, o in opts.items()}
    torch.manual_seed(77)
    new_p, new_m, info = DO.refine(p, m, stats, dcfg, step, NUM_TRAIN_DATA, (H, W))
    assert new_p["means"].shape[0] == int(gold[f"{step}_num_points"])
    if step in (3500, 2500):
        assert info["splits"] > 50 and info["dups"] > 50 and info["after"] != N
    if step == 15100:
        assert info is not None and not info["densified"] and info["after"] < N
    for k in NAMES:
        ref = gold[f"{step}_{k}"] if k != "means" else gold[f"{step}_means"]
        if ref.dtype.kind == "f":
            # (children's means go through quat -> rotation matrix: last-bit differences between two spellings of it)
            torch.testing.assert_close(new_p[NAMES[k]], torch.from_numpy(ref), rtol=0, atol=2e-6)
        else:
            assert digest(new_p[NAMES[k]]) == str(ref), k
        assert digest(new_m[NAMES[k]][0]) == str(gold[f"{step}_{k}_exp_avg"]), k
        assert digest(new_m[NAMES[k]][1]) == str(gold[f"{step}_{k}_exp_avg_sq"]), k
