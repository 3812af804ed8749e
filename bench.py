#!/usr/bin/env python
"""bench.py -- train images/s (fwd + bwd + optimizer) of the rasterizer hot path on BASELINE config 2
(synthetic stand-in for synthetic-mb 'cozyroom': 300k Gaussians, 800x800, 5 motion-blur samples).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path (libb200splat)
    python bench.py --impl reference ...                          # CPU arm: the oracle port on the host cores
    python bench.py --impl refgpu ...                             # extra: unmodified reference CUDA ext (oracle/_ref)

One JSON line on stdout (rank 0).  A "step" = one image per rank: project + SH + tile binning + blur blend
forward, L1 loss, full backward, one gradient allreduce (N > 1) and a fused Adam step -- the render block of
splatfacto.py:816-880 driven through the public gsplat operators.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "3dgs-deblur_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "train images/sec (fwd+bwd) at N=5 blur samples"


def workload_string(cfg, N, W, H, S):
    """One spelling of the workload for every arm (the driver compares the arms' `config.workload`)."""
    return f"{cfg}: {N} Gaussians, {W}x{H}, S={S} blur samples (synthetic stand-in of SURVEY 8d + free space around the cameras)"


def bench_config(cfg, N, W, H, S):
    """`config` of the JSON line: identical for every arm run on the same workload (arm-specific facts go to `details`)."""
    return {"workload": workload_string(cfg, N, W, H, S),
            "step": "1 image per GPU per step: projection + SH + tile binning + blur blend forward, L1 loss, full backward",
            "l2": "no explicit flush: the per-step working set (59 floats x N x {param, grad, 2 Adam moments} = %d MB, + the "
                  "images) exceeds the 126 MB L2 and every step renders a different camera" % (59 * N * 16 // 2**20)}


def usable_cores():
    """Host threads this process may really use: the affinity mask, capped by a cgroup CPU quota if one is set (a
    128-thread OpenMP team on a 16-CPU quota is throttled, not faster)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def _layout(operators):
    """FlatGaussians SH layout each operator set reads: fused kernels take sh_dc / sh_rest apart, spherical_harmonics one block."""
    return "split" if operators == "fused" else "block"


def _api(operators):
    if operators == "fused":
        return ("C ABI raw-parameter kernels: b200_fused_geometry_forward + b200_bin_cull_* | b200_fused_colors_forward + "
                "b200_blend_*_packed + b200_fused_preprocess_backward (gsplat.dp.fused_geometry_phase / fused_shading_phase)")
    return "drop-in gsplat.project_gaussians / spherical_harmonics / rasterize_gaussians under autograd"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400,
                    help="timed steps of the headline and of the end-to-end loop; the side figures beside them (other "
                         "operator set, reference comparators) time their own fixed counts and report them")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "refgpu"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--n", type=int, default=None, help="override the Gaussian count (debug only)")
    ap.add_argument("--no-vel-grad", action="store_true", help="camera velocities constant (reference CUDA-path mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--images", type=int, default=16, help="distinct training images per rank (N > 1: the cost-aware batching groups 16 x N images; more images = tighter groups)")
    ap.add_argument("--profile", action="store_true", help="also report the summed device time of all kernels per step (CUPTI)")
    ap.add_argument("--loss", default="l1", choices=["l1", "photometric"],
                    help="l1 = BASELINE's loss; photometric = Splatfacto's 0.8 L1 + 0.2 (1 - SSIM) through the fused kernels")
    ap.add_argument("--sh-chunks", type=int, default=None,
                    help="pieces of the SH block in the gradient exchange (N > 1); default 1 (measured at N=4, c2: one 57.6 MB allreduce 163 us, two halves 2 x 115 us)")
    ap.add_argument("--optimizer", default="b200", choices=["b200", "torch"], help="FlatAdam kernel or torch's fused Adam")
    ap.add_argument("--no-fused-path", action="store_true", help="skip the extra fused-operator measurement")
    ap.add_argument("--mode", default="image", choices=["image", "scene"],
                    help="image = every rank renders another image of ONE scene, one gradient exchange per step (BASELINE configs "
                         "2-5); scene = whole scenes shard across the GPUs (BASELINE config 5: `--config c5 --mode scene`): rank r "
                         "trains scene r mod --scenes, ranks that share a scene form an image-sharded group, no exchange between scenes")
    ap.add_argument("--scenes", type=int, default=5, help="number of independent scenes in --mode scene")
    ap.add_argument("--no-balance", action="store_true",
                    help="N > 1: keep the default image -> (step, rank) assignment instead of grouping images of similar cost "
                         "(gsplat.dp.balanced_assignment) so that no rank waits for a much slower one")
    ap.add_argument("--timeline", default=None, help="rank 0: write a CUPTI kernel timeline (start, duration, stream, name) of 6 steps to this file")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference-CUDA-kernel measurements (ref_gpu key)")
    ap.add_argument("--trainer", default="pipelined", choices=["pipelined", "sync"],
                    help="pipelined = gsplat.dp.PipelinedTrainer (no host sync, CUDA graphs, exchange behind the next image's "
                         "geometry); sync = gsplat.dp.ImageShardedTrainer (round-1 path: one host sync per step, eager)")
    ap.add_argument("--operators", default="fused", choices=["fused", "dropin"],
                    help="pipelined trainer phases: fused = the raw-parameter kernels on the C ABI (b200_fused_geometry_forward / "
                         "_colors_forward / _preprocess_backward, no autograd glue); dropin = gsplat.project_gaussians / "
                         "spherical_harmonics / rasterize_gaussians under autograd")
    ap.add_argument("--no-graphs", action="store_true", help="pipelined trainer without CUDA-graph capture (debug / A-B)")
    ap.add_argument("--fused", action="store_true",
                    help="render through gsplat.fused.render_gaussians (caller-modified 'next' path) instead of the drop-in operators")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one left the caller (rank 0): the loss and every trained "
                         "parameter as DIR/<name>.npy (float32, at most 64 MB in all: a fixed, seeded sample of the "
                         "Gaussians beyond that; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.sh_chunks is None:
        args.sh_chunks = 1
    return args


# ------------------------------------------------------------------------------------------------ CPU arm

def cpu_step_factory(cfg, n_override=None):
    """One train 'step' on the host: the oracle port of projection + SH + binning + blend, forward and backward."""
    import numpy as np
    import torch

    _forget_flat_oracle()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import oracle as O
    from util_scene import scene_np

    O.build()
    d = scene_np(cfg, n=n_override)
    H, W, S = d["H"], d["W"], d["S"]
    rng = np.random.default_rng(0)
    target = rng.uniform(0, 1, (H, W, 3)).astype(np.float32)
    dirs = d["means"] - d["cam_pos"][None]

    cache = {}

    def step(rows=None, blend_only=False):
        t0 = time.perf_counter()
        if blend_only and cache:
            proj, colors, opac, b = cache["proj"], cache["colors"], cache["opac"], cache["b"]
            t1 = time.perf_counter()
            img, Ts, fi = O.rasterize_forward(H, W, 16, S, b["gaussian_ids_sorted"], b["tile_bins"], proj["xys"],
                                              proj["pix_vels"], d["rs"], d["exposure"], proj["conics"], colors, opac,
                                              d["background"], rows=rows)
            v_out = (np.sign(img - target) / img.size).astype(np.float32)
            O.rasterize_backward(H, W, 16, S, b["gaussian_ids_sorted"], b["tile_bins"], proj["xys"], proj["pix_vels"],
                                 d["rs"], d["exposure"], proj["conics"], colors, opac, d["background"], Ts, fi, v_out,
                                 np.zeros((H, W), np.float32), rows=rows)
            return 0.0, time.perf_counter() - t1
        proj = O.project_forward(d["means"], d["scales"], 1.0, d["quats"], d["lin_vel"], d["ang_vel"], d["rs"],
                                 d["exposure"], d["viewmat"], d["fx"], d["fy"], d["cx"], d["cy"], H, W, 16)
        sh = O.sh_forward("fast", 3, dirs, d["sh"])
        colors = np.maximum(sh + 0.5, 0).astype(np.float32)
        opac = (d["opacity"][:, 0] * proj["compensation"])[:, None].astype(np.float32)
        b = O.bin_and_sort(proj["xys"], proj["depths"], proj["radii"], proj["num_tiles_hit"], H, W, 16)
        cache.update(proj=proj, colors=colors, opac=opac, b=b)
        t1 = time.perf_counter()
        img, Ts, fi = O.rasterize_forward(H, W, 16, S, b["gaussian_ids_sorted"], b["tile_bins"], proj["xys"],
                                          proj["pix_vels"], d["rs"], d["exposure"], proj["conics"], colors, opac,
                                          d["background"], rows=rows)
        v_out = (np.sign(img - target) / img.size).astype(np.float32)  # d(L1 mean)/d(img)
        g = O.rasterize_backward(H, W, 16, S, b["gaussian_ids_sorted"], b["tile_bins"], proj["xys"], proj["pix_vels"],
                                 d["rs"], d["exposure"], proj["conics"], colors, opac, d["background"], Ts, fi, v_out,
                                 np.zeros((H, W), np.float32), rows=rows)
        t2 = time.perf_counter()
        O.sh_backward("fast", 3, 3, dirs, g["v_colors"] * (colors > 0))
        O.project_backward(d["means"], d["scales"], 1.0, d["quats"], d["lin_vel"], d["ang_vel"], d["rs"], d["exposure"],
                           d["viewmat"], d["fx"], d["fy"], proj["cov3d"], proj["radii"], proj["conics"],
                           proj["compensation"], g["v_xy"], np.zeros(d["N"], np.float32), g["v_pix_vels"], g["v_conic"],
                           (g["v_opacity"][:, 0] * d["opacity"][:, 0]).astype(np.float32))
        t3 = time.perf_counter()
        return (t1 - t0) + (t3 - t2), (t2 - t1)  # (per-Gaussian stages, blend fwd+bwd)

    return step, d


def run_cpu_arm(args, one_shot=False):
    """Times the oracle port on the host cores.  The sample is a function of the ARGUMENTS only (never of how fast the
    box happens to be), so two runs of the same command time the same work: with at most 40 steps (warm-up included)
    every step is the full image; beyond that the blend forward + backward runs on a centred band of image rows whose
    height shrinks with the step count (time scaled by H / band) and the per-Gaussian stages (projection, SH, binning)
    run in full every m-th step with their last measured time charged in between.  The sample is stated in the JSON.
    Threads: B200_CPU_THREADS, else every core this process may use (affinity mask / cgroup quota)."""
    cores = int(os.environ.get("B200_CPU_THREADS", usable_cores()))
    # torchrun exports OMP_NUM_THREADS=1 to every rank, which would silently make this a 1-thread baseline; the oracle's
    # OpenMP runtime reads the variable when liboracle.so is loaded (below), so override it here
    os.environ["OMP_NUM_THREADS"] = str(cores)
    step, d = cpu_step_factory(args.config, args.n)
    _forget_flat_oracle()
    from oracle import oracle as _O
    cores = _O.set_threads(cores)  # the count the OpenMP runtime actually uses
    H = d["H"]
    n_steps = 1 if one_shot else args.steps + args.warmup
    full_steps = 40
    rows, pre_every = None, 1
    sample = f"1 image = full {d['W']}x{H} config-{args.config} fwd+bwd (projection, SH, binning, blend) per step"
    if n_steps > full_steps:
        band = int(min(H, max(16, (H * full_steps // n_steps) // 16 * 16)))
        if band < H:
            rows = (H // 2 - band // 2, H // 2 - band // 2 + band)
        pre_every = int(-(-n_steps // full_steps))
        sample = (f"per step: blend fwd+bwd on image rows {rows[0] if rows else 0}..{rows[1] if rows else H} of {H} (time x "
                  f"{H / (rows[1] - rows[0]) if rows else 1:.2f}); per-Gaussian stages (projection, SH, binning) "
                  f"in full every {pre_every}th step, last measured time charged in between")
    pre = 0.0
    scale = 1.0 if rows is None else H / (rows[1] - rows[0])
    state = {"pre": pre, "k": 0}

    def timed_step():
        k = state["k"]
        state["k"] += 1
        if k % pre_every == 0:
            p_, b_ = step(rows)
            state["pre"] = p_
        else:
            _, b_ = step(rows, blend_only=True)
        return state["pre"] + b_ * scale

    if one_shot:
        sec = timed_step()
        return dict(value=1.0 / sec, unit="images/s", cores=cores, kind="port", sample=sample + " (1 repetition)")
    for _ in range(args.warmup):
        timed_step()
    tot = 0.0
    t_wall = time.perf_counter()
    for _ in range(args.steps):
        tot += timed_step()
    wall = time.perf_counter() - t_wall
    ms = 1000.0 * tot / args.steps
    val = 1000.0 / ms
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "gpu_launches": 0,
        "config": bench_config(args.config, d["N"], d["W"], H, d["S"]),
        "details": {"arm": "CPU oracle port of the reference kernels (oracle/splat_oracle.c), OpenMP over image rows", "wall_s": wall},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(out)


# ------------------------------------------------------------------------------------------------ GPU arms

DUMP_LIMIT = 64_000_000 - (64 << 10)  # 64 MB, less room for the .npy headers


def dump_outputs(out_dir, model, loss):
    """What a caller of the timed path holds after its last step, as float32 `out_dir/<name>.npy`: `loss` and every
    trained parameter of the FlatGaussians model (its per-Gaussian views by name, `cam_vel` = the optimised camera
    velocities).  The inputs are seeded, so two builds run with the same arguments can be compared file by file.  When
    the whole set would pass 64 MB (from about 270k Gaussians on), every per-Gaussian parameter is written for the same
    rows only: numpy's default_rng(0).choice(N, rows, replace=False), sorted, with as many rows as fit -- the same rows in
    every run of the same workload.  `loss` and `cam_vel` are always whole."""
    import numpy as np
    import torch

    whole = {"loss": loss.reshape(())}
    if model.cam_vel is not None:
        whole["cam_vel"] = model.cam_vel
    per_gaussian = {k: v.detach().float() for k, v in model.params.items()}
    n = model.N
    whole_bytes = sum(4 * v.numel() for v in whole.values())
    row_bytes = sum(4 * v[0].numel() for v in per_gaussian.values())
    rows = (DUMP_LIMIT - whole_bytes) // row_bytes
    if rows < n:
        idx = np.sort(np.random.default_rng(0).choice(n, size=rows, replace=False))
        idx = torch.from_numpy(idx).to(model.flat.device)
        per_gaussian = {k: v[idx] for k, v in per_gaussian.items()}
    arrays = dict(per_gaussian, **{k: v.detach().float() for k, v in whole.items()})
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def make_cameras(scene, device, optimize_vel):
    import torch

    cams = []
    for c in scene["cameras"]:
        cams.append(dict(viewmat=c["viewmat"].to(device), fx=c["fx"], fy=c["fy"], cx=c["cx"], cy=c["cy"],
                         cam_pos=c["cam_pos"].to(device), lin_vel=c["lin_vel"].to(device), ang_vel=c["ang_vel"].to(device),
                         vel0=torch.cat([c["lin_vel"], c["ang_vel"]]).to(device)))
    return cams


def _forget_flat_oracle():
    """Take oracle/ off sys.path (every occurrence) and drop a top-level module `oracle` that is oracle/oracle.py rather
    than the package: with the directory on the path `from oracle import oracle` finds the FILE first."""
    odir = os.path.realpath(os.path.join(ROOT, "oracle"))
    sys.path[:] = [p for p in sys.path if os.path.realpath(p or ".") != odir]
    m = sys.modules.get("oracle")
    if m is not None and not hasattr(m, "__path__"):
        del sys.modules["oracle"]


def import_oracle_helpers():
    """oracle/ holds both the package `oracle` and flat helper modules that import each other by bare name (and put their
    own directory on sys.path to do so): the directory is on the path only while they are imported.  Round 2 shipped this
    with a single `sys.path.remove`, the helpers' own insert survived it and the CPU baseline of the same process then
    failed to import the package (r2u / r2y bench lines: cpu_baseline None)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import build_ref
        import ref_bench
        import ref_ops  # noqa: F401
        import torch_oracle  # noqa: F401
    finally:
        _forget_flat_oracle()
    return build_ref, ref_bench


def measure_ref_gpu(args, scene_dev, cams, targets, n_img, value, loss_fn, dev):
    """`ref_gpu`: train-step images/s of the UNMODIFIED reference gsplat CUDA kernels (oracle/_ref) on this arm's
    workload, three ways, plus this repo on the zero-motion variant so the ratio without the reference's phantom-tile-0
    tail is visible.  Reported beside the arm's value; never part of a timed region of the arm."""
    import torch

    try:
        build_ref, ref_bench = import_oracle_helpers()

        if not os.path.exists(build_ref.so_path()):
            return {"unavailable": "oracle/_ref/gsplat_ref_csrc.so not built (needs /root/reference at build time)"}
        out = {"kernels": "unmodified reference CUDA extension (forward.cu / backward.cu / bindings.cu, -O3 --use_fast_math, sm_100), "
                          "driven with the reference's own op sequence (oracle/ref_ops.py), torch L1 + torch fused Adam"}
        # the reference extension launches on the legacy default stream (bindings.cu: `<<<grid, block>>>`); torch's side
        # streams are non-blocking, i.e. NOT ordered against it -- so the reference runs with torch on the default stream too
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.default_stream(dev)):
            out["cuda_projection"] = ref_bench.measure(args.config, args.n, n_img, 30, 5, "cuda", breakdown=True)
            out["torch_projection_velocity_grad"] = ref_bench.measure(args.config, args.n, n_img, 20, 3, "torch")
            out["static_zero_velocity"] = ref_bench.measure(args.config, args.n, n_img, 30, 5, "static")
        torch.cuda.synchronize()
        # this repo on the zero-velocity variant (same trainer as the arm)
        from gsplat.dp import FlatGaussians, PipelinedTrainer

        rows0 = []
        for c in cams:
            z = torch.zeros(3, device=dev)
            rows0.append(torch.cat([c["viewmat"].reshape(-1), z, z, c["cam_pos"]]).contiguous())
        m0 = FlatGaussians(scene_dev, dev, n_cameras=n_img, optimize_velocities=True, sh_layout=_layout(args.operators))
        t0 = PipelinedTrainer(m0, scene_dev, lr=1e-4, loss_fn=loss_fn, use_graphs=not args.no_graphs, operators=args.operators)
        t0.prepare(rows0[0], 0)
        n_w, n_t = n_img + 4, 60
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(n_w + n_t):
            if k == n_w:
                t0.finish()
                e0.record()
            t0.train_step(targets[k % n_img], rows0[(k + 1) % n_img], (k + 1) % n_img)
        t0.finish()
        e1.record()
        torch.cuda.synchronize()
        ms0 = e0.elapsed_time(e1) / n_t
        out["this_repo_static_zero_velocity"] = {"value": 1000.0 / ms0, "unit": "images/s", "ms_per_step": ms0, "steps": n_t}
        out["ratio_vs_cuda_projection"] = round(value / out["cuda_projection"]["value"], 2)
        out["ratio_vs_torch_projection"] = round(value / out["torch_projection_velocity_grad"]["value"], 2)
        out["ratio_static"] = round(out["this_repo_static_zero_velocity"]["value"] / out["static_zero_velocity"]["value"], 2)
        out["note"] = ("ratios = this arm's `value` (velocities carry gradients) / the reference variant; `torch_projection` is what "
                       "train.py runs by default (velocity optimisation on: project_gaussians.py:81-112), timed through "
                       "oracle/torch_oracle.py's restatement of _torch_impl.project_gaussians_forward")
        return out
    except Exception as e:  # a reported comparator, never a reason to lose the arm's line
        return {"unavailable": repr(e)[:300]}


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from gsplat import _lib, synthetic
    from gsplat.dp import FlatGaussians, ImageShardedTrainer

    lib = _lib.load()
    n_img = args.images
    # image mode: the same scene (parameters) on every rank; rank r trains on its own cameras / images.
    # scene mode: rank r holds scene r mod S; the ranks of one scene form its (image-sharded) group, groups never talk.
    group, gworld, grank, scene_id = None, world, rank, 0
    if args.mode == "scene":
        n_sc = max(1, min(args.scenes, world))
        scene_id = rank % n_sc
        members = [r for r in range(world) if r % n_sc == scene_id]
        gworld, grank = len(members), members.index(rank)
        if world > 1:
            groups = [dist.new_group([r for r in range(world) if r % n_sc == s_]) for s_ in range(n_sc)]  # (collective: every rank creates every group)
            group = groups[scene_id]
    scene = synthetic.make_scene(args.config, device="cpu", n_override=args.n, n_cameras=n_img * gworld, seed_offset=100 * scene_id)
    my = [scene["cameras"][i * gworld + grank] for i in range(n_img)]
    targets_u8 = [(c["target"] * 255).to(torch.uint8).contiguous().pin_memory() for c in my]
    scene_dev = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in scene.items() if k != "cameras"}
    scene_dev["cameras"] = my
    cams = make_cameras(scene_dev, dev, not args.no_vel_grad)
    targets = [t.to(dev).float() / 255 for t in targets_u8]
    vel_grad = not args.no_vel_grad
    loss_fn = None
    if args.loss == "photometric":
        from gsplat.losses import photometric_loss as loss_fn
    pipelined = args.trainer == "pipelined" and not args.fused
    H, W, S, N = scene["H"], scene["W"], scene["blur_samples"], scene["N"]
    cam_rows = [torch.cat([c["viewmat"].reshape(-1), c["lin_vel"], c["ang_vel"], c["cam_pos"]]).contiguous() for c in cams]  # device
    if pipelined:
        from gsplat.dp import PipelinedTrainer

        scene_dev.update(fx=cams[0]["fx"], fy=cams[0]["fy"], cx=cams[0]["cx"], cy=cams[0]["cy"])
        model = FlatGaussians(scene_dev, dev, n_cameras=n_img, optimize_velocities=vel_grad, sh_layout=_layout(args.operators))
        trainer = PipelinedTrainer(model, scene_dev, lr=1e-4, loss_fn=loss_fn, use_graphs=not args.no_graphs, group=group,
                                   operators=args.operators, sh_chunks=args.sh_chunks)
        torch.cuda.set_stream(trainer.main)  # everything below (events, prefetcher, timing) runs on the trainer's stream
    else:
        model = FlatGaussians(scene_dev, dev, n_cameras=n_img, optimize_velocities=vel_grad)
        trainer = ImageShardedTrainer(model, scene_dev, lr=1e-4, fused=args.fused, sh_chunks=args.sh_chunks, optimizer=args.optimizer,
                                      loss_fn=loss_fn, group=group)

    class Stepper:
        """step(k): one train step on image k % n_img (consecutive k: the pipelined trainer stages image k+1 inside step k)."""

        def __init__(self, images, cam_source):
            self.images, self.cam_source, self.staged = images, cam_source, None

        def step(self, k, image=None):
            i = k % n_img
            tgt = self.images[i] if image is None else image
            if not pipelined:
                return trainer.train_step(cams[i] if self.cam_source is None else self.cam_source(i), tgt, i)
            if self.staged != k:
                trainer.prepare(cam_rows[i] if self.cam_source is None else self.cam_source(i), i)
            nxt = (k + 1) % n_img
            self.staged = k + 1
            return trainer.train_step(tgt, cam_rows[nxt] if self.cam_source is None else self.cam_source(nxt), nxt)

    stepper = Stepper(targets, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- cost-aware batching (N > 1): a synchronous step lasts as long as its slowest rank, and images differ in cost (tile
    # list entries 0.6-0.84 M at config 2).  One pass measures every image's entries (phase A's status word), the ranks
    # share them, and gsplat.dp.balanced_assignment regroups the SAME images so that each step holds images of similar cost.
    balance = None
    if world > 1 and pipelined and args.mode == "image" and not args.no_balance:
        from gsplat.dp import balanced_assignment

        local = [0] * n_img
        for i in range(n_img + 1):
            stepper.step(i)
            trainer.finish()
            torch.cuda.synchronize()
            local[(i + 1) % n_img] = int(trainer.status[1])  # (step i also prepared image i + 1: its entries are in the status word)
        gathered = [torch.zeros(n_img, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor(local, dtype=torch.int64, device=dev))
        costs = [0] * (n_img * world)
        for r_ in range(world):
            for i in range(n_img):
                costs[i * world + r_] = int(gathered[r_][i])
        steps_ = balanced_assignment(costs, world)
        mine = [steps_[j][rank] for j in range(n_img)]
        spread = lambda groups: sum(max(costs[g] for g in grp) / (sum(costs[g] for g in grp) / world) for grp in groups) / len(groups)
        balance = {"max_over_mean_cost_before": round(spread([[i * world + r_ for r_ in range(world)] for i in range(n_img)]), 4),
                   "max_over_mean_cost_after": round(spread(steps_), 4), "cost": "tile-list entries after culling (phase A status word)"}
        my[:] = [scene["cameras"][g] for g in mine]
        new_cams = make_cameras(dict(scene_dev, cameras=my), dev, not args.no_vel_grad)
        cams[:] = new_cams
        targets_u8[:] = [(c["target"] * 255).to(torch.uint8).contiguous().pin_memory() for c in my]
        targets[:] = [t.to(dev).float() / 255 for t in targets_u8]
        cam_rows[:] = [torch.cat([c["viewmat"].reshape(-1), c["lin_vel"], c["ang_vel"], c["cam_pos"]]).contiguous() for c in cams]
        stepper.staged = None
        # every rank now knows every image's entry count: size the lists once, identically everywhere, so that no rank
        # grows them (= captures new graphs, ~10 ms, which its peers then wait for in the next allreduce) later on
        trainer.reserve(max(costs))

    # ---- kernel-resident metric: inputs already in HBM, CUDA-event timing, max over ranks
    # warm-up: at least one pass over every training image, so no timed step meets a new camera (first-use allocations,
    # list capacities) -- args.warmup is a lower bound
    n_warm = max(args.warmup, n_img + 4)  # (+ the two eager rounds before the pipelined trainer captures its graphs)
    for w in range(n_warm):
        stepper.step(w)
    # ... and until the trainer is steady: the list capacity follows a high-water mark that the host learns one step late,
    # a growth means two eager steps and a graph capture (~10 ms) -- if the image that triggers it comes late in the pass,
    # the capture would land in the timed region (r3n8: one 11.7 ms step among twenty of 1.4 ms at N = 8, where eight ranks
    # make a late trigger eight times as likely and every rank waits for the one that captures).  Whole extra passes, the
    # ranks agree on them (a rank that went on alone would deadlock the exchange), at most three.
    if pipelined:
        sig = (tuple(targets[0].shape), targets[0].dtype)
        for attempt in range(3):
            cap0 = trainer.capacity
            trainer.finish()
            trainer.sync_status()
            unsteady = not (trainer.capacity == cap0 and trainer.steady(sig))
            if attempt == 0 and os.environ.get("B200_BENCH_FORCE_EXTRA_PASS") == "1":
                unsteady = True  # (exercises the extra-pass branch on a box where the trainer is already steady)
            more = torch.tensor([1 if unsteady else 0], device=dev)
            if world > 1:
                dist.all_reduce(more, op=dist.ReduceOp.MAX)
            if int(more.item()) == 0:
                break
            for w in range(n_img):
                stepper.step(n_warm + w)
            n_warm += n_img
    # the clock sampler forks nvidia-smi: start it BEFORE the barrier that opens the timed region (round 1 started it
    # on rank 0 after the barrier, so the other ranks waited for rank 0's fork/exec inside their first allreduce and
    # that latency was charged to the max-over-ranks time)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)  # first samples in hand before the region opens
    barrier()
    # one event per step boundary: total = last - first (what `value` uses), per-step spread shows one-off stalls
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    l0 = lib.b200_launch_count() + (trainer.graph_kernel_launches if pipelined else 0)
    evs[0].record()
    for k in range(args.steps):
        loss = stepper.step(n_warm + k)
        if pipelined and k == args.steps - 1:
            trainer.finish()  # the last step's SH update (side stream) belongs to the timed region
        evs[k + 1].record()
    barrier()
    if args.dump_outputs and rank == 0:  # now: the measurements below train the same model further
        dump_outputs(args.dump_outputs, model, loss)
    launches = (lib.b200_launch_count() + (trainer.graph_kernel_launches if pipelined else 0) - l0) / args.steps
    ms = evs[0].elapsed_time(evs[-1]) / args.steps
    per_step = sorted(evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps))
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms, per_step[len(per_step) // 2], per_step[min(len(per_step) - 1, int(0.99 * len(per_step)))], per_step[-1]],
                     device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, p50, p99, pmax = (float(x) for x in t.tolist())
    step_ms = {"p50": round(p50, 4), "p99": round(p99, 4), "max": round(pmax, 4),
               "note": "per-step device time between consecutive events on the compute stream, max over ranks of each statistic"}
    value = world * 1000.0 / ms

    # ---- the same trainer on the OTHER operator set (fused raw-parameter kernels <-> drop-in operators under autograd),
    # reported beside the headline (one GPU only: it is an A/B of the per-GPU step, not of the exchange)
    other_ops = None
    if pipelined and world == 1 and not args.no_fused_path:
        from gsplat.dp import PipelinedTrainer as _PT

        other = "dropin" if args.operators == "fused" else "fused"
        model_o = FlatGaussians(scene_dev, dev, n_cameras=n_img, optimize_velocities=vel_grad, sh_layout=_layout(other))
        trainer_o = _PT(model_o, scene_dev, lr=1e-4, loss_fn=loss_fn, use_graphs=not args.no_graphs, operators=other)
        osteps = max(40, args.steps // 4)
        trainer_o.prepare(cam_rows[0], 0)
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_w = n_img + 4
        for k in range(n_w + osteps):
            if k == n_w:
                trainer_o.finish()
                o0.record()
            trainer_o.train_step(targets[k % n_img], cam_rows[(k + 1) % n_img], (k + 1) % n_img)
        trainer_o.finish()
        o1.record()
        torch.cuda.synchronize()
        ms_o = o0.elapsed_time(o1) / osteps
        other_ops = {"operators": other, "value": 1000.0 / ms_o, "unit": "images/s", "ms_per_step": ms_o, "steps": osteps,
                     "api": _api(other)}
        del trainer_o, model_o

    if args.timeline:  # every rank steps (collectives), rank 0 records
        from torch.profiler import ProfilerActivity, profile

        k0 = stepper.staged if (pipelined and stepper.staged is not None) else 0
        if rank == 0:
            with profile(activities=[ProfilerActivity.CUDA]) as prof_t:
                for k in range(6):
                    stepper.step(k0 + k)
                torch.cuda.synchronize()
            from torch.autograd import DeviceType
            evs = sorted((e for e in prof_t.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start)
            t0_ = evs[0].time_range.start if evs else 0
            with open(args.timeline, "w") as f:
                f.write("start_us\tdur_us\tname\n")
                for e in evs:
                    f.write(f"{e.time_range.start - t0_:.1f}\t{e.time_range.end - e.time_range.start:.1f}\t{e.name[:90]}\n")
        else:
            for k in range(6):
                stepper.step(k0 + k)
            torch.cuda.synchronize()

    gpu_busy = None
    if args.profile and rank == 0:
        from torch.profiler import ProfilerActivity, profile

        nprof = 20
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            k0 = stepper.staged if (pipelined and stepper.staged is not None) else 0
            for k in range(nprof):
                stepper.step(k0 + k)
            torch.cuda.synchronize()
        dev_us = sum(e.device_time_total for e in prof.key_averages())
        gpu_busy = {"kernel_ms_per_step": dev_us / nprof / 1000.0, "note": "sum of device time of every kernel in a step (CUPTI); "
                    "ms_per_step minus this is GPU idle time (launch latency, the host sync, CPU-side Python)"}
        try:  # where the GPU waits: idle gaps between consecutive device activities, keyed by the activity that follows
            from torch.autograd import DeviceType

            evs = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA),
                         key=lambda e: e.time_range.start)
            gaps, end = {}, None
            for e in evs:
                if end is not None and e.time_range.start > end:
                    k = e.name[:60]
                    g = gaps.setdefault(k, [0.0, 0])
                    g[0] += e.time_range.start - end
                    g[1] += 1
                end = e.time_range.end if end is None else max(end, e.time_range.end)
            top = sorted(gaps.items(), key=lambda kv: -kv[1][0])[:12]
            gpu_busy["idle_before_us_per_step"] = {k: [round(v[0] / nprof, 1), round(v[1] / nprof, 1)] for k, v in top}
            gpu_busy["idle_total_us_per_step"] = round(sum(v[0] for v in gaps.values()) / nprof, 1)
        except Exception as e:  # diagnostic only
            gpu_busy["idle_error"] = repr(e)[:200]

    # ---- end to end: host buffers in, loss out, every step (pinned uint8 image + camera H2D, loss D2H)
    cam_host = [torch.cat([c["viewmat"].reshape(-1), c["lin_vel"], c["ang_vel"], c["cam_pos"]]).pin_memory() for c in my]
    e2e_steps = args.steps  # (wall-clock timed: at a few steps, filling the prefetch pipeline shows in the figure)

    # double-buffered prefetch on a copy stream (gsplat.data.ImagePrefetcher: what a datamanager does -- pinned uint8
    # image + camera floats), the loss of step k-1 is read back while step k is already queued; every step's inputs cross
    # PCIe inside the timed region and every step's loss is read.
    from gsplat.data import ImagePrefetcher

    prefetcher = ImagePrefetcher(targets_u8, cam_host, dev)
    main_stream = torch.cuda.current_stream()

    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event() for _ in range(2)]

    # the pipelined trainer takes the uint8 image as it arrives (the conversion is the first node of its B graph) and the
    # NEXT image's camera row straight from pinned host memory (84 bytes H2D inside its step)
    e2e_stepper = Stepper(None, (lambda i: cam_host[i]) if pipelined else None)

    def e2e_loop(n_steps):
        losses = []
        prefetcher.start(0)
        e2e_stepper.staged = None
        for k in range(n_steps):
            b, i = k % 2, k % n_img
            img_u8, ch = prefetcher.get(next_index=(k + 1) % n_img)
            if pipelined:
                loss = e2e_stepper.step(k, image=img_u8)
            else:
                tgt = img_u8.float() / 255
                cam = dict(cams[i], viewmat=ch[:12].view(3, 4), lin_vel=ch[12:15], ang_vel=ch[15:18], vel0=ch[12:18], cam_pos=ch[18:21])
                loss = trainer.train_step(cam, tgt, i)
            prefetcher.done()
            loss_host[b].copy_(loss.detach().reshape(1), non_blocking=True)  # loss D2H (4 bytes) every step
            loss_done[b].record(main_stream)
            if k > 0:  # read the previous step's loss while this step is queued / running
                loss_done[1 - b].synchronize()
                losses.append(float(loss_host[1 - b][0]))
        loss_done[(n_steps - 1) % 2].synchronize()
        losses.append(float(loss_host[(n_steps - 1) % 2][0]))
        assert all(x == x for x in losses)  # no NaNs, and every step's loss reached the host
        return losses

    e2e_loop(max(4, n_img + 4))  # (first use of the uint8 targets: two eager rounds, then graph capture)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(e2e_steps)
    barrier()
    e2e_ms = 1000.0 * (time.perf_counter() - t0) / e2e_steps
    t = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    h2d = prefetcher.bytes_per_step
    e2e = {"value": world * 1000.0 / e2e_ms, "unit": "images/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 4 + 8, "steps": e2e_steps,
           "path": (_api(args.operators) if pipelined else _api("dropin")) + " via gsplat.dp." + (
               "PipelinedTrainer" if pipelined else "ImageShardedTrainer") + "; uint8 image + camera row from pinned host memory "
                   "every step (gsplat.data.ImagePrefetcher), loss read back every step"}
    trainer_status = None
    if pipelined:
        trainer.finish()
        trainer_status = trainer.sync_status()
        trainer_status["graphs"] = sum(1 for e in trainer._graphs.values() if e["gA"] is not None and e["gB"] is not None)

    # ---- per-kernel timing + roofline of the dominant kernel (rank 0), CUDA events on the launch stream
    kernels, roofline = {}, None
    if rank == 0:
        import gsplat.cuda as _C

        with torch.no_grad():
            p = model.params
            q = p["quats"] / p["quats"].norm(dim=-1, keepdim=True)
            cam = cams[0]
            lin, ang = cam["lin_vel"], cam["ang_vel"]
            args_proj = (N, p["means"].detach().contiguous(), torch.exp(p["log_scales"]).contiguous(), 1.0, q.contiguous(), None,
                         None, scene["rolling_shutter_time"], scene["exposure_time"], cam["viewmat"], cam["fx"], cam["fy"],
                         cam["cx"], cam["cy"], H, W, 16, 0.01)
            cov3d, xys, depths, pix_vels, radii, conics, comp, nth = _C.project_gaussians_forward(*args_proj, _vel_tensors=(lin, ang))
            coeffs = model.sh_coeffs().detach().contiguous()
            dirs = (p["means"] - cam["cam_pos"]).contiguous()
            colors = torch.clamp(_C.compute_sh_forward("fast", N, 3, 3, dirs, coeffs) + 0.5, min=0).contiguous()
            opac = (torch.sigmoid(p["opacity_logit"]) * comp[:, None]).contiguous()
            I, cum = _C.cumulative_intersects(nth)
            tb = ((W + 15) // 16, (H + 15) // 16, 1)
            isect, gids = _C.map_gaussian_to_intersects(N, I, xys, depths, radii, cum, tb, 16)
            isect_s, gids_s = _C.sort_intersects(tb[0] * tb[1], isect, gids)
            bins = _C.get_tile_bin_edges(I, isect_s, tb)
            bg = scene_dev["background"]
            rs, ex = scene["rolling_shutter_time"], scene["exposure_time"]
            # what rasterize_gaussians actually runs: pack once, culled binning, blend on the culled lists
            packed = _C.pack_records(xys, pix_vels, conics, colors, opac)
            _, ids_c, bins_c = _C.bin_cull(packed, depths, radii, nth, H, W, 16, S, rs, ex)
            M = int(ids_c.numel())
            img, Ts, fi = _C.blend_forward_packed(H, W, 16, S, ids_c, bins_c, packed, rs, ex, bg)
            v_out = torch.sign(img - targets[0]) / img.numel()
            v_alpha = torch.zeros(H, W, device=dev)
            V = int((nth > 0).sum().item())
            gr = _C.blend_backward_packed(N, H, W, 16, S, ids_c, bins_c, packed, rs, ex, bg, Ts, fi, v_out, v_alpha)
            img_f, Ts_f, fi_f = _C.rasterize_forward(tb, (16, 16, 1), (W, H, 1), S, gids_s, bins, xys, pix_vels, rs, ex, conics, colors, opac, bg)
            v_comp = (gr[5][:, 0] * torch.sigmoid(p["opacity_logit"])[:, 0]).contiguous()

            def timeit(fn, reps=20):
                for _ in range(3):
                    fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a.record()
                for _ in range(reps):
                    fn()
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b) / reps

            P = H * W
            stages = {
                "project_fwd": (lambda: _C.project_gaussians_forward(*args_proj, _vel_tensors=(lin, ang)), 108 * N),
                "sh_fwd": (lambda: _C.compute_sh_forward("fast", N, 3, 3, dirs, coeffs), 216 * N),
                "map_intersects": (lambda: _C.map_gaussian_to_intersects(N, I, xys, depths, radii, cum, tb, 16), 20 * N + 12 * I),
                "sort": (lambda: _C.sort_intersects(tb[0] * tb[1], isect, gids), 24 * I),
                "bin_edges": (lambda: _C.get_tile_bin_edges(I, isect_s, tb), 8 * I + 8 * tb[0] * tb[1]),
                "bin_tiles_fused": (lambda: _C.bin_tiles(I, xys, depths, radii, nth, tb, 16), 20 * N + 12 * I + 24 * I + 8 * I),
                "pack_records": (lambda: _C.pack_records(xys, pix_vels, conics, colors, opac), 108 * N),
                "bin_cull": (lambda: _C.bin_cull(packed, depths, radii, nth, H, W, 16, S, rs, ex), 20 * N + 12 * I + 24 * I + 8 * I),
                "blend_fwd": (lambda: _C.blend_forward_packed(H, W, 16, S, ids_c, bins_c, packed, rs, ex, bg), 48 * I + P * (12 + 8 * S)),
                "blend_bwd": (lambda: _C.blend_backward_packed(N, H, W, 16, S, ids_c, bins_c, packed, rs, ex, bg, Ts, fi, v_out,
                                                               v_alpha), 48 * I + P * (16 + 8 * S) + 52 * V),
                "blend_fwd_full_lists": (lambda: _C.rasterize_forward(tb, (16, 16, 1), (W, H, 1), S, gids_s, bins, xys, pix_vels, rs,
                                                                      ex, conics, colors, opac, bg), 48 * I + P * (12 + 8 * S)),
                "blend_bwd_full_lists": (lambda: _C.rasterize_backward(H, W, 16, S, gids_s, bins, xys, pix_vels, rs, ex, conics,
                                                                       colors, opac, bg, Ts_f, fi_f, v_out, v_alpha),
                                         48 * I + P * (16 + 8 * S) + 52 * V),
                "sh_bwd": (lambda: _C.compute_sh_backward("fast", N, 3, 3, dirs, gr[4]), 216 * N),
                "project_bwd": (lambda: _C.project_gaussians_backward(
                    N, args_proj[1], args_proj[2], 1.0, args_proj[4], None, None, rs, ex, cam["viewmat"], cam["fx"], cam["fy"],
                    cam["cx"], cam["cy"], H, W, cov3d, radii, conics, comp, gr[0], torch.zeros_like(depths), gr[2], gr[3], v_comp,
                    _vel_tensors=(lin, ang), _exact=vel_grad, _want_vel=vel_grad), 160 * N),
            }
            peaks = {}
            pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
            if os.path.exists(pk):
                peaks = json.load(open(pk))
            peak = float(peaks.get("hbm_gbs", 6650.0))
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
            for name, (fn, nbytes) in stages.items():
                t_ms = timeit(fn)
                kernels[name] = {"ms": round(t_ms, 4), "alg_bytes": int(nbytes), "gbs": round(nbytes / t_ms / 1e6, 1)}
            for k in ("map_intersects", "sort", "bin_edges", "bin_tiles_fused", "blend_fwd_full_lists", "blend_bwd_full_lists"):
                kernels[k]["note"] = "not on the train step: reference-faithful key path / un-culled lists, timed for comparison"
            kernels["bin_cull"]["note"] = "includes its host sync; algorithmic bytes are those of the reference's binning"
            on_path = [k for k in kernels if "note" not in kernels[k] or k == "bin_cull"]
            dom = max(on_path, key=lambda k: kernels[k]["ms"])
            traffic, traffic_src, issue = None, None, None
            tp = os.path.join(ROOT, "profiles", "traffic.json")  # per-launch figures from the committed ncu --set full captures
            if os.path.exists(tp) and args.n is None:
                tj = json.load(open(tp)).get(args.config, {})
                if dom in tj:
                    traffic, traffic_src = tj[dom]["dram_bytes"], tj[dom]["source"]
                    if tj[dom].get("warp_instructions") and clocks and clocks.get("sm_mhz"):
                        # the roofline that actually binds the blend (SURVEY 8d): FP32 lanes x clock.  Instruction count
                        # per launch from the ncu capture of this workload, duration measured live above.
                        lane_instr = tj[dom]["warp_instructions"] * tj[dom]["active_lanes_per_instruction"]
                        sms = torch.cuda.get_device_properties(dev).multi_processor_count
                        peak_li = sms * 128 * clocks["sm_mhz"] * 1e6
                        ach = lane_instr / (kernels[dom]["ms"] * 1e-3)
                        issue = {"bound": "fp32-lane issue", "lane_instructions_per_launch": int(lane_instr), "achieved": ach,
                                 "peak": peak_li, "unit": "lane-instr/s", "frac": round(ach / peak_li, 4),
                                 "peak_source": "%d SMs x 128 FP32 lanes x %.0f MHz (median SM clock sampled during the timed region)" % (
                                     sms, clocks["sm_mhz"])}
                        if tj[dom].get("pixel_sample_evaluations"):
                            # what the issued instructions buy: (pixel, sample, Gaussian) evaluations executed per launch and
                            # the share of them that passes the reference's sigma / alpha tests (the -DB200_BLEND_COUNTERS build)
                            ev, ok_ = tj[dom]["pixel_sample_evaluations"], tj[dom]["evaluations_passing_the_alpha_test"]
                            issue.update(evaluations_per_launch=ev, useful_evaluations_per_launch=ok_,
                                         useful_fraction=round(ok_ / ev, 4),
                                         useful_evaluations_per_s=ok_ / (kernels[dom]["ms"] * 1e-3),
                                         note=tj[dom].get("packed_fp32x2_note"))
            roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
                        "frac": round(kernels[dom]["gbs"] / peak, 5), "traffic": traffic, "traffic_source": traffic_src,
                        "peak_source": peak_src, "issue": issue,
                        "note": "blend kernels are FP32-issue / MUFU / SHFL / atomic bound, not HBM bound (SURVEY 0.5); see `issue`",
                        "intersections": I, "culled_list_entries": M, "visible": V}

    # ---- the comparator north_star names: the reference's own gsplat CUDA kernels (oracle/_ref = the unmodified extension
    # built by oracle/build_ref.py) on the same workload, same GPU, outside every timed region of this arm
    ref_gpu = None
    if rank == 0 and world == 1 and not args.no_ref_gpu and not args.fused:
        ref_gpu = measure_ref_gpu(args, scene_dev, cams, targets, n_img, value, loss_fn, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu_baseline = run_cpu_arm(args, one_shot=True)
        except Exception as e:  # the baseline is informative only
            cpu_baseline = {"value": None, "unit": "images/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e!r}"[:200]}
    out = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "warmup_run": n_warm,
        "config": bench_config(args.config, N, W, H, S),
        "details": {"step": "project+SH+bin/sort+blend fwd, L1 (gsplat.losses.l1_loss), full bwd, grad allreduce (N>1), Adam over the flat buffer; 1 image per GPU per step",
                    "optimizer": "gsplat.optim.FlatAdam (device step state)" if pipelined else ("gsplat.optim.FlatAdam (b200_adam_step)" if args.optimizer == "b200" else "torch.optim.Adam(fused=True)"),
                    "sh_chunks": args.sh_chunks, "loss": args.loss, "velocity_grad": vel_grad, "global_batch": world,
                    "api": ("gsplat.fused.render_gaussians (raw parameters, caller-modified)" if args.fused else
                            _api(args.operators if pipelined else "dropin")),
                    "operators": args.operators if pipelined else "dropin",
                    "parallelism": (f"image-sharded dp{world}" if args.mode == "image" else
                                    f"scene-sharded: {min(args.scenes, world)} independent scenes over {world} GPUs "
                                    f"(groups of {world // min(args.scenes, world)}-{-(-world // min(args.scenes, world))} ranks per scene, image-sharded inside a group)"),
                    "trainer": ("gsplat.dp.PipelinedTrainer: no host sync (capacity-mode tile lists, device-side veto), two CUDA "
                                "graphs per step, gradient exchange + SH update behind the next image's projection/binning"
                                if pipelined else "gsplat.dp.ImageShardedTrainer (one host sync per step, eager launches)"),
                    "trainer_status": trainer_status, "balance": balance},
        "step_ms": step_ms, "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "kernels": kernels,
        "cpu_baseline": cpu_baseline,
    }
    if ref_gpu:
        out["ref_gpu"] = ref_gpu
    if other_ops:
        out["other_operators"] = other_ops
    if gpu_busy:
        out["gpu_busy"] = gpu_busy
    _emit(out)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    # stdout carries exactly ONE line (the JSON): anything a library prints there (NCCL's version banner, ...) is
    # sent to stderr instead, including C-level writes.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _run(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if _RESULT:
        print(_RESULT[0], flush=True)


_RESULT = []


def _emit(obj):
    _RESULT.append(json.dumps(obj))


def _run(args):
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            run_cpu_arm(args)
        return
    if args.impl == "refgpu":
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_bench

        ref_bench.run(args)
        return
    run_gpu_arm(args)


if __name__ == "__main__":
    main()
