"""Benchmark of the RoHM denoising hot path on B200 (contract: see the task brief / DESIGN.md "Measurement").

  python bench.py --gpus 1 --steps 3 --warmup 3            # one process, cuda:0, BASELINE configs[1] (the headline)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W            # one rank per GPU, NCCL
  python bench.py --impl reference ...                     # the reference algorithm on the host CPU cores
  python bench.py --config {posenet,trajcontrol,pipeline,respaced100,lbs}   # the other BASELINE configs (one line each)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Workloads (BASELINE.json configs, per GPU; clips shard over ranks, weak scaling, one all-gather of final outputs per step):
  posenet      configs[1]  PoseNet denoiser, 32 clips x 145 frames (T = 144 motion frames, 145 tokens), 1000 DDPM steps
  trajcontrol  configs[2]  TrajNet + TrajControl, 64 clips x 144 frames, 1000 DDPM steps
  pipeline     configs[3]  full iterative inference: 3 rounds of TrajNet(100 steps, reference-faithful; --traj-steps) ->
                           device glue -> PoseNet(1000 steps, in-loop SMPL-X skating guidance on t <= 50), 32 clips per GPU,
                           then the post-loop SMPL-X reconstruction with vertices
  respaced100  configs[4]  100-step respaced ('ddim100' retained steps, ancestral) PoseNet + TrajNet, 128 clips per GPU
  lbs          row L2/N3   SMPL-X full LBS (joints + 10 475 vertices) of 32 x 143 frames from the motion representation
One "step" of the benchmark = one complete pass of the workload over the batch; metric = denoised clips / second, whole job.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

C_FEATS = 294
DIFFUSION_STEPS = 1000
LBS_BYTES_PER_FRAME = 126280  # SURVEY.md 8(d): 10 475 x 3 fp32 vertices + 55 joints out, 145 fp32 in
DUMP_WHOLE_MAX_ELEMS = 8 << 20  # --dump-outputs: arrays up to 32 MB are written whole, larger ones as a sample
DUMP_SAMPLE_ELEMS = 1 << 20
DUMP_LIMIT_BYTES = 64 << 20

CONFIGS = {
    "posenet": dict(clips=32, frames=144, label="BASELINE configs[1]: PoseNet denoiser, batch 32 x 145-frame clips (T=144 "
                    "motion frames, 145 tokens, 294 channels), 1000 DDPM steps, p_sample (no guidance)",
                    metric="denoised motion clips/sec (145-frame, 1000-step PoseNet p_sample_loop)"),
    "trajcontrol": dict(clips=64, frames=144, label="BASELINE configs[2]: TrajNet + TrajControl conditioning module, batch "
                        "64 x 144 frames x 13 channels, 1000 DDPM steps, p_sample_with_grad (no guidance in the reference)",
                        metric="denoised motion clips/sec (145-frame, 1000-step TrajNet+TrajControl p_sample_loop)"),
    "pipeline": dict(clips=32, frames=144, label="BASELINE configs[3]: full iterative inference, 3 rounds of TrajNet -> glue "
                     "-> PoseNet (1000 steps, skating guidance on t<=50) + post-loop SMPL-X LBS reconstruction, 32 clips/GPU",
                     metric="denoised motion clips/sec (145-frame clips through the 3-round TrajNet->PoseNet pipeline)"),
    "respaced100": dict(clips=128, frames=144, label="BASELINE configs[4]: 100-step respaced ('ddim100' retained steps, "
                        "ancestral) PoseNet + TrajNet sampling, 128 clips/GPU",
                        metric="denoised motion clips/sec (145-frame, 100-step respaced PoseNet+TrajNet)"),
    "lbs": dict(clips=32, frames=143, label="SURVEY row L2/N3: SMPL-X full LBS (22 joints + 10475 vertices) of 32 clips x "
                "143 frames from the motion representation (recover_from_repr_smpl, return_verts=True)",
                metric="SMPL-X LBS motion clips/sec (143 frames x 10475 vertices per clip)"),
}


def gemm_flops_per_forward(B, S, D=512, F=1024, C=294, Cout=272, L=8):
    """Algorithmic FLOPs of the tensor-core GEMMs of one PoseNet forward (SURVEY.md 8d)."""
    per_tok = L * (2 * D * 3 * D + 2 * D * D + 2 * D * F + 2 * F * D) + 2 * C * D + 2 * D * Cout
    return float(B) * S * per_tok


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "bf16_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1400.0, "bf16_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop, self.th = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self.stop.wait(0.5)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace('.', '').isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace('.', '').isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


# -------------------------------------------------------------------------------------------------------------
# model builders (synthetic weights of the exact architectures; there is no network for checkpoints)
# -------------------------------------------------------------------------------------------------------------
def build_posenet(device, ds=None):
    from rohm_b200 import synthetic
    from rohm_b200.posenet import PoseNet
    ds = ds if ds is not None else synthetic.make_dataset('pose')
    model = PoseNet(dataset=ds, body_feat_dim=C_FEATS, latent_dim=512, ff_size=1024, num_layers=8, num_heads=4,
                    device=device, traj_feat_dim=22)
    sd = synthetic.synth_state_dict(model, 1)
    model.load_state_dict(sd)
    if device is not None:
        model.to(device)
    return model.eval(), sd


def build_trajnet(device, control, ds=None, seed=2):
    from rohm_b200 import synthetic
    from rohm_b200.trajnet import TrajNet
    ds = ds if ds is not None else synthetic.make_dataset('traj')
    model = TrajNet(time_dim=32, mid_dim=512, cond_dim=13, traj_feat_dim=13, trajcontrol=control, device=device,
                    dataset=ds, repr_abs_only=True)
    sd = synthetic.synth_state_dict(model, seed)
    model.load_state_dict(sd)
    if device is not None:
        model.to(device)
    return model.eval(), sd


def make_diffusion(kind, steps, respacing, device):
    from rohm_b200 import diffusion
    a = argparse.Namespace(noise_schedule='cosine', sigma_small=True)
    cls = diffusion.SpacedDiffusionPoseNet if kind == 'pose' else diffusion.SpacedDiffusionTrajNet
    return diffusion.create_gaussian_diffusion(a, diffusion, cls, steps, respacing, device)


def host_threads():
    """Threads for the CPU legs: every core up to 32 (torch's intra-op pool stops scaling, then collapses, on this
    workload's GEMM sizes beyond that -- measured 25 s/step with 128 threads on the 128-core GPU host)."""
    return max(1, min(os.cpu_count() or 1, 32))


# -------------------------------------------------------------------------------------------------------------
# CPU legs: the oracle port of the reference algorithm on the host cores (bounded samples, extrapolated, labelled)
# -------------------------------------------------------------------------------------------------------------
def cpu_posenet_step_s(sd, n_clips, frames, n_steps, threads, guided=False):
    """Seconds per ancestral PoseNet step (denoiser + posterior update + RNG [+ skating guidance autograd])."""
    from oracle import diffusion_oracle as do
    from oracle import pipeline_oracle
    from rohm_b200 import synthetic
    torch.set_num_threads(threads)
    tables, tmap = do.create_diffusion('cosine', DIFFUSION_STEPS, '')
    ds = synthetic.make_dataset('pose', seed=3, realistic_std=True) if guided else synthetic.make_dataset('pose')
    cond = (synthetic.plausible_motion(n_clips, frames, 3, ds) if guided else synthetic.posenet_batch(n_clips, frames, 3)['cond'])
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n_clips, C_FEATS, 1, frames, generator=g)
    body = synthetic.smplx_like_model(0) if guided else None
    mean, std = torch.from_numpy(ds.Mean), torch.from_numpy(ds.Std)
    first = 40 if guided else DIFFUSION_STEPS - 1
    pipeline_oracle.posenet_guided_step(tables, tmap, first, x, cond, sd, mean, std, body, torch.randn(x.shape, generator=g),
                                        guided=guided)  # warm-up
    t0 = time.perf_counter()
    for i in range(first, first - n_steps, -1):
        x, _ = pipeline_oracle.posenet_guided_step(tables, tmap, i, x, cond, sd, mean, std, body,
                                                   torch.randn(x.shape, generator=g), guided=guided)
    return (time.perf_counter() - t0) / n_steps


def cpu_trajnet_step_s(sd, n_clips, frames, n_steps, threads, control):
    from oracle import diffusion_oracle as do
    from oracle import trajnet_oracle
    from rohm_b200 import synthetic
    torch.set_num_threads(threads)
    tables, tmap = do.create_diffusion('cosine', DIFFUSION_STEPS, '')
    b = synthetic.trajnet_batch(n_clips, frames, 3, control=control)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n_clips, frames, 13, generator=g)
    fwd = lambda x_, t: trajnet_oracle.trajnet_forward(sd, x_, b['cond'], torch.full((n_clips,), t, dtype=torch.long),
                                                       control_cond=b.get('control_cond'))
    with torch.no_grad():
        fwd(x, 999)
        t0 = time.perf_counter()
        for i in range(DIFFUSION_STEPS - 1, DIFFUSION_STEPS - 1 - n_steps, -1):
            x = do.p_sample_step(tables, i, x, fwd(x, tmap[i]), torch.randn(x.shape, generator=g))
        return (time.perf_counter() - t0) / n_steps


def cpu_lbs_frame_s(n_frames, threads):
    from oracle import kinematics_oracle as ko
    from rohm_b200 import synthetic
    torch.set_num_threads(threads)
    model = synthetic.smplx_like_model(0)
    g = torch.Generator().manual_seed(0)
    go, bp = 0.3 * torch.randn(n_frames, 3, generator=g), 0.3 * torch.randn(n_frames, 63, generator=g)
    be, tr = torch.randn(n_frames, 10, generator=g), torch.randn(n_frames, 3, generator=g)
    ko.smplx_forward(model, go[:8], bp[:8], be[:8], tr[:8], return_verts=True)
    t0 = time.perf_counter()
    ko.smplx_forward(model, go, bp, be, tr, return_verts=True)
    return (time.perf_counter() - t0) / n_frames


def cpu_leg(config, traj_steps, samples, cores):
    """(clips/s of the oracle port on `cores` host threads, description of the bounded sample)."""
    B, T = CONFIGS[config]["clips"], CONFIGS[config]["frames"]
    if config == "posenet":
        _, sd = build_posenet(None)
        s = cpu_posenet_step_s(sd, B, T, samples, cores)
        return B / (s * DIFFUSION_STEPS), (f"{B} clips x {samples} consecutive DDPM steps of the oracle port (PoseNet forward + "
                                           f"posterior update + RNG, {s:.2f} s/step), extrapolated linearly to 1000 steps")
    if config == "trajcontrol":
        _, sd = build_trajnet(None, True)
        s = cpu_trajnet_step_s(sd, B, T, samples, cores, True)
        return B / (s * DIFFUSION_STEPS), (f"{B} clips x {samples} consecutive DDPM steps of the oracle port (TrajNet+TrajControl, "
                                           f"{s:.2f} s/step), extrapolated linearly to 1000 steps")
    if config == "respaced100":
        _, sdp = build_posenet(None)
        _, sdt = build_trajnet(None, False)
        nb = 32  # a quarter of the 128-clip batch (step cost is linear in clips at this size)
        sp = cpu_posenet_step_s(sdp, nb, T, max(2, samples // 4), cores)
        st = cpu_trajnet_step_s(sdt, nb, T, max(2, samples // 4), cores, False)
        return nb / (100 * (sp + st)), (f"{nb} clips x {max(2, samples // 4)} steps of each denoiser's oracle port ({sp:.2f} + "
                                        f"{st:.2f} s/step), extrapolated to 100 + 100 steps")
    if config == "pipeline":
        _, sdp = build_posenet(None)
        _, sdt = build_trajnet(None, False)
        _, sdc = build_trajnet(None, True, seed=4)
        nb = 8
        sp = cpu_posenet_step_s(sdp, nb, 143, max(2, samples // 8), cores)
        sg = cpu_posenet_step_s(sdp, nb, 143, 5, cores, guided=True)
        st = cpu_trajnet_step_s(sdt, nb, T, 4, cores, False)
        sc = cpu_trajnet_step_s(sdc, nb, T, 4, cores, True)
        total = 3 * (949 * sp + 51 * sg) + traj_steps * (st + 2 * sc)
        return nb / total, (f"{nb} clips: {max(2, samples // 8)} unguided + 5 guided PoseNet steps, 4 TrajNet + 4 TrajControl steps "
                            f"of the oracle port ({sp:.2f} / {sg:.2f} / {st:.2f} / {sc:.2f} s/step), extrapolated to 3 rounds x "
                            f"(949 + 51 guided) + {traj_steps} x 3 steps; host glue and LBS excluded (favours the CPU)")
    if config == "lbs":
        n = 64
        s = cpu_lbs_frame_s(n, cores)
        return 1.0 / (s * T), f"{n} frames of the oracle SMPL-X forward with vertices ({s * 1e3:.1f} ms/frame), x {T} frames per clip"
    raise SystemExit(f"unknown config {config}")


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = host_threads()
    cfg = CONFIGS[args.config]
    vals, descr = [], ""
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_leg(args.config, args.traj_steps, 2, cores)
    for _ in range(args.steps):
        v, descr = cpu_leg(args.config, args.traj_steps, 16, cores)
        vals.append(v)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": "clips/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * cfg["clips"] / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus, "cpu"),
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": "port", "sample": descr},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference is pure python with absent dependencies (smplx, configargparse, torch 1.9) and cannot travel "
                "to the GPU box; this is the oracle port (pinned to the reference by tests/golden) on the host cores, "
                "extrapolated from a bounded sample",
    }
    print(json.dumps(line))


def workload_config(args, n_gpus, device_kind):
    cfg = CONFIGS[args.config]
    d = {"workload": cfg["label"], "name": args.config, "clips_per_gpu": cfg["clips"], "global_batch": cfg["clips"] * n_gpus,
         "frames": cfg["frames"], "diffusion_steps": 100 if args.config == "respaced100" else DIFFUSION_STEPS,
         "parallelism": f"clip-sharded x{n_gpus} (no intra-step collective)",
         "precision_mode": os.environ.get("ROHM_B200_PRECISION", "f16x2"),
         "l2": "flushed (256 MiB write) between timed iterations", "device": device_kind}
    if args.config == "pipeline":
        d["rounds"], d["traj_steps"] = 3, args.traj_steps
    return d


# -------------------------------------------------------------------------------------------------------------
# GPU workloads: each returns (resident_fn, e2e_fn, h2d_bytes, d2h_bytes, extras_fn)
# -------------------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, args, dev, rank, world):
        self.args, self.dev, self.rank, self.world = args, dev, rank, world
        self.cfg = CONFIGS[args.config]
        self.B, self.T = self.cfg["clips"], self.cfg["frames"]
        self.launches_per_step = 0
        getattr(self, "_setup_" + args.config)()

    # ---- posenet -------------------------------------------------------------------------------------------
    def _setup_posenet(self):
        from rohm_b200 import synthetic
        self.model, self.sd = build_posenet(self.dev)
        self.diff = make_diffusion('pose', DIFFUSION_STEPS, '', self.dev)
        self.shape = [self.B, C_FEATS, 1, self.T]
        self.host_in = {'cond': synthetic.posenet_batch(self.B, self.T, 100 + self.rank)['cond'].pin_memory()}
        self.dev_in = {k: v.to(self.dev) for k, v in self.host_in.items()}
        self.out_shape = self.shape

    def _run_posenet(self, batch):
        return self.diff.eval_losses(model=self.model, batch=batch, shape=self.shape, progress=False, clip_denoised=False,
                                     cond_fn_with_grad=False, compute_loss=False)[1]

    # ---- trajcontrol ---------------------------------------------------------------------------------------
    def _setup_trajcontrol(self):
        from rohm_b200 import synthetic
        self.model, self.sd = build_trajnet(self.dev, True)
        self.diff = make_diffusion('traj', DIFFUSION_STEPS, '', self.dev)
        self.shape = [self.B, self.T, 13]
        hb = synthetic.trajnet_batch(self.B, self.T, 100 + self.rank, control=True)
        self.host_in = {k: hb[k].pin_memory() for k in ('cond', 'control_cond')}
        self.dev_in = {k: v.to(self.dev) for k, v in self.host_in.items()}
        self.out_shape = self.shape

    def _run_trajcontrol(self, batch):
        return self.diff.eval_losses(model=self.model, batch=batch, shape=self.shape, progress=False, clip_denoised=False,
                                     cond_fn_with_grad=True, compute_loss=False)[1]

    # ---- respaced100 ---------------------------------------------------------------------------------------
    def _setup_respaced100(self):
        from rohm_b200 import synthetic
        self.model, self.sd = build_posenet(self.dev)
        self.tmodel, self.tsd = build_trajnet(self.dev, False)
        self.diff = make_diffusion('pose', DIFFUSION_STEPS, 'ddim100', self.dev)
        self.tdiff = make_diffusion('traj', DIFFUSION_STEPS, 'ddim100', self.dev)
        self.shape, self.tshape = [self.B, C_FEATS, 1, self.T], [self.B, self.T, 13]
        self.host_in = {'cond': synthetic.posenet_batch(self.B, self.T, 100 + self.rank)['cond'].pin_memory(),
                        'tcond': synthetic.trajnet_batch(self.B, self.T, 200 + self.rank)['cond'].pin_memory()}
        self.dev_in = {k: v.to(self.dev) for k, v in self.host_in.items()}
        self.out_shape = self.shape

    def _run_respaced100(self, batch):
        # respaced ancestral sampling: what the reference can run on a 'ddim100'-respaced object (SURVEY D4)
        t = self.tdiff.p_sample_loop(self.tmodel, {'cond': batch['tcond']}, self.tshape, clip_denoised=False,
                                     cond_fn_with_grad=True)
        p = self.diff.p_sample_loop(self.model, {'cond': batch['cond']}, self.shape, clip_denoised=False,
                                    cond_fn_with_grad=False)
        self._traj_out = t
        return p

    # ---- pipeline ------------------------------------------------------------------------------------------
    def _setup_pipeline(self):
        from rohm_b200 import pipeline, synthetic
        from rohm_b200.body_model import BodyModel
        self.ds_pose = synthetic.make_dataset('pose', seed=3, realistic_std=True)
        self.ds_traj = synthetic.make_dataset('traj', seed=3, realistic_std=True)
        self.model, self.sd = build_posenet(self.dev, self.ds_pose)
        self.tmodel, _ = build_trajnet(self.dev, False, self.ds_traj)
        self.cmodel, _ = build_trajnet(self.dev, True, self.ds_traj, seed=4)
        self.body = BodyModel.create('', device=self.dev, seed=0)
        self.diff = make_diffusion('pose', DIFFUSION_STEPS, '', self.dev)
        self.tdiff = make_diffusion('traj', self.args.traj_steps, '', self.dev)
        self.cdiff = make_diffusion('traj', self.args.traj_steps, '', self.dev)
        self.pargs = pipeline.make_args(sample_iter=3, mask_scheme='lower')
        pose, traj = synthetic.pipeline_batches(self.B, 100 + self.rank, self.ds_pose, frames=self.T)
        self.host_in = {f"pose_{k}": v.pin_memory() for k, v in pose.items()}
        self.host_in.update({f"traj_{k}": v.pin_memory() for k, v in traj.items()})
        self.dev_in = {k: v.to(self.dev) for k, v in self.host_in.items()}
        self.out_shape = [self.B, C_FEATS, 1, self.T - 1]
        self.stage_ms = {}

    def _run_pipeline(self, batch):
        from rohm_b200 import pipeline
        pose = {k[5:]: v.clone() for k, v in batch.items() if k.startswith("pose_")}
        traj = {k[5:]: v.clone() for k, v in batch.items() if k.startswith("traj_")}
        vp, vt, tn = pipeline.run_rounds(self.pargs, self.model, self.tmodel, self.cmodel, self.diff, self.tdiff, self.cdiff,
                                         self.ds_pose, self.ds_traj, self.body, pose, traj)
        self._traj_out, self._traj_noisy = vt, tn
        self._recon = pipeline.reconstruct_outputs(self.pargs, self.ds_pose, self.body, pose, vp, tn, return_verts=True)
        return vp

    # ---- lbs -----------------------------------------------------------------------------------------------
    def _setup_lbs(self):
        from rohm_b200 import glue, synthetic
        from rohm_b200.body_model import BodyModel, kernels_for
        self.ds_pose = synthetic.make_dataset('pose', seed=3, realistic_std=True)
        self.body = BodyModel.create('', device=self.dev, seed=0)
        x = synthetic.plausible_motion(self.B, self.T, 100 + self.rank, self.ds_pose)
        self.host_in = {'x': x.pin_memory()}
        self.dev_in = {'x': x.to(self.dev)}
        self.mean, self.std = glue.stats_on(self.ds_pose, self.dev)
        self.k = kernels_for(self.body, self.dev, self.B * self.T, with_vertices=True)
        self.out_shape = [self.B, self.T, 10475, 3]

    def _run_lbs(self, batch):
        self._joints, verts = self.k.from_repr(batch['x'], self.mean, self.std, want_vertices=True)
        return verts

    # ---- common --------------------------------------------------------------------------------------------
    def run(self, batch):
        return getattr(self, "_run_" + self.args.config)(batch)

    def outputs(self, out):
        """Every array a caller of run() receives from the step that returned `out`, by name."""
        c = self.args.config
        if c == "respaced100":
            return {"pose": out, "traj": self._traj_out}
        if c == "pipeline":
            return {"val_output_pose": out, "val_output_traj": self._traj_out, "traj_noisy_full": self._traj_noisy,
                    **{k: v for k, v in self._recon.items() if v is not None}}
        if c == "lbs":
            return {"joints": self._joints, "vertices": out}
        return {"pose" if c == "posenet" else "traj": out}

    def h2d_bytes(self):
        return int(sum(v.numel() * v.element_size() for v in self.host_in.values()))


def dump_outputs(dirname, arrays):
    """Writes each array as <dirname>/<name>.npy (float64 stays float64, everything else becomes float32).  An array of more
    than DUMP_WHOLE_MAX_ELEMS elements is written as <name>_sample.npy instead: DUMP_SAMPLE_ELEMS elements of its flattened
    contents at sorted indices drawn from a fixed seed, so two runs with the same shapes sample the same positions."""
    host = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.dtype != torch.float64:
            t = t.float()
        if t.numel() > DUMP_WHOLE_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        host[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rohm_b200", choices=["rohm_b200", "reference"])
    ap.add_argument("--config", default="posenet", choices=list(CONFIGS))
    ap.add_argument("--traj-steps", type=int, default=100, help="TrajNet diffusion steps of the pipeline config "
                    "(100 = every shipped RoHM config; 1000 = BASELINE's wording)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as "
                    "DIR/<name>.npy (rank 0's clips; arrays over 32 MB as a fixed, seeded sample; 64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun for --gpus > 1 (one rank per GPU)")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)

    w = Workload(args, dev, rank, world)
    B = w.B
    # lbs: the host reads the joints back; the 575 MB of vertices stay on the device (rendering / metrics consume them there)
    out_host = torch.empty(w.out_shape if args.config != "lbs" else [B, w.T, 22, 3], dtype=torch.float32).pin_memory()
    gathered = torch.empty([world * B] + list(w.out_shape[1:]), device=dev) if (distributed and args.config != "lbs") else None
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB L2
    torch.manual_seed(1234 + rank)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def one_step_resident():
        out = w.run(w.dev_in)
        if gathered is not None:
            dist.all_gather_into_tensor(gathered, out)
        last["out"] = out
        return out

    def one_step_e2e():
        batch = {k: v.to(dev, non_blocking=True) for k, v in w.host_in.items()}
        out = w.run(batch)
        if gathered is not None:
            dist.all_gather_into_tensor(gathered, out)
        out_host.copy_(w._joints if args.config == "lbs" else out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, k):
        """k iterations, each bracketed by CUDA events on the launching stream, L2 flushed in between (untimed)."""
        evs = []
        for _ in range(k):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)

    def maxreduce(ms):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        one_step_resident()
    barrier()
    with ClockSampler(local) as clocks:
        ms_total = timed(one_step_resident, args.steps)
        barrier()
    ms_per_step = maxreduce(ms_total) / args.steps
    value = world * B / (ms_per_step / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w.outputs(last["out"]))

    one_step_e2e()
    barrier()
    e2e_ms = timed(one_step_e2e, args.steps)
    barrier()
    e2e_value = world * B / (maxreduce(e2e_ms) / args.steps / 1000.0)

    peaks = read_peaks()
    roofline, launches, dtype = ROOFLINES[args.config](w, peaks, ms_per_step)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_threads()
        v, descr = cpu_leg(args.config, args.traj_steps, 48 if args.config == "posenet" else 16, cores)
        cpu_baseline = {"value": v, "unit": "clips/s", "cores": cores, "kind": "port",
                        "sample": f"{descr} ({cores} of {os.cpu_count()} host threads)"}

    if rank == 0:
        d2h = out_host.numel() * 4
        line = {
            "metric": w.cfg["metric"], "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": workload_config(args, world, "B200"),
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": w.h2d_bytes(), "d2h_bytes_per_step": d2h},
            "gpu_launches": args.steps * launches,
            "roofline": roofline,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line))
    if distributed:
        dist.destroy_process_group()


# -------------------------------------------------------------------------------------------------------------
# per-config roofline objects (measured live with CUDA events; ncu traffic figures come from profiles/)
# -------------------------------------------------------------------------------------------------------------
def _traffic(name):
    tp = os.path.join(ROOT, "profiles", name)
    if os.path.exists(tp):
        tj = json.load(open(tp))
        return tj.get("dram_bytes_per_launch"), f"profiles/{name} ({tj.get('source', 'ncu --set full')})"
    return None, None


def _event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def posenet_roofline(w, peaks, ms_per_step, model=None, B=None, T=None):
    model = model if model is not None else w.model
    B, T = (B or w.B), (T or w.T)
    engine = model._engine
    x = torch.randn([B, C_FEATS, 1, T], device=w.dev)
    ts = torch.full((B,), 500, device=w.dev, dtype=torch.int64)
    cat_ms = {"gemm": 0.0, "attention": 0.0, "layernorm": 0.0, "other": 0.0}
    cat_n = dict.fromkeys(cat_ms, 0)
    reps = 10
    for _ in range(reps):
        ms, n = engine.profile(x, ts)
        for k in cat_ms:
            cat_ms[k] += ms[k] / reps
            cat_n[k] = n[k]
    out = torch.empty_like(x)
    graph_ms = _event_ms(lambda: engine.forward(x, ts, out), 50)  # the forward as it runs in the loop (CUDA graph, warm L2)
    # the whole sampler step as it runs in the loop (forward + in-kernel-noise update, one graph launch), device and host side
    coef_row = torch.zeros(8, device=w.dev)
    step_graph_ms = _event_ms(lambda: engine.sample_step(x, ts, coef_row), 50)
    t0 = time.perf_counter()
    for _ in range(50):
        engine.sample_step(x, ts, coef_row)
    host_us = (time.perf_counter() - t0) / 50 * 1e6  # enqueue cost (the GPU runs behind): must stay below the device time
    torch.cuda.synchronize()
    flops = gemm_flops_per_forward(B, T + 1)
    gemm_s = cat_ms["gemm"] / 1000.0
    achieved = flops / gemm_s / 1e12 if gemm_s > 0 else None
    share = cat_ms["gemm"] / max(sum(cat_ms.values()), 1e-9)
    achieved_graph = flops / (graph_ms * share / 1000.0) / 1e12  # GEMM share of the graph time (no per-launch event overhead)
    prec = engine.precision
    passes = 1 if prec == 1 else 3
    kernel_kind = {3: "tcgen05 kind::tf32 on TF32 hi/lo pairs, 3 products", 2: "tcgen05 kind::f16 on fp16 hi/lo pairs, 3 products",
                   1: "tcgen05 kind::tf32, single pass"}[prec]
    pipe_peak = peaks["bf16_tflops"] if prec == 2 else peaks["bf16_tflops"] / 2.0
    traffic, traffic_src = _traffic("r2_gemm_traffic.json")
    if traffic is None:
        traffic, traffic_src = _traffic("r1_gemm_traffic.json")
    roofline = {
        "kernel": f"gemm kernels ({kernel_kind}), {cat_n['gemm']} launches per PoseNet forward",
        # achieved = algorithmic GEMM FLOPs / (GEMM share of the forward x forward time as it runs in the loop).  The share comes
        # from CUDA events around every launch (rohm_posenet_profile: serialised, no PDL overlap, ~4 us of event overhead per
        # launch -- so only the SHARE is taken from it, which the ncu launch list under profiles/ reproduces); the forward time
        # is the captured graph timed with events on the launching stream, warm L2.  The raw event-timed figure is kept below.
        "bound": "tensor", "achieved": achieved_graph, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": achieved_graph / peaks["bf16_tflops"], "traffic": traffic,
        "traffic_source": traffic_src, "traffic_note": "cold-cache ncu figure; inside the loop operands are L2 hits",
        "peak_source": peaks["source"] + ", sustained bf16",
        "algorithmic_flops_per_forward": flops, "avg_launch_us": 1000.0 * graph_ms * share / max(cat_n["gemm"], 1),
        "achieved_event_timed": achieved, "frac_event_timed": (achieved / peaks["bf16_tflops"]) if achieved else None,
        "avg_launch_us_event_timed": 1000.0 * cat_ms["gemm"] / max(cat_n["gemm"], 1),
        "tensor_pipe_frac": achieved_graph * passes / pipe_peak,
        "tensor_pipe_frac_note": "issued tensor work (3 products per algorithmic flop) / peak of that operand type",
        "share_of_forward": {k: cat_ms[k] / max(sum(cat_ms.values()), 1e-9) for k in cat_ms},
        "forward_ms_by_kernel_class": cat_ms, "launches_by_kernel_class": cat_n,
        "forward_graph_ms": graph_ms, "step_graph_ms": step_graph_ms, "host_enqueue_us_per_step": host_us,
        # GEMMs + attention (QK^T and PV: 4 S^2 D per clip and layer) over the whole forward graph
        "whole_forward_tflops": (flops + B * 8 * 4.0 * (T + 1) * (T + 1) * 512) / (graph_ms / 1000.0) / 1e12,
    }
    dtype = {3: "f32 (TF32 hi/lo error-compensated tensor-core GEMMs)", 2: "f32 (fp16 hi/lo error-compensated tensor-core GEMMs)",
             1: "tf32"}[prec]
    return roofline, engine.launches_per_forward, dtype


def _roof_posenet(w, peaks, ms_per_step):
    r, lf, dtype = posenet_roofline(w, peaks, ms_per_step)
    return r, DIFFUSION_STEPS * (lf + 1), dtype


def trajnet_roofline(w, peaks, model, B, T, control):
    from rohm_b200 import synthetic
    b = {k: v.to(w.dev) for k, v in synthetic.trajnet_batch(B, T, 5, control=control).items()}
    b['x_t'] = torch.randn(B, T, 13, device=w.dev)
    ts = torch.full((B,), 500, device=w.dev, dtype=torch.long)
    fwd_ms = _event_ms(lambda: model(b, ts), 50)
    eng = model._engine
    per_clip = 1.144e9 if control else 0.723e9
    step_invariant = 0.152e9  # cond pyramid, hoisted out of the step (SURVEY 8d)
    flops = B * (per_clip - step_invariant)
    achieved = flops / (fwd_ms / 1000.0) / 1e12
    traffic, src = _traffic("r2_trajnet_traffic.json")
    return {
        "kernel": f"TrajNet{'+TrajControl' if control else ''} forward: conv-as-GEMM tcgen05 kernels (fp16 hi/lo pairs, 3 products) + "
                  f"GroupNorm/Mish, {eng.launches_per_forward} launches, one CUDA graph",
        "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": achieved / peaks["bf16_tflops"], "traffic": traffic, "traffic_source": src,
        "peak_source": peaks["source"] + ", sustained bf16",
        "algorithmic_flops_per_forward": flops, "forward_ms": fwd_ms,
        "note": "achieved = per-step algorithmic conv FLOPs (step-invariant cond pyramid excluded) / WHOLE forward time: the "
                "forward is launch-latency bound at this size, so the whole graph is the honest denominator",
    }, eng.launches_per_forward


def _roof_trajcontrol(w, peaks, ms_per_step):
    r, lf = trajnet_roofline(w, peaks, w.model, w.B, w.T, True)
    return r, DIFFUSION_STEPS * (lf + 1), "f32 (fp16 hi/lo error-compensated tensor-core conv GEMMs)"


def lbs_roofline(w, peaks, body, B, T):
    from rohm_b200 import glue, synthetic
    from rohm_b200.body_model import kernels_for
    ds = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    x = synthetic.plausible_motion(B, T, 7, ds).to(w.dev)
    mean, std = glue.stats_on(ds, w.dev)
    k = kernels_for(body, w.dev, B * T, with_vertices=True)
    ms = _event_ms(lambda: k.from_repr(x, mean, std, want_vertices=True), 10)
    frames = B * T
    achieved = frames * LBS_BYTES_PER_FRAME / (ms / 1000.0) / 1e9
    traffic, src = _traffic("r2_lbs_traffic.json")
    return {
        "kernel": "SMPL-X LBS: repr->axis-angle, 55-joint FK, pose/shape blend (tcgen05 GEMM on fp16 pairs) + skinning",
        "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
        "traffic": traffic, "traffic_source": src, "peak_source": peaks["source"] + ", STREAM-style copy",
        "algorithmic_bytes_per_frame": LBS_BYTES_PER_FRAME, "frames": frames, "call_ms": ms,
        "note": "the pose-corrective blend is 30.5 MFLOP/frame x 3 tensor passes: at the HBM rate of 70 % of peak it would need "
                "> 1.7 PFLOP/s of tensor work, so this kernel is tensor-bound, not HBM-bound (SURVEY H5); the fraction against HBM "
                "is reported because north_star asks for it",
    }, ms


def _roof_lbs(w, peaks, ms_per_step):
    r, _ = lbs_roofline(w, peaks, w.body, w.B, w.T)
    return r, 5, "f32 (fp16 hi/lo error-compensated blend GEMM, fp32 skinning)"


def _roof_respaced100(w, peaks, ms_per_step):
    r, lf, dtype = posenet_roofline(w, peaks, ms_per_step)
    rt, ltf = trajnet_roofline(w, peaks, w.tmodel, w.B, w.T, False)
    r["trajnet"] = rt
    return r, 100 * (lf + 1) + 100 * (ltf + 1), dtype


def _roof_pipeline(w, peaks, ms_per_step):
    from rohm_b200 import glue
    r, lf, dtype = posenet_roofline(w, peaks, ms_per_step, B=w.B, T=w.T - 1)
    rt, ltf = trajnet_roofline(w, peaks, w.cmodel, w.B, w.T, True)
    rl, lbs_ms = lbs_roofline(w, peaks, w.body, w.B, w.T - 1)
    # stage costs (CUDA events, warm): glue, guidance
    traj_out = torch.randn(w.B, w.T, 13, device=w.dev)
    clean = w.dev_in["traj_motion_repr_clean"]
    glue_ms = _event_ms(lambda: glue.traj_to_full_repr(w.body, traj_out, clean, w.ds_traj, w.ds_pose), 20)
    x0 = torch.randn(w.B, C_FEATS, 1, w.T - 1, device=w.dev)
    guide_ms = _event_ms(lambda: w.model.guide_skating_with_smpl({}, {'pred_xstart': x0}, None, compute_grad='x_0'), 20)
    cond_ms = _event_ms(lambda: glue.build_pose_cond(w.dev_in["pose_motion_repr_noisy"], None, glue.channel_keep_mask('lower'),
                                                     zero_contact=True, frames=w.T - 1), 20)
    r["trajnet_control"] = rt
    r["lbs"] = rl
    r["stages_ms_per_pipeline_pass"] = {
        "posenet_sampling_3x1000": 3 * DIFFUSION_STEPS * r["forward_graph_ms"], "skating_guidance_3x51_calls": 3 * 51 * guide_ms,
        "trajnet_sampling": w.args.traj_steps * 3 * rt["forward_ms"], "inter_round_glue_3_calls": 3 * glue_ms,
        "pose_cond_assembly_3_calls": 3 * cond_ms, "post_loop_lbs_3_calls": 3 * lbs_ms, "whole_pass_measured": ms_per_step}
    r["glue_fraction_of_pass"] = 3 * (glue_ms + cond_ms) / ms_per_step
    launches = 3 * (DIFFUSION_STEPS * (lf + 1) + 51 * 5 + w.args.traj_steps * (ltf + 1) + 8) + 15
    return r, launches, dtype


ROOFLINES = {"posenet": _roof_posenet, "trajcontrol": _roof_trajcontrol, "lbs": _roof_lbs, "respaced100": _roof_respaced100,
             "pipeline": _roof_pipeline}


if __name__ == "__main__":
    main()
