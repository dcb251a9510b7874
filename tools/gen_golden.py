"""Generates tests/golden/*.npz by running the UNMODIFIED reference (sanweiliti/RoHM mounted at /root/reference) on
seeded synthetic weights and inputs.  Run in the build container only (the reference does not travel to the GPU box):

    python tools/gen_golden.py

Everything needed to regenerate an input is a seed: weights come from rohm_b200.synthetic.synth_state_dict, inputs
from torch.Generator streams.  The only stand-in is the third-party ``smplx`` package (absent, licence-gated model):
``smplx.create`` returns the oracle's SMPL-X restatement on the synthetic body model, so the reference code around
the body-model call (rot6d -> axis-angle, losses, autograd) is the real thing.
"""
import argparse
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.append('/root/reference')  # AFTER the repo: only used for the reference's own top-level packages below

import numpy as np
import torch
import torch.nn as nn

from oracle import kinematics_oracle as ko
from rohm_b200 import synthetic

OUT = os.path.join(ROOT, "tests", "golden")


class _StubBody(nn.Module):
    """smplx stand-in: same call signature / output attributes, arithmetic = oracle restatement."""

    def __init__(self):
        super().__init__()
        self.model = synthetic.smplx_like_model(0)

    def forward(self, transl=None, global_orient=None, body_pose=None, betas=None, **unused):
        joints, verts = ko.smplx_forward(self.model, global_orient, body_pose, betas, transl, return_verts=False)
        return types.SimpleNamespace(joints=joints, vertices=verts)


def import_reference():
    stub = types.ModuleType('smplx')
    stub.create = lambda **kw: _StubBody()
    sys.modules['smplx'] = stub
    # make sure the reference's namespace packages win for these imports
    for name in ("model", "diffusion", "utils", "data_loaders"):
        sys.modules.pop(name, None)
    sys.path.insert(0, '/root/reference')
    import diffusion.gaussian_diffusion_posenet as gdp
    import diffusion.gaussian_diffusion_trajnet as gdt
    import diffusion.respace as respace
    import utils.model_util as model_util
    import model.posenet as ref_posenet
    import model.trajnet as ref_trajnet
    import data_loaders.motion_representation as mr
    import data_loaders.common.quaternion as quat
    import utils.konia_transform as kt
    import utils.other_utils as ou
    sys.path.pop(0)
    return types.SimpleNamespace(gdp=gdp, gdt=gdt, respace=respace, model_util=model_util, posenet=ref_posenet,
                                 trajnet=ref_trajnet, mr=mr, quat=quat, kt=kt, ou=ou)


TABLES = ("betas", "alphas_cumprod", "alphas_cumprod_prev", "alphas_cumprod_next", "sqrt_alphas_cumprod",
          "sqrt_one_minus_alphas_cumprod", "log_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
          "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
          "posterior_mean_coef1", "posterior_mean_coef2")


def gen_schedules(ref):
    out = {}
    cases = [("cosine", 1000, ''), ("cosine", 100, ''), ("cosine", 50, ''), ("cosine", 1000, 'ddim100'),
             ("cosine", 1000, '100'), ("cosine", 1000, 'ddim50'), ("cosine", 300, '10,15,20'), ("linear", 100, ''),
             ("linear", 1000, 'ddim20')]
    for idx, (sched, steps, resp) in enumerate(cases):
        args = argparse.Namespace(noise_schedule=sched, sigma_small=True)
        d = ref.model_util.create_gaussian_diffusion(args, gd=ref.gdp, return_class=ref.respace.SpacedDiffusionPoseNet,
                                                     num_diffusion_timesteps=steps, timestep_respacing=resp, device='cpu')
        out[f"c{idx}_meta"] = np.array([sched, str(steps), resp])
        out[f"c{idx}_timestep_map"] = np.array(d.timestep_map, dtype=np.int64)
        for t in TABLES:
            out[f"c{idx}_{t}"] = getattr(d, t)
    out["n_cases"] = np.array(len(cases))
    # space_timesteps known answers
    out["space_300_10_15_20"] = np.array(sorted(ref.respace.space_timesteps(300, [10, 15, 20])), dtype=np.int64)
    out["space_1000_ddim100"] = np.array(sorted(ref.respace.space_timesteps(1000, "ddim100")), dtype=np.int64)
    out["space_1000_100"] = np.array(sorted(ref.respace.space_timesteps(1000, "100")), dtype=np.int64)
    out["space_1000_7_13_29"] = np.array(sorted(ref.respace.space_timesteps(1000, "7,13,29")), dtype=np.int64)
    try:
        ref.respace.space_timesteps(1000, "ddim300")
        out["ddim300_raises"] = np.array(0)
    except ValueError:
        out["ddim300_raises"] = np.array(1)
    np.savez_compressed(os.path.join(OUT, "schedules.npz"), **out)
    print("schedules.npz", len(out), "arrays")


def build_ref_posenet(ref, seed, device='cpu'):
    ds = synthetic.make_dataset('pose')
    m = ref.posenet.PoseNet(dataset=ds, body_feat_dim=294, latent_dim=512, ff_size=1024, num_layers=8, num_heads=4,
                            dropout=0.1, activation="gelu", body_model_path='', device=device, traj_feat_dim=22)
    sd = synthetic.synth_state_dict(m, seed)
    m.load_state_dict(sd)
    return m.eval(), sd


def build_ref_trajnet(ref, seed, control):
    ds = synthetic.make_dataset('traj')
    m = ref.trajnet.TrajNet(time_dim=32, mid_dim=512, cond_dim=13, traj_feat_dim=13, trajcontrol=control, device='cpu',
                            dataset=ds, repr_abs_only=True)
    sd = synthetic.synth_state_dict(m, seed)
    m.load_state_dict(sd)
    return m.eval(), sd


def gen_posenet(ref):
    out = {}
    m, _ = build_ref_posenet(ref, seed=1)
    for idx, (B, T, s) in enumerate([(2, 16, 11), (1, 8, 12), (1, 143, 13)]):
        g = torch.Generator().manual_seed(s)
        x = torch.randn(B, 294, 1, T, generator=g)
        cond = synthetic.posenet_batch(B, T, s + 100)['cond']
        ts = torch.randint(0, 1000, (B,), generator=g)
        with torch.no_grad():
            y = m({'x_t': x, 'cond': cond}, ts)
        out[f"c{idx}_meta"] = np.array([B, T, s])
        out[f"c{idx}_timesteps"] = ts.numpy()
        out[f"c{idx}_out"] = y.numpy()
    out["n_cases"] = np.array(3)
    out["weight_seed"] = np.array(1)
    np.savez_compressed(os.path.join(OUT, "posenet_forward.npz"), **out)
    print("posenet_forward.npz")


def gen_trajnet(ref):
    out = {}
    idx = 0
    for control in (False, True):
        m, _ = build_ref_trajnet(ref, seed=2, control=control)
        for (B, T, s) in [(2, 32, 21), (1, 144, 22)]:
            g = torch.Generator().manual_seed(s)
            x = torch.randn(B, T, 13, generator=g)
            batch = synthetic.trajnet_batch(B, T, s + 100, control=control)
            batch['x_t'] = x
            ts = torch.randint(0, 100, (B,), generator=g)
            with torch.no_grad():
                y = m(batch, ts)
            out[f"c{idx}_meta"] = np.array([B, T, s, int(control)])
            out[f"c{idx}_timesteps"] = ts.numpy()
            out[f"c{idx}_out"] = y.numpy()
            idx += 1
    out["n_cases"] = np.array(idx)
    out["weight_seed"] = np.array(2)
    np.savez_compressed(os.path.join(OUT, "trajnet_forward.npz"), **out)
    print("trajnet_forward.npz")


class _NoiseTape:
    """A stand-in for the ``th`` name inside a reference diffusion module: forwards everything to torch except
    randn / randn_like, which draw from a seeded CPU stream (so the oracle and the CUDA path can replay it)."""

    def __init__(self, seed):
        self.g = torch.Generator().manual_seed(seed)

    def randn(self, *shape, device=None, **kw):
        return torch.randn(*shape, generator=self.g)

    def randn_like(self, x):
        return torch.randn(x.shape, generator=self.g)

    def __getattr__(self, name):
        return getattr(torch, name)


class _patched_th:
    def __init__(self, module, seed):
        self.module, self.tape = module, _NoiseTape(seed)

    def __enter__(self):
        self.real = self.module.th
        self.module.th = self.tape

    def __exit__(self, *a):
        self.module.th = self.real


def gen_sampling(ref):
    out = {}
    # (a) BASELINE config 1: TrajNet vanilla, 1 clip of 144 frames, 50 DDPM steps, through eval_losses
    m, _ = build_ref_trajnet(ref, seed=2, control=False)
    args = argparse.Namespace(noise_schedule='cosine', sigma_small=True)
    d = ref.model_util.create_gaussian_diffusion(args, gd=ref.gdt, return_class=ref.respace.SpacedDiffusionTrajNet,
                                                 num_diffusion_timesteps=50, timestep_respacing='', device='cpu')
    batch = synthetic.trajnet_batch(1, 144, 31)
    with _patched_th(ref.gdt, 41), torch.no_grad():
        _, y = d.eval_losses(model=m, batch=batch, shape=[1, 144, 13], progress=False, clip_denoised=False,
                             timestep_respacing='', cond_fn_with_grad=True, compute_loss=False, smplx_model=None)
    out["traj50_out"] = y.numpy()
    out["traj50_meta"] = np.array([1, 144, 31, 41, 50])

    # (b) PoseNet, respaced ancestral sampling ('ddim20' retained steps of a 1000-step base), 1 clip x 16 frames
    mp, _ = build_ref_posenet(ref, seed=1)
    dp = ref.model_util.create_gaussian_diffusion(args, gd=ref.gdp, return_class=ref.respace.SpacedDiffusionPoseNet,
                                                  num_diffusion_timesteps=1000, timestep_respacing='ddim20', device='cpu')
    batch = synthetic.posenet_batch(1, 16, 32)
    with _patched_th(ref.gdp, 42), torch.no_grad():
        y = dp.p_sample_loop(mp, batch, [1, 294, 1, 16], clip_denoised=False, cond_fn_with_grad=False)
    out["pose_ddim20_out"] = y.numpy()
    out["pose_ddim20_meta"] = np.array([1, 16, 32, 42, 20])

    # (c) PoseNet guided sampling (p_sample_with_grad, grad_type='amass') in the regime the guidance weights were
    #     tuned for: the last 12 steps of the 1000-step chain (skip_timesteps=988 -> t = 11..0, all guided), started
    #     from q_sample(init_image = a plausible motion).
    ds = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    mp.dataset = ds
    mp.device = 'cpu'
    dg = ref.model_util.create_gaussian_diffusion(args, gd=ref.gdp, return_class=ref.respace.SpacedDiffusionPoseNet,
                                                  num_diffusion_timesteps=1000, timestep_respacing='', device='cpu')
    init = synthetic.plausible_motion(2, 12, 33, ds)
    batch = {'cond': init.clone()}
    traj = []
    with _patched_th(ref.gdp, 43):
        for o in dg.p_sample_loop_progressive(mp, batch, [2, 294, 1, 12], clip_denoised=False, cond_fn_with_grad=True,
                                              grad_type='amass', skip_timesteps=994, init_image=init):
            traj.append((o['x_t'].detach().clone(), o['pred_xstart'].detach().clone(), o['sample'].detach().clone()))
    # The guided chain is ill-conditioned (weight 3e6 on a loss with hard masks; the reference README says results
    # are not reproducible across machines), so the fixture stores every step for teacher-forced comparison.
    out["pose_guided_xt"] = torch.stack([t[0] for t in traj]).numpy()
    out["pose_guided_x0"] = torch.stack([t[1] for t in traj]).numpy()
    out["pose_guided_sample"] = torch.stack([t[2] for t in traj]).numpy()
    out["pose_guided_meta"] = np.array([2, 12, 33, 43, 994])
    np.savez_compressed(os.path.join(OUT, "sampling.npz"), **out)
    print("sampling.npz")


def gen_kinematics(ref):
    out = {}
    g = torch.Generator().manual_seed(51)
    # rotations: generic, near identity, near pi, exactly identity
    r6 = torch.randn(64, 6, generator=g)
    near_id = torch.tensor([1., 0, 0, 1, 0, 0]).repeat(8, 1) + 1e-4 * torch.randn(8, 6, generator=g)
    ident = torch.tensor([[1., 0, 0, 1, 0, 0]])
    # rotation by ~pi about random axes, given as 6d (first two columns, row-major 3x2)
    ax = torch.nn.functional.normalize(torch.randn(8, 3, generator=g), dim=1)
    ang = (np.pi - 1e-3 * torch.rand(8, generator=g))
    K = torch.zeros(8, 3, 3)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 0], K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -ax[:, 2], ax[:, 1], ax[:, 2], -ax[:, 0], -ax[:, 1], ax[:, 0]
    Rpi = torch.eye(3) + torch.sin(ang)[:, None, None] * K + (1 - torch.cos(ang))[:, None, None] * (K @ K)
    r6 = torch.cat([r6, near_id, ident, Rpi[:, :, :2].reshape(8, 6)], dim=0)
    R = ref.quat.rot6d_to_rotmat(r6)
    aa = ref.kt.rotation_matrix_to_angle_axis(R)
    out["rot6d_in"], out["rotmat_out"], out["aa_out"] = r6.numpy(), R.numpy(), aa.numpy()

    # joint_abs_traj recovery and the skating guidance gradient on a plausible motion
    ds = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    x = synthetic.plausible_motion(2, 12, 52, ds)  # [2,294,1,12]
    full = x[:, :, 0].permute(0, 2, 1) * torch.from_numpy(ds.Std) + torch.from_numpy(ds.Mean)
    rep, cur = {}, 0
    for name in ko.REPR_LIST:
        rep[name] = full[..., cur:cur + ko.REPR_DIM_DICT[name]]
        cur += ko.REPR_DIM_DICT[name]
    body = _StubBody()
    out["abs_traj_joints"] = ref.mr.recover_from_repr_smpl(rep, recover_mode='joint_abs_traj', smplx_model=body).numpy()
    out["smplx_joints"] = ref.mr.recover_from_repr_smpl(rep, recover_mode='smplx_params', smplx_model=body).numpy()
    m, _ = build_ref_posenet(ref, seed=1)
    m.dataset, m.device = ds, 'cpu'
    grad = m.guide_skating_with_smpl({'x_t': x}, {'pred_xstart': x}, None, compute_grad='x_0')
    out["skating_grad"] = grad.detach().numpy()
    out["kin_meta"] = np.array([2, 12, 52, 3])
    np.savez_compressed(os.path.join(OUT, "kinematics.npz"), **out)
    print("kinematics.npz  grad absmax", float(grad.abs().max()))


def _rep_dict(full):
    rep, cur = {}, 0
    for name in ko.REPR_LIST:
        rep[name] = full[..., cur:cur + ko.REPR_DIM_DICT[name]]
        cur += ko.REPR_DIM_DICT[name]
    return rep


def gen_glue(ref):
    """Driver-side functions around the loops: get_repr_smplx (trajectory block), 'joint_rel_traj' recovery, the two
    compute_losses_with_smpl dictionaries and the 2-D reprojection guidance gradient (reference autograd)."""
    out = {}
    body = _StubBody()
    ds = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    # (a) get_repr_smplx on SMPL-X joints of a plausible motion, 2 clips x 24 frames (+ a clip that faces -y at one frame so
    #     the NaN repair of motion_representation.py:212-215 is exercised)
    x = synthetic.plausible_motion(2, 24, 61, ds)
    full = x[:, :, 0].permute(0, 2, 1) * torch.from_numpy(ds.Std) + torch.from_numpy(ds.Mean)
    rep = _rep_dict(full)
    joints = ref.mr.recover_from_repr_smpl(rep, recover_mode='smplx_params', smplx_model=body).numpy()
    traj = []
    for i in range(2):
        go = ref.kt.rotation_matrix_to_angle_axis(ref.quat.rot6d_to_rotmat(rep['smplx_rot_6d'][i]))
        bp = ref.kt.rotation_matrix_to_angle_axis(ref.quat.rot6d_to_rotmat(rep['smplx_body_pose_6d'][i].reshape(-1, 6)))
        params = {'transl': rep['smplx_trans'][i].numpy(), 'global_orient': go.numpy(),
                  'body_pose': bp.reshape(-1, 63).numpy(), 'betas': rep['smplx_betas'][i].numpy()}
        d = ref.mr.get_repr_smplx(positions=joints[i], smplx_params_dict=params, feet_vel_thre=5e-5)
        traj.append(np.concatenate([d[k] for k in ko.REPR_LIST], axis=-1)[:, 0:22])
    out["repr_x"] = x.numpy()
    out["repr_joints"] = joints
    out["repr_traj22"] = np.asarray(traj)
    out["repr_meta"] = np.array([2, 24, 61, 3])
    # NaN repair: hips/shoulders arranged so that the forward direction is exactly -y at frame 5
    pos = joints[0].copy()
    pos[5, 1], pos[5, 2], pos[5, 17], pos[5, 16] = [0, 0, 0], [1, 0, 0], [0, 0, 0], [1, 0, 0]
    go0 = ref.kt.rotation_matrix_to_angle_axis(ref.quat.rot6d_to_rotmat(rep['smplx_rot_6d'][0])).numpy()
    params = {'transl': rep['smplx_trans'][0].numpy(), 'global_orient': go0,
              'body_pose': np.zeros((24, 63), np.float32), 'betas': rep['smplx_betas'][0].numpy()}
    d = ref.mr.get_repr_smplx(positions=pos, smplx_params_dict=params, feet_vel_thre=5e-5)
    out["nan_positions"], out["nan_go"] = pos, go0
    out["nan_traj22"] = np.concatenate([d[k] for k in ko.REPR_LIST], axis=-1)[:, 0:22]
    # (b) joint_rel_traj recovery
    out["rel_traj_joints"] = ref.mr.recover_from_repr_smpl(rep, recover_mode='joint_rel_traj', smplx_model=body).numpy()
    # (c) evaluation loss dictionaries
    mp, _ = build_ref_posenet(ref, seed=1)
    mp.dataset, mp.device = ds, 'cpu'
    g = torch.Generator().manual_seed(62)
    rec = x + 0.05 * torch.randn(x.shape, generator=g)
    ld = mp.compute_losses_with_smpl({'motion_repr_clean': x}, rec, smplx_model=body, epoch=0)
    out["pose_loss_names"] = np.array(list(ld.keys()))
    out["pose_loss_values"] = np.array([float(v) for v in ld.values()], dtype=np.float64)
    out["pose_loss_rec"] = rec.numpy()
    dst = synthetic.make_dataset('traj', seed=3, realistic_std=True)
    mt, _ = build_ref_trajnet(ref, seed=2, control=False)
    mt.dataset, mt.device = dst, 'cpu'
    clean_cl = x[:, :, 0].permute(0, 2, 1).contiguous()
    traj_rec = torch.cat([clean_cl[..., 0:1], clean_cl[..., 2:4], clean_cl[..., 6:7], clean_cl[..., 7:13],
                          clean_cl[..., 16:19]], dim=-1) + 0.05 * torch.randn(2, 24, 13, generator=g)
    ld = mt.compute_losses_with_smpl({'motion_repr_clean': clean_cl}, traj_rec, smplx_model=body)
    out["traj_loss_names"] = np.array(list(ld.keys()))
    out["traj_loss_values"] = np.array([float(v) for v in ld.values()], dtype=np.float64)
    out["traj_loss_rec"] = traj_rec.numpy()
    # (d) 2-D reprojection guidance (autograd through the reference code + stub body)
    B, T = 2, 24
    cam2world = torch.eye(4)
    ang = 0.3
    cam2world[:3, :3] = torch.tensor([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]]).float() @ \
        torch.tensor([[1., 0, 0], [0, 0, 1], [0, -1, 0]])
    cam2world[:3, 3] = torch.tensor([0.3, -4.0, 1.2])
    ds.cam_R, ds.cam_t = cam2world[:3, :3].reshape(3, 3).float(), cam2world[:3, 3].reshape(1, 3).float()
    tm = torch.eye(4).repeat(B, 1, 1)
    for b in range(B):
        a = 0.4 * (b + 1)
        tm[b, :3, :3] = torch.tensor([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]).float()
        tm[b, :3, 3] = torch.tensor([0.1 * b, -0.2, 0.05])
    batch = {'x_t': x, 'transf_matrix': tm.float(), 'focal_length': torch.tensor([[1060.0, 1058.0]]).repeat(B, 1),
             'camera_center': torch.tensor([[951.0, 536.0]]).repeat(B, 1)}
    kp = torch.zeros(B, T + 2, 22, 3)
    kp[..., 0] = 951.0 + 300.0 * torch.randn(B, T + 2, 22, generator=g)
    kp[..., 1] = 536.0 + 200.0 * torch.randn(B, T + 2, 22, generator=g)
    kp[..., 2] = (torch.rand(B, T + 2, 22, generator=g) > 0.3).float() * torch.rand(B, T + 2, 22, generator=g)
    batch['keypoints_2d'] = kp
    gr = mp.guide_2d_projection_with_smpl(batch, {'pred_xstart': x}, None, compute_grad='x_0')
    out["proj_grad"] = gr.detach().numpy()
    out["proj_cam_R"], out["proj_cam_t"] = ds.cam_R.numpy(), ds.cam_t.numpy()
    out["proj_transf"], out["proj_focal"], out["proj_center"] = tm.numpy(), batch['focal_length'].numpy(), batch['camera_center'].numpy()
    out["proj_kp"] = kp.numpy()
    np.savez_compressed(os.path.join(OUT, "glue.npz"), **out)
    print("glue.npz  proj grad absmax", float(gr.abs().max()), " nan-repair traj finite:", bool(np.isfinite(out["nan_traj22"]).all()))


POSE_RESPACING = "12" + ",0" * 19
POSE_RECORDED_STEPS = (6, 5, 1, 0)
# Twelve [B, 294, 1, frames - 1] float32 states are stored: 32 frames keep the fixture under 1 MB.
PIPELINE_FRAMES = 32


def gen_pipeline(ref):
    """BASELINE config 4 in miniature, driven through the UNMODIFIED reference: the call sequence of
    test_amass_full.py:231-384 (TrajNet -> host glue -> PoseNet with in-loop skating guidance, 2 rounds, round 2 through
    TrajControl) on 2 clips x 32 frames with 10-step TrajNet and 12-step PoseNet schedules (every PoseNet step guided)."""
    get_repr_smplx = ref.mr.get_repr_smplx
    out = {}
    B, Tn_steps, Pn_steps, rounds, frames = 2, 10, 12, 2, PIPELINE_FRAMES
    ds_pose = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    ds_traj = synthetic.make_dataset('traj', seed=3, realistic_std=True)
    body = _StubBody()
    mp, _ = build_ref_posenet(ref, seed=1)
    mp.dataset, mp.device = ds_pose, 'cpu'
    mt, _ = build_ref_trajnet(ref, seed=2, control=False)
    mc, _ = build_ref_trajnet(ref, seed=4, control=True)
    args = argparse.Namespace(noise_schedule='cosine', sigma_small=True)
    mk = ref.model_util.create_gaussian_diffusion
    # PoseNet: the last 50 steps of the 1000-step schedule thinned to 12 (respacing "12,0,...,0" over 20 sections of 50),
    # i.e. the regime the guidance weights were tuned for (posterior variance ~1e-3..1e-5); every step index is <= 50, so
    # every step is guided
    dp = mk(args, gd=ref.gdp, return_class=ref.respace.SpacedDiffusionPoseNet, num_diffusion_timesteps=1000,
            timestep_respacing=POSE_RESPACING, device='cpu')
    dt = mk(args, gd=ref.gdt, return_class=ref.respace.SpacedDiffusionTrajNet, num_diffusion_timesteps=Tn_steps, device='cpu')
    dc = mk(args, gd=ref.gdt, return_class=ref.respace.SpacedDiffusionTrajNet, num_diffusion_timesteps=Tn_steps, device='cpu')
    pose, traj = synthetic.pipeline_batches(B, 71, ds_pose, frames=frames)
    tfd, pfd = ds_traj.traj_feat_dim, ds_traj.pose_feat_dim
    val_pose = None
    with _patched_th(ref.gdp, 72), _patched_th(ref.gdt, 73):
        for it in range(rounds):
            shape = list(traj['motion_repr_clean'][:, :, 0:tfd].shape)
            if it == 0:
                _, val_traj = dt.eval_losses(model=mt, batch=traj, shape=shape, progress=False, clip_denoised=False,
                                             timestep_respacing='', cond_fn_with_grad=True, compute_loss=False, smplx_model=body)
            else:
                traj['control_cond'] = torch.zeros([shape[0], shape[1], pfd])
                traj['control_cond'][:, 0:-1] = val_pose[:, :, 0].permute(0, 2, 1)[:, :, -pfd:]
                traj['control_cond'][:, -1] = traj['control_cond'][:, -2].clone()
                _, val_traj = dc.eval_losses(model=mc, batch=traj, shape=shape, progress=False, clip_denoised=False,
                                             timestep_respacing='', cond_fn_with_grad=True, compute_loss=False, smplx_model=body)
            comp = traj['motion_repr_clean'].clone()
            comp[..., 0], comp[..., 2:4], comp[..., 6] = val_traj[..., 0], val_traj[..., 1:3], val_traj[..., 3]
            comp[..., 7:13], comp[..., 16:19] = val_traj[..., 4:10], val_traj[..., 10:13]
            if it == 0:
                traj['motion_repr_noisy'] = comp
            full = comp.detach().numpy() * ds_traj.Std + ds_traj.Mean
            rep = _rep_dict(torch.from_numpy(full))
            joints, _ = ref.mr.recover_from_repr_smpl(rep, recover_mode='smplx_params', smplx_model=_VertsBody(body), return_verts=True)
            joints = joints.detach().numpy()
            rows = []
            for i in range(B):
                go = ref.kt.rotation_matrix_to_angle_axis(ref.quat.rot6d_to_rotmat(rep['smplx_rot_6d'][i]))
                bp = ref.kt.rotation_matrix_to_angle_axis(ref.quat.rot6d_to_rotmat(rep['smplx_body_pose_6d'][i].reshape(-1, 6)))
                d = get_repr_smplx(positions=joints[i], smplx_params_dict={
                    'transl': rep['smplx_trans'][i].numpy(), 'global_orient': go.numpy(),
                    'body_pose': bp.reshape(-1, 63).numpy(), 'betas': rep['smplx_betas'][i].numpy()}, feet_vel_thre=5e-5)
                row = np.concatenate([d[k] for k in ko.REPR_LIST], axis=-1)
                rows.append(((row - ds_pose.Mean) / ds_pose.Std)[:, 0:22])
            traj_full = torch.tensor(np.asarray(rows))
            if it == 0:
                pose['motion_repr_noisy'] = pose['motion_repr_noisy'][:, 0:-1]
                pose['motion_repr_clean'] = pose['motion_repr_clean'][:, 0:-1]
            pose['cond'] = pose['motion_repr_noisy'].clone()  # input_noise, iter2_cond_noisy_pose
            pose['cond'][:, :, 0:22] = traj_full
            ids = np.asarray([1, 2, 4, 5, 7, 8, 10, 11])      # mask_scheme 'lower', applied in every round
            for k in range(3):
                pose['cond'][:, :, 22 + ids * 3 + k] = 0.
                pose['cond'][:, :, 22 + 66 + ids * 3 + k] = 0.
            for k in range(6):
                pose['cond'][:, :, 22 + 132 + (ids - 1) * 6 + k] = 0.
            pose['cond'][:, :, -4:] = 0.
            pose['cond'] = torch.permute(pose['cond'], (0, 2, 1)).unsqueeze(-2)
            if it == 0:
                pose['motion_repr_clean'] = torch.permute(pose['motion_repr_clean'], (0, 2, 1)).unsqueeze(-2)
            # The guided chain is chaotic at this batch size (3e6-weighted gradient of a hard-masked mean over only 2 clips:
            # |x_t| reaches 1e3 and a 1e-6 perturbation grows to O(1) within three steps), so the states entering steps
            # 6, 5, 1 and 0 are recorded for teacher-forced comparison of single guided steps and of the final output.
            seen = {}
            orig = dp.p_sample_with_grad

            def recording(model, batch, x, t, **kw):
                seen[int(t[0])] = x.detach().clone()
                return orig(model, batch, x, t, **kw)

            dp.p_sample_with_grad = recording
            _, val_pose = dp.eval_losses(model=mp, batch=pose, shape=list(pose['motion_repr_clean'].shape), progress=False,
                                         clip_denoised=False, timestep_respacing='', cond_fn_with_grad=True, early_stop=False,
                                         compute_loss=False, grad_type='amass', smplx_model=body)
            dp.p_sample_with_grad = orig
            for i in POSE_RECORDED_STEPS:
                out[f"r{it}_xt{i}"] = seen[i].numpy()
            out[f"r{it}_val_traj"] = val_traj.detach().numpy()
            out[f"r{it}_traj_full"] = traj_full.numpy().astype(np.float32)
            out[f"r{it}_cond"] = pose['cond'].detach().numpy()
            out[f"r{it}_val_pose"] = val_pose.detach().numpy()
            print(f"pipeline round {it}: |val_traj| {float(val_traj.abs().max()):.3f} |val_pose| {float(val_pose.abs().max()):.3f}")
    out["meta"] = np.array([B, Tn_steps, Pn_steps, rounds, 71, 72, 73, frames])
    np.savez_compressed(os.path.join(OUT, "pipeline.npz"), **out)
    print("pipeline.npz")


class _VertsBody(nn.Module):
    """The driver asks for vertices (return_verts=True) and discards them; hand back a placeholder of the right shape."""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner

    def forward(self, **kw):
        o = self.inner(**kw)
        o.vertices = torch.zeros(o.joints.shape[0], 10475, 3)
        return o


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    ref = import_reference()
    which = sys.argv[1:] or ["schedules", "posenet", "trajnet", "sampling", "kinematics", "glue", "pipeline"]
    for w in which:
        {"schedules": gen_schedules, "posenet": gen_posenet, "trajnet": gen_trajnet, "sampling": gen_sampling,
         "kinematics": gen_kinematics, "glue": gen_glue, "pipeline": gen_pipeline}[w](ref)
