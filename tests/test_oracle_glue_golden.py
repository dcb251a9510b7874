"""CPU: pins the glue / pipeline oracles (oracle/glue_oracle.py, oracle/pipeline_oracle.py) to golden vectors produced by the
unmodified reference (tools/gen_golden.py: gen_glue, gen_pipeline -> tests/golden/glue.npz, pipeline.npz)."""
import numpy as np
import torch

from helpers import NoiseTape, TOL, golden
from oracle import glue_oracle as go
from oracle import kinematics_oracle as ko
from oracle import pipeline_oracle
from rohm_b200 import synthetic


PIPELINE_POSE_RESPACING = "12" + ",0" * 19  # tools/gen_golden.py POSE_RESPACING: 12 guided steps inside t < 50


def _plausible(meta):
    B, T, seed, ds_seed = [int(v) for v in meta]
    ds = synthetic.make_dataset('pose', seed=ds_seed, realistic_std=True)
    return synthetic.plausible_motion(B, T, seed, ds), ds


def test_traj_repr_matches_reference_get_repr_smplx():
    g = golden("glue.npz")
    x, ds = _plausible(g["repr_meta"])
    full = x[:, :, 0].permute(0, 2, 1) * torch.from_numpy(ds.Std) + torch.from_numpy(ds.Mean)
    rep = ko.split_repr(full)
    joints = ko.joints_from_smplx(rep, synthetic.smplx_like_model(0)).numpy()
    assert np.abs(joints - g["repr_joints"]).max() < 1e-5
    for i in range(joints.shape[0]):
        aa = ko.rotmat_to_aa(ko.rot6d_to_rotmat(rep['smplx_rot_6d'][i])).numpy()
        r = go.traj_repr_from_joints(g["repr_joints"][i], aa, rep['smplx_trans'][i].numpy())
        assert r.shape == (23, 22)
        assert np.abs(r - g["repr_traj22"][i]).max() < 1e-5, i


def test_traj_repr_nan_repair_matches_reference():
    g = golden("glue.npz")
    x, ds = _plausible(g["repr_meta"])
    full = x[:, :, 0].permute(0, 2, 1) * torch.from_numpy(ds.Std) + torch.from_numpy(ds.Mean)
    transl = ko.split_repr(full)['smplx_trans'][0].numpy()
    r = go.traj_repr_from_joints(g["nan_positions"], g["nan_go"], transl)
    assert np.isfinite(r).all()
    assert np.abs(r - g["nan_traj22"]).max() < 1e-5


def test_rel_traj_joints_match_reference():
    g = golden("glue.npz")
    x, ds = _plausible(g["repr_meta"])
    full = x[:, :, 0].permute(0, 2, 1) * torch.from_numpy(ds.Std) + torch.from_numpy(ds.Mean)
    j = go.joints_from_rel_traj(ko.split_repr(full)).numpy()
    assert np.abs(j - g["rel_traj_joints"]).max() < 1e-5


def test_projection_guidance_matches_reference_autograd():
    g = golden("glue.npz")
    x, ds = _plausible(g["repr_meta"])
    t = lambda k: torch.from_numpy(g[k])
    grad, _ = go.guide_projection(x, torch.from_numpy(ds.Mean), torch.from_numpy(ds.Std), synthetic.smplx_like_model(0),
                                  t("proj_transf"), t("proj_cam_R"), t("proj_cam_t"), t("proj_focal"), t("proj_center"),
                                  t("proj_kp"))
    ref = g["proj_grad"]
    assert np.abs(grad.numpy() - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    assert np.abs(ref[:, 0:22]).max() == 0 and np.abs(ref[:, -4:]).max() == 0 and np.abs(ref).max() > 0


def test_pipeline_oracle_matches_reference_rounds():
    """2 clips x 32 frames, 10-step TrajNet / 12-step guided PoseNet, 2 rounds (round 2 through TrajControl)."""
    from rohm_b200.posenet import PoseNet
    from rohm_b200.trajnet import TrajNet
    g = golden("pipeline.npz")
    B, tn, pn, rounds, s_in, s_pose, s_traj, frames = [int(v) for v in g["meta"]]
    ds_pose = synthetic.make_dataset('pose', seed=3, realistic_std=True)
    ds_traj = synthetic.make_dataset('traj', seed=3, realistic_std=True)
    sd_pose = synthetic.synth_state_dict(PoseNet(dataset=ds_pose, body_feat_dim=294, latent_dim=512, traj_feat_dim=22), 1)
    mk = lambda c: TrajNet(time_dim=32, mid_dim=512, cond_dim=13, traj_feat_dim=13, trajcontrol=c, repr_abs_only=True)
    sd_traj, sd_ctrl = synthetic.synth_state_dict(mk(False), 2), synthetic.synth_state_dict(mk(True), 4)
    pose, traj = synthetic.pipeline_batches(B, s_in, ds_pose, frames=frames)
    res = pipeline_oracle.run_rounds(sd_pose, sd_traj, sd_ctrl, ds_pose, ds_traj, synthetic.smplx_like_model(0), pose, traj,
                                     1000, tn, rounds, NoiseTape(s_pose), NoiseTape(s_traj),
                                     pose_respacing=PIPELINE_POSE_RESPACING, teacher=g, teacher_steps=(6, 1, 0))
    for it in range(rounds):
        err = {k: float(np.abs(res[it][k].numpy() - g[f"r{it}_{k}"]).max()) for k in ("val_traj", "traj_full", "cond", "val_pose")}
        # teacher-forced single steps: x_6 -> x_5, x_1 -> x_0 (guided, |x| up to 1e3: relative bound), x_0 -> output (absolute)
        tf = res[it]['tf']
        e65 = float((tf[6] - torch.from_numpy(g[f"r{it}_xt5"])).abs().max()) / float(np.abs(g[f"r{it}_xt5"]).max())
        e10 = float((tf[1] - torch.from_numpy(g[f"r{it}_xt0"])).abs().max()) / float(np.abs(g[f"r{it}_xt0"]).max())
        e0 = float((tf[0] - torch.from_numpy(g[f"r{it}_val_pose"])).abs().max())
        print(f"round {it}: stages {err} | teacher-forced: step6 rel {e65:.2e}, step1 rel {e10:.2e}, final abs {e0:.2e}")
        assert err["val_traj"] < TOL and err["traj_full"] < TOL and err["cond"] < TOL, (it, err)
        assert e65 < 1e-3 and e10 < 1e-3 and e0 < TOL, (it, e65, e10, e0)
