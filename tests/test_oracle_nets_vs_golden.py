"""Pin the oracle's learned-prior restatement (oracle/nets.py) against outputs of the executed reference networks
(tests/golden/nets.npz: reference modules with the seeded stand-in weights, injected latents).  CPU only."""
import numpy as np
import pytest
import torch

from helpers import load_golden
from glamr_b200.synthetic_nets import make_prior_states
from oracle.nets import MotionTrajJoint
from oracle.smpl import OracleSMPL

NETS_CASES = ['b3_t75', 'b1_t300', 'b2_t40']


@pytest.fixture(scope='module')
def joint_model(smpl_assets):
    st_m, st_t = make_prior_states(1234)
    return MotionTrajJoint(st_m, st_t, OracleSMPL(smpl_assets))


@pytest.mark.parametrize('tag', NETS_CASES)
def test_motion_traj_inference_matches_reference(tag, joint_model):
    g = load_golden('nets')
    batch = {k: torch.tensor(g[f'{tag}/in/{k}']) for k in ['in_body_pose', 'frame_mask', 'in_motion_latent', 'in_traj_latent']}
    out = joint_model.inference(batch, sample_num=1)
    for k, tol in [('infer_out_body_pose', 2e-5), ('infer_out_local_traj_tp', 2e-5), ('infer_out_orient', 1e-4), ('infer_out_trans', 1e-4),
                   ('infer_out_pose', 1e-4)]:
        np.testing.assert_allclose(out[k].numpy(), g[f'{tag}/{k}'], atol=tol, err_msg=f'{tag} {k}')


def test_c3_shape_matches_reference(joint_model, smpl_assets):
    """BASELINE.json configs[2] shape: 64 x 120 with frames 40-69 masked.  Four whole sequences element-wise in float32; all 64
    through per-sequence sums, in float64 for every output (tests/golden/nets_c3_f64.npz: the reference run in float64).  The
    float32 sums of the translation are not compared: it integrates a heading that reaches a few hundred radians over 120
    frames (seeded stand-in weights), where one float32 ulp is 3e-5 rad, so its float32 sums change with the host's
    thread count and SIMD width by more than 1e-5."""
    from helpers import C3_ROWS, c3_prior_inputs
    g = load_golden('nets')
    out = joint_model.inference(c3_prior_inputs(), sample_num=1)
    sel = torch.tensor(C3_ROWS)
    for k, bdim, tol in [('infer_out_body_pose', 0, 2e-5), ('infer_out_local_traj_tp', 1, 2e-5), ('infer_out_trans', 0, 1e-4), ('infer_out_orient', 0, 1e-4)]:
        np.testing.assert_allclose(out[k].index_select(bdim, sel).numpy(), g[f'c3_b64_t120/{k}'], atol=tol, err_msg=k)
        red = [d for d in range(out[k].dim()) if d != bdim]
        if k != 'infer_out_trans':
            np.testing.assert_allclose(out[k].double().abs().sum(dim=red).numpy(), g[f'c3_b64_t120/{k}/abs_sum'], rtol=1e-5, err_msg=k)
    st_m, st_t = make_prior_states(1234)
    model64 = MotionTrajJoint(st_m, st_t, OracleSMPL(smpl_assets, dtype=torch.float64))
    model64.mfiller.double()
    model64.traj_predictor.double()
    g64 = load_golden('nets_c3_f64')
    out = model64.inference({k: v.double() if v.is_floating_point() else v for k, v in c3_prior_inputs().items()}, sample_num=1)
    for k, bdim in [('infer_out_body_pose', 0), ('infer_out_local_traj_tp', 1), ('infer_out_trans', 0), ('infer_out_orient', 0)]:
        assert out[k].dtype == torch.float64, k
        red = [d for d in range(out[k].dim()) if d != bdim]
        np.testing.assert_allclose(out[k].abs().sum(dim=red).numpy(), g64[f'c3_b64_t120/{k}/abs_sum'], rtol=1e-5, err_msg=k + ' (float64)')
