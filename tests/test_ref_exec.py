"""Parity against vectors produced by EXECUTING THE REFERENCE'S OWN SOURCE (tests/golden/ref_exec_v1.npz and the wider sweeps in
tests/golden/ref_sweeps_v1.npz, made by tests/golden/make_ref_exec_golden.py from the reference's src/... over the numpy TensorFlow
stand-in in oracle/ref_exec/; the sweeps' seeded inputs are rebuilt here from tests/golden/sweep_cases.py).

What these vectors pin: everything the reference authored for the path -- op order, indices, reshapes, the variable names the
graph creates and restores from the checkpoint, the IEF / delta-head wiring, the 14-key fetch dict, the sliding window,
process_image, the eval metrics.  What they do not pin: TensorFlow's own kernels and the tf.contrib layers (slim
resnet_v2_50, group_norm, ...), which the stand-in restates from their published definitions ([TF-ext]).

CPU: the oracle (oracle/*.py) reproduces them -> the restatement follows the reference's source.
GPU: the CUDA path reproduces them through the drop-in surface (src.evaluation.tester.Tester etc.), no oracle involved.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, 'golden', 'ref_exec_v1.npz')
SWEEPS = os.path.join(HERE, 'golden', 'ref_sweeps_v1.npz')
REFERENCE = os.environ.get('HD_REFERENCE_ROOT', '')        # a checkout of the reference, for the one test that re-executes it
REL = 1e-4                     # BASELINE.json north_star tolerance for the CUDA path
REL_ORACLE = 2e-5              # float32 oracle vs float32 stand-in execution: rounding-order differences only
KEYS = tuple(a + b for b in ('', '_delta') for a in ('cams', 'joints', 'kps', 'poses', 'shapes', 'verts', 'omegas'))
SMPL_VARS = {'v_template', 'shapedirs', 'J_regressor', 'posedirs', 'lbs_weights', 'cocoplus_regressor'}


def rel_err(a, b):
    b = np.asarray(b, np.float64)
    a = np.asarray(a, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-12))


def _golden_module(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location('_golden_' + name, os.path.join(HERE, 'golden', name + '.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


SC = _golden_module('sweep_cases')


@pytest.fixture(scope='module')
def gold():
    with np.load(GOLD) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope='module')
def sweeps():
    with np.load(SWEEPS) as z:
        return {k: z[k] for k in z.files}


def _smpl_inputs(gold):
    from human_dynamics_b200 import synthetic
    beta, theta = synthetic.make_smpl_inputs(5, seed=12)
    theta[0] = 0
    return beta, theta, gold['smpl_cam']


def _tester_images():
    from human_dynamics_b200 import synthetic
    return synthetic.make_images(40, seed=21, size=224).reshape(2, 20, 224, 224, 3)


def _sub(v, k, ids):
    """verts tensors are stored at 130 sampled vertices."""
    if k == 'verts':
        return v[:, :, ids]
    if k == 'verts_delta':
        return v[:, :, :, ids]
    return v


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: the oracle restatement follows the reference's source
# ---------------------------------------------------------------------------------------------------------------------------
def test_oracle_smpl_matches_reference_source(gold, smpl_model):
    from oracle import smpl_ref
    beta, theta, cam = _smpl_inputs(gold)
    ids = gold['vert_ids']
    s = smpl_ref.SMPLRef(smpl_model)
    v, j, Rs = s(beta, theta, get_skin=True)
    assert rel_err(v[:, ids], gold['smpl_verts']) < REL_ORACLE
    assert rel_err(v.astype(np.float64).sum(axis=1), gold['smpl_verts_sum']) < REL_ORACLE       # all 6890 vertices, as a checksum
    assert rel_err(j, gold['smpl_joints']) < REL_ORACLE
    assert rel_err(Rs, gold['smpl_Rs']) < REL_ORACLE
    assert rel_err(s.J_transformed, gold['smpl_Jtr']) < REL_ORACLE
    assert rel_err(smpl_ref.batch_orth_proj_idrot(j, cam), gold['smpl_kps']) < REL_ORACLE
    assert np.array_equal(np.asarray(s.parents, np.int64), gold['smpl_parents'].astype(np.int64))   # kintree cast, batch_smpl.py:66
    lsp = smpl_ref.SMPLRef(smpl_model, joint_type='lsp')(beta, theta)
    assert rel_err(lsp, gold['smpl_joints_lsp']) < REL_ORACLE
    # helpers
    R = smpl_ref.batch_rodrigues(gold['lbs_aa'])
    assert rel_err(R, gold['lbs_rodrigues']) < REL_ORACLE
    aa = smpl_ref.batch_rot2aa(gold['lbs_rodrigues'])
    ok = np.isfinite(gold['lbs_rot2aa']).all(axis=1)
    assert ok.sum() >= 62 and np.array_equal(np.isfinite(aa).all(axis=1), ok)      # theta = 0 is 0/0 = NaN in the reference too
    far = np.linalg.norm(gold['lbs_rot2aa'][ok], axis=1) < 3.0                     # acos near pi amplifies float32 rounding
    assert np.abs(aa[ok][far] - gold['lbs_rot2aa'][ok][far]).max() < 2e-4
    for rb in (0, 1):
        nj, A = smpl_ref.batch_global_rigid_transformation(gold['smpl_Rs'][:4], gold['lbs_fk_Js'], s.parents, rotate_base=bool(rb))
        assert rel_err(nj, gold['lbs_fk_newJ_rb%d' % rb]) < REL_ORACLE
        assert rel_err(A, gold['lbs_fk_A_rb%d' % rb]) < REL_ORACLE


def test_oracle_networks_match_reference_source(gold, weights):
    from human_dynamics_b200 import synthetic
    from oracle import nets_ref
    img = synthetic.make_images(3, seed=41, size=64)
    phi = nets_ref.encoder_resnet(img, weights).numpy()
    assert rel_err(phi, gold['resnet64_phi']) < REL_ORACLE
    rng = np.random.RandomState(42)
    x = rng.normal(0, 1, size=(2, 20, 2048)).astype(np.float32)
    for k, y in (('fmovie_out', nets_ref.az_fc2_groupnorm(torch.from_numpy(x), weights, 3).numpy()),
                 ('fc2res_out', nets_ref.fc2_res(torch.from_numpy(x), weights).numpy())):
        assert rel_err(y[..., ::16], gold[k]) < REL_ORACLE, k                                 # stored at every 16th channel
        assert rel_err(SC.checksum(y, lead=2), gold[k + '_proj']) < REL_ORACLE, k           # + checksums of all 2048
    B, T = 2, 5
    feats = rng.normal(0, 1, size=(B, T, 2048)).astype(np.float32)
    omega_mean = np.tile(np.asarray(weights['mean_param'], np.float32).reshape(1, 85), (B * T, 1))
    om, deltas = nets_ref.batch_pred_omega(torch.from_numpy(feats), B, weights, 85, omega_mean, T, 'single_view_ief', [0, -5, 5],
                                           use_delta_from_pred=True, use_optcam=True)
    assert rel_err(om.numpy(), gold['ief_omega']) < REL_ORACLE
    assert sorted(deltas.keys()) == [-5, 5]
    for dt in (-5, 5):
        assert rel_err(deltas[dt].numpy(), gold['ief_delta_%d' % dt]) < REL_ORACLE


def test_variable_names_the_reference_graph_creates(gold, weights):
    """SURVEY A.6: the weight dict / checkpoint keys of this repo are exactly the variables the reference's graph creates and
    restores (tester.py:92-116,163-167) -- nothing missing, nothing extra except the SMPL tf.Variables."""
    restored = set(str(n) for n in gold['tester_restored_var_names'])
    mine = set(k for k in weights if not k.startswith('fc2_res/'))
    assert mine <= restored, sorted(mine - restored)[:5]
    assert restored - mine == SMPL_VARS, sorted(restored - mine - SMPL_VARS)[:5]
    every = set(str(n) for n in gold['all_var_names'])                 # models.py functions incl. fc2_res
    assert set(weights) - {'mean_param'} <= every
    from human_dynamics_b200 import nets
    assert nets.BN_EPS == 1e-5 and nets.GN_EPS == 1e-6 and nets.GN_GROUPS == 32


@pytest.mark.timeout(900)
def test_oracle_full_tester_matches_reference_source(gold, weights, smpl_model):
    """Tester.__init__ + build_test_model + predict of the reference, B=2, T=20, 224x224, vs oracle.nets_ref.hmmr_predict."""
    from oracle import nets_ref
    img = _tester_images()
    ids = gold['vert_ids']
    r = nets_ref.hmmr_predict(img, weights, smpl_model)
    for k in KEYS:
        assert rel_err(_sub(r[k], k, ids), gold['tester_' + k]) < 3e-5, k
    assert rel_err(r['verts'].astype(np.float64).sum(axis=2), gold['tester_verts_sum']) < 3e-5
    # the delta heads start from the main prediction and report [1,0,0] cams in `omegas_delta` but are projected with the
    # main camera (tester.py:205-214, omega.py:322-327): visible in the reference's own output
    assert np.array_equal(gold['tester_omegas_delta'][..., 0], np.ones_like(gold['tester_omegas_delta'][..., 0]))
    assert np.array_equal(gold['tester_cams_delta'][:, :, 0], gold['tester_cams'])
    rh = nets_ref.hmmr_predict(img[:1, :4], weights, smpl_model, pred_mode='hal')
    assert rel_err(rh['omegas'], gold['hal_omegas']) < 3e-5 and rel_err(rh['omegas_delta'], gold['hal_omegas_delta']) < 3e-5
    assert rel_err(rh['kps'], gold['hal_kps']) < 3e-5


def _three_delta_inputs():
    from human_dynamics_b200 import synthetic
    w = synthetic.make_synthetic_weights(seed=9, delta_t_values=(-5, 5, 10))
    img = synthetic.make_images(4, seed=23, size=224).reshape(1, 4, 224, 224, 3)
    return w, img


def test_oracle_three_delta_heads_match_reference_source(gold, smpl_model):
    """config.delta_t_values = ['10', '-5', '5'] (unsorted): the reference stacks `_delta` outputs in ascending delta_t order."""
    from oracle import nets_ref
    w, img = _three_delta_inputs()
    r = nets_ref.hmmr_predict(img, w, smpl_model, delta_t_values=(10, -5, 5))
    ids = gold['vert_ids']
    assert rel_err(r['omegas'], gold['three_omegas']) < 3e-5
    assert rel_err(r['omegas_delta'], gold['three_omegas_delta']) < 3e-5
    assert rel_err(r['kps_delta'], gold['three_kps_delta']) < 3e-5
    assert rel_err(r['verts_delta'][:, :, :, ids], gold['three_verts_delta']) < 3e-5
    d = gold['three_omegas_delta']
    assert not np.allclose(d[:, :, 0], d[:, :, 1]) and not np.allclose(d[:, :, 1], d[:, :, 2])       # three different heads
    names = set(str(n) for n in gold['three_var_names'])
    for sc in ('single_view_ief_past5', 'single_view_ief_future5', 'single_view_ief_future10'):     # models.py:344-347
        assert sc + '/3D_module/fc1/weights' in names
    assert set(k for k in w) <= names


def test_oracle_feature_extractor_matches_reference_source(gold, weights):
    """resnet_extractor.py executed from the reference: 6 frames through a batch-4 placeholder (zero-padded tail, :88-92)."""
    from human_dynamics_b200 import synthetic
    from oracle import nets_ref
    frames = synthetic.make_images(6, seed=61, size=64)
    assert rel_err(nets_ref.encoder_resnet(frames, weights).numpy(), gold['fe_phis']) < REL_ORACLE     # frames are independent
    names = set(str(n) for n in gold['fe_restored_var_names'])
    assert names == set(k for k in weights if k.startswith('resnet_v2_50/'))       # Saver() restores exactly the ResNet variables


def test_process_image_oracle_matches_reference_source(gold):
    """run_video.py:56-107 executed from the reference (PNG round trip through its imread) vs oracle/preproc_ref.py."""
    sys.path.insert(0, os.path.join(HERE, 'golden'))
    try:
        from preproc_cases import CASES, frame
    finally:
        sys.path.pop(0)
    from oracle import preproc_ref
    assert np.array_equal(np.array(CASES, np.float64), gold['pi_cases'])
    for i, (H, W, cx, cy, s) in enumerate(CASES):
        r = preproc_ref.process_image(frame(i, H, W), [cx, cy, s])
        meta = np.array(list(r['center']) + list(r['start_pt']) + list(r['im_shape']), np.int64)
        assert np.array_equal(meta, gold['pi_meta_%d' % i]), i
        assert np.abs(r['image'][::7, ::7].astype(np.float32) - gold['pi_img_%d' % i]).max() < 1e-6, i


def test_eval_util_dropin_matches_reference_source(gold):
    """src/evaluation/eval_util.py of this repo vs the reference's module run on the same seeded inputs."""
    import src.evaluation.eval_util as E
    gt, pr, vis = gold['ev_gt'], gold['ev_pr'], gold['ev_vis']
    assert np.allclose(E.compute_accel(gt), gold['ev_accel'], rtol=1e-10, atol=1e-12)
    assert np.allclose(E.compute_error_accel(gt, pr), gold['ev_error_accel'], rtol=1e-10, atol=1e-12)
    assert np.allclose(E.compute_error_accel(gt, pr, vis), gold['ev_error_accel_vis'], rtol=1e-10, atol=1e-12)
    e, pa = E.compute_error_3d(gt, pr)
    assert np.allclose(e, gold['ev_mpjpe'], rtol=1e-9) and np.allclose(pa, gold['ev_pampjpe'], rtol=1e-7)
    assert np.allclose(E.compute_similarity_transform(pr[0], gt[0]), gold['ev_similarity'], atol=1e-9)
    assert np.allclose(E.align_by_pelvis(gt[0]), gold['ev_align_pelvis'], atol=1e-12)
    assert np.allclose(E.compute_error_verts(gold['ev_vg'], gold['ev_vp']), gold['ev_error_verts'], rtol=1e-10)
    ek, epa, pck = E.compute_error_kp(gold['ev_kg'], gold['ev_kp'])
    assert np.allclose(ek, gold['ev_error_kp'], rtol=1e-10) and np.allclose(epa, gold['ev_error_kp_pa'], rtol=1e-9)
    assert np.allclose(pck, gold['ev_pck'])
    al, cam = E.compute_opt_cam_with_vis(got=gold['ev_kp'][0], want=gold['ev_kg'][0, :, :2], vis=gold['ev_kg'][0, :, 2].astype(bool))
    assert np.allclose(al, gold['ev_optcam_aligned'], atol=1e-10) and np.allclose(cam, gold['ev_optcam_cam'], atol=1e-10)
    Rm = E.axis_angle_to_rot_mat(gold['ev_aa'])
    assert np.allclose(Rm, gold['ev_aa2rot'], atol=1e-9)
    assert np.allclose(E.rot_mat_to_axis_angle(Rm), gold['ev_rot2aa'], atol=1e-9)


@pytest.mark.timeout(600)
def test_fixture_is_reproducible_from_the_reference_tree(gold, tmp_path):
    """The cheap sections of the generator (SMPL path, process_image, eval metrics), executed from the reference's source again in a run
    of their own (`make_ref_exec_golden.py regen`, stored as tests/golden/ref_exec_regen_v1.npz), agree with the committed fixture: the
    fixture really is what the reference's source produces.  With HD_REFERENCE_ROOT naming a reference checkout the regeneration is
    also repeated live, in a fresh interpreter, and compared the same way."""
    runs = [os.path.join(HERE, 'golden', 'ref_exec_regen_v1.npz')]
    if REFERENCE:
        runs.append(str(tmp_path / 'regen.npz'))
        env = dict(os.environ)
        env.pop('PYTHONPATH', None)
        subprocess.check_call([sys.executable, '-W', 'ignore', os.path.join(HERE, 'golden', 'make_ref_exec_golden.py'), 'regen', runs[-1]],
                              cwd=str(tmp_path), env=env)
    for path in runs:
        with np.load(path) as z:
            assert len(z.files) > 40
            for k in z.files:
                a, b = z[k], gold[k]
                assert a.shape == b.shape and a.dtype == b.dtype, k
                if a.dtype.kind == 'f':
                    assert np.allclose(a, b, rtol=1e-6, atol=1e-7, equal_nan=True), k
                else:
                    assert np.array_equal(a, b), k


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: wider sweeps through the reference's own source (tests/golden/ref_sweeps_v1.npz) vs this repo
# ---------------------------------------------------------------------------------------------------------------------------
def test_eval_metrics_random_sweep_against_the_reference_tree(sweeps):
    """24 random cases (incl. mirrored point sets, where the similarity transform needs the reflection fix, and sparse visibility) through
    the reference's own eval_util.py vs the drop-in src/evaluation/eval_util.py."""
    import src.evaluation.eval_util as E
    z = sweeps
    for i, (gt, pr, vis, kg, kp) in enumerate(SC.eval_sweep()):
        e, pa = E.compute_error_3d(gt, pr)
        assert np.allclose(e, z['ev_e'][i], rtol=1e-9) and np.allclose(pa, z['ev_pa'][i], rtol=1e-6, atol=1e-9), i
        assert np.allclose(E.compute_similarity_transform(pr[0], gt[0]), z['ev_sim'][i], atol=1e-8), i
        assert np.allclose(E.compute_error_accel(gt, pr, vis), z['ev_acc_%d' % i], rtol=1e-9, atol=1e-12), i
        ek, epa, pck = E.compute_error_kp(kg, kp)
        for a, b in ((ek, z['ev_ek'][i]), (epa, z['ev_epa'][i]), (pck, z['ev_pck'][i])):
            assert np.allclose(np.asarray(a, np.float64), b, rtol=1e-8, atol=1e-10, equal_nan=True), i
        assert np.allclose(E.compute_error_verts(gt, pr), z['ev_verts'][i], rtol=1e-9), i


def test_sliding_window_arithmetic_equals_the_reference_tree(sweeps):
    """tester.py:260-312 (margins, zero-frame padding, stride, which prediction is kept for which frame) executed from the reference
    with `predict` replaced by a probe that returns the frame ids it was shown, vs the drop-in Tester's literal window path with the
    same probe -- for window shapes the network-level fixture does not cover.  (The drop-in's cached-feature path is checked against its
    literal path bit for bit on the GPU.)"""
    from src.evaluation.tester import Tester
    z = sweeps
    for ci, (N, B, T, L) in enumerate(SC.SLIDING_CASES):
        t = Tester.__new__(Tester)
        t.batch_size, t.sequence_length, t.img_size, t.fov = B, T, 2, L * 4 + 1
        t.predict = lambda images, copy=True: {'ids': np.asarray(images)[:, :, 0, 0, 0].copy(), 'two': np.asarray(images)[:, :, :, 0, 0] * 2.0}
        r = t.predict_all_images(SC.sliding_frames(N, np.float32), cache_features=False)
        assert np.array_equal(r['ids'], z['sw_ids_%d' % ci]), (N, B, T, L)
        assert np.array_equal(r['two'], z['sw_two_%d' % ci]), (N, B, T, L)
        assert np.array_equal(z['sw_ids_%d' % ci], np.arange(N) + 1.0)           # every frame is predicted from a window that saw it at full fov


def test_models_other_configuration_against_the_reference_tree(sweeps):
    """A configuration the fixture does not hold -- num_conv_layers=2, B=3, T=7, delta heads (-3, +3), other weights (seed 31)
    -- through the reference's own models.py (az_fc2_groupnorm, batch_pred_omega -> call_hmr_ief -> hmr_ief) vs the oracle."""
    from human_dynamics_b200 import synthetic
    from oracle import nets_ref
    w, x, om0 = SC.other_config_inputs(synthetic)
    strips = nets_ref.az_fc2_groupnorm(torch.from_numpy(x), w, 2)
    om, deltas = nets_ref.batch_pred_omega(strips, 3, w, 85, om0, 7, 'single_view_ief', [3, 0, -3], use_delta_from_pred=True, use_optcam=True)
    z = sweeps
    assert rel_err(strips.numpy()[..., ::16], z['mo_strips']) < REL_ORACLE
    assert rel_err(SC.checksum(strips.numpy(), lead=2), z['mo_strips_proj']) < REL_ORACLE
    assert rel_err(om.numpy(), z['mo_omega']) < REL_ORACLE
    assert rel_err(deltas[-3].numpy(), z['mo_dm3']) < REL_ORACLE and rel_err(deltas[3].numpy(), z['mo_dp3']) < REL_ORACLE
    names = set(str(n) for n in z['mo_names'])
    assert names == set(k for k in w if not k.startswith('resnet_v2_50/') and k != 'mean_param')      # scopes _past3 / _future3, 2 blocks


def test_smpl_random_sweep_against_the_reference_tree(sweeps, smpl_model_dense):
    """48 random poses with LARGE rotations (theta ~ N(0, 1), beta ~ N(0, 2)) and the dense-skinning-weight 19-keypoint model through the
    reference's own SMPL / batch_lbs source (over the stand-in) vs the oracle -- beyond the 5 poses of the fixture.  Vertices are
    stored at 65 sampled vertices plus checksums of all 6890."""
    from human_dynamics_b200 import synthetic
    from oracle import smpl_ref
    m = SC.smpl_sweep_model(synthetic)
    for k in ('v_template', 'shapedirs', 'posedirs', 'weights', 'J_regressor', 'cocoplus_regressor'):
        assert np.array_equal(np.asarray(m[k]), np.asarray(smpl_model_dense[k])), k
    beta, theta, cam = SC.smpl_sweep_inputs()
    o = smpl_ref.SMPLRef(smpl_model_dense)
    v, j, Rs = o(beta, theta, get_skin=True)
    z = sweeps
    assert z['sm_joints'].shape == (48, 19, 3)
    assert rel_err(v[:, SC.VERT_IDS], z['sm_verts']) < REL_ORACLE and rel_err(SC.checksum(v), z['sm_verts_proj']) < REL_ORACLE
    assert rel_err(j, z['sm_joints']) < REL_ORACLE and rel_err(Rs, z['sm_Rs']) < REL_ORACLE
    assert rel_err(o.J_transformed, z['sm_Jtr']) < REL_ORACLE
    assert rel_err(smpl_ref.batch_orth_proj_idrot(j, cam), z['sm_kps']) < REL_ORACLE
    v64 = smpl_ref.SMPLRef(smpl_model_dense, dtype=np.float64)(beta, theta, get_skin=True)[0]
    # the reference's float32 graph itself is this close to float64 truth
    assert rel_err(z['sm_verts'], v64[:, SC.VERT_IDS]) < 1e-5 and rel_err(z['sm_verts_proj'], SC.checksum(v64)) < 1e-5


def test_process_image_random_sweep_against_the_reference_tree(sweeps):
    """40 random (frame size, bbox) cases through the reference's own process_image (run_video.py:56-107, frames handed over as PNG
    files) vs the oracle (32 sampled pixels per crop to 1e-12, checksums of every pixel) and vs the host bookkeeping the CUDA path uses
    (human_dynamics_b200.preprocess.crop_geometry: centre / start point / shape must be equal integers)."""
    from oracle import preproc_ref
    from human_dynamics_b200.preprocess import crop_geometry
    z = sweeps
    for i, (H, W, cx, cy, s, frame) in enumerate(SC.process_image_sweep()):
        assert frame.astype(np.int64).sum() == z['pi_frame_sum'][i], i                 # the same input frame
        r = preproc_ref.process_image(frame, [cx, cy, s])
        meta = np.array(list(r['center']) + list(r['start_pt']) + list(r['im_shape']), np.int64)
        assert np.array_equal(meta, z['pi_meta'][i]), i
        img = np.asarray(r['image'], np.float64)
        assert np.array_equal(img.shape, z['pi_shape'][i]), i
        assert np.abs(SC.pixel_sample(img, i) - z['pi_sample'][i]).max() < 1e-12, i
        assert rel_err(SC.checksum(img[None])[0], z['pi_proj'][i]) < 1e-10, i
        if list(z['pi_meta'][i][4:]) == [224, 224]:            # (ragged crops are refused by the static-shape CUDA path)
            gm = crop_geometry((int(H), int(W)), [cx, cy, s])
            assert list(gm['center']) + list(gm['start_pt']) + list(gm['im_shape']) == list(z['pi_meta'][i]), i


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the CUDA path reproduces the reference-source vectors through the drop-in surface
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cuda_smpl_matches_reference_source(gold, smpl_model):
    from human_dynamics_b200.smpl import SMPLConstants
    import src.tf_smpl.batch_lbs as L
    from src.tf_smpl.projection import batch_orth_proj_idrot
    beta, theta, cam = _smpl_inputs(gold)
    ids = torch.from_numpy(gold['vert_ids']).cuda()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()      # noqa: E731
    m = SMPLConstants(smpl_model, device='cuda')
    o = m.forward(dev(beta), dev(theta), cam=dev(cam))
    assert rel_err(o['verts'][:, ids].cpu().numpy(), gold['smpl_verts']) < REL
    assert rel_err(o['verts'].double().sum(dim=1).cpu().numpy(), gold['smpl_verts_sum']) < REL
    assert rel_err(o['joints'].cpu().numpy(), gold['smpl_joints']) < REL
    assert rel_err(o['Rs'].cpu().numpy(), gold['smpl_Rs']) < REL
    assert rel_err(o['Jtr'].cpu().numpy(), gold['smpl_Jtr']) < REL
    assert rel_err(o['kps'].cpu().numpy(), gold['smpl_kps']) < REL
    assert rel_err(batch_orth_proj_idrot(o['joints'], dev(cam)).cpu().numpy(), gold['smpl_kps']) < REL
    assert rel_err(L.batch_rodrigues(dev(gold['lbs_aa'])).cpu().numpy(), gold['lbs_rodrigues']) < REL
    aa = L.batch_rot2aa(dev(gold['lbs_rodrigues'])).cpu().numpy()
    ok = np.isfinite(gold['lbs_rot2aa']).all(axis=1)
    far = np.linalg.norm(gold['lbs_rot2aa'][ok], axis=1) < 3.0
    assert np.abs(aa[ok][far] - gold['lbs_rot2aa'][ok][far]).max() < 2e-4
    for rb in (0, 1):
        nj, A = L.batch_global_rigid_transformation(dev(gold['smpl_Rs'][:4]), dev(gold['lbs_fk_Js']), gold['smpl_parents'],
                                                    rotate_base=bool(rb))
        assert rel_err(nj.cpu().numpy(), gold['lbs_fk_newJ_rb%d' % rb]) < REL
        assert rel_err(A.cpu().numpy(), gold['lbs_fk_A_rb%d' % rb]) < REL


@pytest.mark.gpu
def test_cuda_tester_matches_reference_source(gold, weights, smpl_model):
    """The reference's Tester (executed from its source) vs this repo's drop-in Tester on the GPU: predict()'s 14 keys at B=2,
    T=20, 224x224, and predict_all_images over 23 frames."""
    from human_dynamics_b200 import synthetic, HMMRConfig
    from src.evaluation.tester import Tester
    ids = gold['vert_ids']
    w = {k: v for k, v in weights.items() if not k.startswith('fc2_res/')}
    t = Tester(HMMRConfig(batch_size=2, sequence_length=20, weights=w, smpl_model=smpl_model, pred_mode='pred'))
    r = t.predict(_tester_images())
    assert sorted(r.keys()) == sorted(KEYS)
    for k in KEYS:
        assert rel_err(_sub(np.asarray(r[k]), k, ids), gold['tester_' + k]) < REL, k
    assert rel_err(np.asarray(r['verts']).astype(np.float64).sum(axis=2), gold['tester_verts_sum']) < REL
    assert rel_err(np.asarray(r['verts_delta']).astype(np.float64).sum(axis=3), gold['tester_verts_delta_sum']) < REL
    ra = t.predict_all_images(synthetic.make_images(23, seed=22, size=224))
    for k in ('omegas', 'kps', 'joints', 'omegas_delta', 'cams_delta'):
        assert rel_err(ra[k], gold['window_' + k]) < REL, k
    assert rel_err(np.asarray(ra['verts'])[:, ids], gold['window_verts']) < REL


@pytest.mark.gpu
def test_cuda_three_delta_heads_match_reference_source(gold, smpl_model):
    from human_dynamics_b200 import HMMRConfig
    from src.evaluation.tester import Tester
    w, img = _three_delta_inputs()
    t = Tester(HMMRConfig(batch_size=1, sequence_length=4, weights=w, smpl_model=smpl_model, pred_mode='pred', delta_t_values=['10', '-5', '5']))
    r = t.predict(img)
    ids = gold['vert_ids']
    assert np.asarray(r['omegas_delta']).shape == (1, 4, 3, 85)
    assert rel_err(r['omegas'], gold['three_omegas']) < REL
    assert rel_err(r['omegas_delta'], gold['three_omegas_delta']) < REL
    assert rel_err(r['kps_delta'], gold['three_kps_delta']) < REL
    assert rel_err(np.asarray(r['verts_delta'])[:, :, :, ids], gold['three_verts_delta']) < REL


@pytest.mark.gpu
def test_cuda_hal_mode_matches_reference_source(gold, weights, smpl_model):
    from human_dynamics_b200 import HMMRConfig
    from src.evaluation.tester import Tester
    t = Tester(HMMRConfig(batch_size=1, sequence_length=4, weights=weights, smpl_model=smpl_model, pred_mode='hal'))
    r = t.predict(_tester_images()[:1, :4])
    assert rel_err(r['omegas'], gold['hal_omegas']) < REL and rel_err(r['omegas_delta'], gold['hal_omegas_delta']) < REL
    assert rel_err(r['kps'], gold['hal_kps']) < REL


@pytest.mark.gpu
def test_cuda_feature_extractor_matches_reference_source(gold, weights):
    """Drop-in src.datasets.resnet_extractor.FeatureExtractor (ragged last batch) vs the reference's, executed from its source."""
    from human_dynamics_b200 import synthetic
    from src.datasets.resnet_extractor import FeatureExtractor
    fe = FeatureExtractor({k: v for k, v in weights.items() if k.startswith('resnet_v2_50/')}, img_size=64, batch_size=4)
    phis = fe.compute_all_phis(synthetic.make_images(6, seed=61, size=64))
    assert phis.shape == (6, 2048) and rel_err(phis, gold['fe_phis']) < REL
    with pytest.raises(ValueError):
        fe.compute_phis(np.zeros((3, 64, 64, 3), np.float32))        # static batch like the TF placeholder


@pytest.mark.gpu
def test_cuda_process_image_matches_reference_source(gold):
    sys.path.insert(0, os.path.join(HERE, 'golden'))
    try:
        from preproc_cases import CASES, frame
    finally:
        sys.path.pop(0)
    from src.evaluation.run_video import process_image
    for i, (H, W, cx, cy, s) in enumerate(CASES):
        r = process_image(frame(i, H, W), np.array([cx, cy, s]))
        img = np.asarray(r['image'].cpu() if hasattr(r['image'], 'cpu') else r['image'])
        meta = np.array(list(r['center']) + list(r['start_pt']) + list(r['im_shape']), np.int64)
        assert np.array_equal(meta, gold['pi_meta_%d' % i]), i
        assert np.abs(img[::7, ::7].astype(np.float32) - gold['pi_img_%d' % i]).max() < 2e-6, i
