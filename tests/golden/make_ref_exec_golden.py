"""Generates tests/golden/ref_exec_v1.npz by EXECUTING THE REFERENCE'S OWN SOURCE FILES from /root/reference:

    src/tf_smpl/batch_lbs.py, batch_smpl.py, projection.py      (batch_rodrigues, batch_rot2aa, FK, SMPL.__call__, projection)
    src/models.py                                               (encoder_resnet, az_fc2_groupnorm, fc2_res, batch_pred_omega -> IEF)
    src/omega.py, src/evaluation/tester.py                      (Tester.__init__ / build_test_model / predict / predict_all_images)
    src/datasets/resnet_extractor.py                            (FeatureExtractor: restore + compute_all_phis with a ragged last batch)
    src/evaluation/run_video.py + src/util/common.py            (process_image, resize_img)
    src/evaluation/eval_util.py                                 (metrics)

unmodified, with `import tensorflow` resolving to the numpy stand-in under oracle/ref_exec/stubs (TensorFlow 1.8 has no
wheel for this interpreter and there is no network).  The vectors therefore pin everything the reference authored -- op order,
indices, reshapes, variable scopes, checkpoint-restore by variable name, the 14-key fetch wiring, the sliding window -- while
the TF op definitions themselves (matmul, reshape, ... and the tf.contrib layers incl. slim's resnet_v2_50, marked [TF-ext])
are the stand-in's restatement of their documented semantics, NOT TensorFlow's kernels.  That residue is what "oracle
unpinned" still means for this repo; see oracle/ref_exec/README.md.

Inputs are not stored: they are regenerated from seeds by human_dynamics_b200.synthetic (weights seed 1, SMPL seed 2, ...),
exactly as listed in CASES below; large outputs are stored sub-sampled (130 vertices).

Needs a checkout of the reference, named by HD_REFERENCE_ROOT.  Run from the repo root:
    HD_REFERENCE_ROOT=<reference checkout> python tests/golden/make_ref_exec_golden.py          (about 2 minutes, ~3 GB RAM,
                                                                                               writes ~0.5 GB to a temp dir)
    HD_REFERENCE_ROOT=<reference checkout> python tests/golden/make_ref_exec_golden.py sweeps   (ref_sweeps_v1.npz)
    HD_REFERENCE_ROOT=<reference checkout> python tests/golden/make_ref_exec_golden.py regen    (ref_exec_regen_v1.npz: the cheap
                                                                                               sections again, in a run of their own)
"""
import importlib.util
import os
import pickle
import shutil
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get('HD_REFERENCE_ROOT', '')
STUBS = os.path.join(ROOT, 'oracle', 'ref_exec', 'stubs')
VERT_IDS = np.arange(0, 6890, 53)


def _by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def setup_paths():
    """`src` must resolve to the REFERENCE package (this repo has a drop-in package of the same name), `tensorflow` etc. to
    the stand-ins.  Repo helpers (synthetic inputs, checkpoint writer) are loaded by file path, never through sys.path."""
    if not REF or not os.path.isdir(os.path.join(REF, 'src')):
        raise SystemExit('set HD_REFERENCE_ROOT to a checkout of the reference (got %r)' % REF)
    for p in (ROOT, os.path.join(ROOT, 'tests'), ''):
        while p in sys.path:
            sys.path.remove(p)
    sys.path[:0] = [STUBS, REF]
    for m in [m for m in sys.modules if m == 'src' or m.startswith('src.')]:
        del sys.modules[m]
    for alias, typ in (('int', int), ('float', float)):
        if not hasattr(np, alias):
            setattr(np, alias, typ)   # run_video.py:78 / eval_util.py:241 use the aliases numpy removed in 1.24; same types
    # rendering (neural_renderer, outside the path) is imported at run_video.py's top: satisfy the import only
    stub = types.ModuleType('src.util.render.nmr_renderer')
    stub.VisRenderer = stub.visualize_img = stub.visualize_img_orig = None
    sys.modules['src.util.render.nmr_renderer'] = stub
    syn = _by_path('_hd_synthetic', os.path.join(ROOT, 'human_dynamics_b200', 'synthetic.py'))
    ckpt = _by_path('_hd_tf_checkpoint', os.path.join(ROOT, 'human_dynamics_b200', 'tf_checkpoint.py'))
    return syn, ckpt


def write_smpl_pickle(smpl, path):
    """The official file's structure: dense arrays + scipy-sparse regressors (batch_smpl.py:50,77 call .T.todense())."""
    import scipy.sparse as sp
    dd = dict(smpl)
    dd['J_regressor'] = sp.csc_matrix(smpl['J_regressor'])
    dd['cocoplus_regressor'] = sp.csc_matrix(smpl['cocoplus_regressor'])
    with open(path, 'wb') as f:
        pickle.dump(dd, f, protocol=2)


def smpl_checkpoint_vars(smpl):
    """The SMPL tf.Variables are in GLOBAL_VARIABLES, so Tester.prepare restores them from the checkpoint too
    (tester.py:163-167,110-115): same values as the pickle, under the names batch_smpl.py:34-81 gives them."""
    V = smpl['v_template'].shape[0]
    return {
        'v_template': smpl['v_template'],
        'shapedirs': np.reshape(smpl['shapedirs'], [-1, 10]).T,
        'J_regressor': np.asarray(smpl['J_regressor']).T,
        'posedirs': np.reshape(smpl['posedirs'], [-1, 207]).T,
        'lbs_weights': smpl['weights'],
        'cocoplus_regressor': np.asarray(smpl['cocoplus_regressor']).T,
    }, V


def gen_smpl(out, syn, smpl_pkl):
    import tensorflow as tf
    from src.tf_smpl.batch_smpl import SMPL
    from src.tf_smpl import batch_lbs, projection
    sess = tf.Session()
    beta, theta = syn.make_smpl_inputs(5, seed=12)
    theta[0] = 0
    cam = np.tile(np.array([[0.9, 0.1, -0.2]], np.float32), (5, 1))
    cam[3] = [1.3, -0.4, 0.25]
    s = SMPL(smpl_pkl)
    verts, joints, Rs = s(tf.constant(beta), tf.constant(theta), get_skin=True)
    kps = projection.batch_orth_proj_idrot(joints, tf.constant(cam))
    v, j, R, Jt, k = sess.run([verts, joints, Rs, s.J_transformed, kps])
    out.update(smpl_verts=v[:, VERT_IDS], smpl_joints=j, smpl_Rs=R, smpl_Jtr=Jt, smpl_kps=k, smpl_cam=cam,
               smpl_verts_sum=v.astype(np.float64).sum(axis=1))
    s_lsp = SMPL(smpl_pkl, joint_type='lsp')
    out['smpl_joints_lsp'] = sess.run(s_lsp(tf.constant(beta), tf.constant(theta)))
    # helpers on their own
    rng = np.random.RandomState(31)
    aa = rng.normal(0, 0.8, size=(64, 3)).astype(np.float32)
    aa[0] = 0
    aa[1] = [1e-6, 0, 0]
    aa[2] = [np.pi - 1e-3, 0, 0]
    Rm = batch_lbs.batch_rodrigues(tf.constant(aa))
    out['lbs_aa'] = aa
    out['lbs_rodrigues'] = sess.run(Rm)
    out['lbs_rot2aa'] = sess.run(batch_lbs.batch_rot2aa(Rm))
    Rs4 = tf.constant(R[:4])
    Js = tf.constant(rng.normal(0, 0.3, size=(4, 24, 3)).astype(np.float32))
    out['lbs_fk_Js'] = sess.run(Js)
    for rb in (False, True):
        nj, A = batch_lbs.batch_global_rigid_transformation(Rs4, Js, s.parents, rotate_base=rb)
        nj, A = sess.run([nj, A])
        out['lbs_fk_newJ_rb%d' % rb], out['lbs_fk_A_rb%d' % rb] = nj, A
    out['smpl_parents'] = np.asarray(s.parents)
    tf.reset_default_graph()


def gen_models(out, syn, weights):
    """models.py functions on their own (small shapes), variables assigned by NAME from the TF-keyed weight dict."""
    import tensorflow as tf
    from src import models

    def assign_all():
        for v in tf.global_variables():
            if not v.initialized:
                v.load(weights[v.op_name])

    sess = tf.Session()
    # encoder_resnet on 64x64 frames (models.py:50-77)
    img = syn.make_images(3, seed=41, size=64)
    phi, scope = models.encoder_resnet(tf.constant(img), is_training=False, reuse=False)
    assert scope == 'resnet_v2_50'
    assign_all()
    out['resnet64_phi'] = sess.run(phi)
    out['resnet_var_names'] = np.array(sorted(v.op_name for v in tf.global_variables()))
    # az_fc2_groupnorm (models.py:121-228); 2048-wide outputs are stored at every 16th channel + checksums of all channels
    sc = _by_path('_sweep_cases', os.path.join(ROOT, 'tests', 'golden', 'sweep_cases.py'))
    rng = np.random.RandomState(42)
    x = rng.normal(0, 1, size=(2, 20, 2048)).astype(np.float32)
    y = models.az_fc2_groupnorm(is_training=False, net=tf.constant(x), num_conv_layers=3)
    assign_all()
    y = sess.run(y)
    out['fmovie_out'], out['fmovie_out_proj'] = y[..., ::16], sc.checksum(y, lead=2)
    # fc2_res (models.py:270-296)
    z = models.fc2_res(tf.constant(x))
    assign_all()
    z = sess.run(z)
    out['fc2res_out'], out['fc2res_out_proj'] = z[..., ::16], sc.checksum(z, lead=2)
    # batch_pred_omega -> call_hmr_ief -> hmr_ief -> encoder_fc3_dropout (models.py:233-267,299-415,80-116)
    B, T = 2, 5
    feats = rng.normal(0, 1, size=(B, T, 2048)).astype(np.float32)
    omega_mean = np.tile(np.asarray(weights['mean_param'], np.float32).reshape(1, 85), (B * T, 1))
    om, deltas = models.batch_pred_omega(input_features=tf.constant(feats), batch_size=B, is_training=False, num_output=85,
                                         omega_mean=tf.constant(omega_mean), sequence_length=T, scope='single_view_ief',
                                         predict_delta_keys=[0, -5, 5], use_delta_from_pred=True, use_optcam=True)
    assign_all()
    r = sess.run({'omega': om, 'deltas': deltas})
    out['ief_omega'] = r['omega']
    for dt, v in r['deltas'].items():
        out['ief_delta_%d' % dt] = v
    out['all_var_names'] = np.array(sorted(v.op_name for v in tf.global_variables()))
    tf.reset_default_graph()


def gen_tester(out, syn, ckpt, weights, smpl, tmp):
    import tensorflow as tf
    from src.evaluation.tester import Tester
    from src.omega import OmegasPred
    smpl_pkl = os.path.join(tmp, 'neutral_smpl_with_cocoplus_reg.pkl')
    # initial mean_param (tester.py:118-141): deliberately NOT the checkpoint's value, the restore must win
    mp0 = syn.make_mean_param(seed=77)
    np.savez(os.path.join(tmp, 'neutral_smpl_meanwjoints.npz'), pose=mp0[0, 3:75], shape=mp0[0, 75:])
    smpl_vars, _ = smpl_checkpoint_vars(smpl)
    tensors = {k: np.ascontiguousarray(v, np.float32) for k, v in weights.items()}
    tensors.update({k: np.ascontiguousarray(v, np.float32) for k, v in smpl_vars.items()})
    prefix = os.path.join(tmp, 'model.ckpt-1')
    ckpt.save_checkpoint(prefix, tensors)

    def config(B, T, mode):
        return types.SimpleNamespace(load_path=prefix, batch_size=B, sequence_length=T, pred_mode=mode, num_conv_layers=3,
                                     delta_t_values=['-5', '5'], smpl_model_path=smpl_pkl, num_kps=25)

    B, T = 2, 20
    images = syn.make_images(B * T, seed=21, size=224).reshape(B, T, 224, 224, 3)
    OmegasPred.omega_instances[:] = []
    t = Tester(config(B, T, 'pred'))
    names = sorted(v.op_name for v in t.encoder_vars)
    out['tester_restored_var_names'] = np.array(names)
    missing = sorted(set(weights) - set(names) - set(k for k in weights if k.startswith('fc2_res/')))
    assert not missing, ('weights the reference graph never created', missing[:5])
    r = t.predict(images)
    assert sorted(r.keys()) == sorted(['cams', 'joints', 'kps', 'poses', 'shapes', 'verts', 'omegas'] +
                                      [k + '_delta' for k in ('cams', 'joints', 'kps', 'poses', 'shapes', 'verts', 'omegas')])
    for k, v in r.items():
        v = np.asarray(v)
        if k == 'verts':
            out['tester_verts_sum'] = v.astype(np.float64).sum(axis=2)
            v = v[:, :, VERT_IDS]
        elif k == 'verts_delta':
            out['tester_verts_delta_sum'] = v.astype(np.float64).sum(axis=3)
            v = v[:, :, :, VERT_IDS]
        out['tester_' + k] = v
    # sliding window (tester.py:260-312): 23 frames, B=2, T=20 -> margin 6, 8 good frames per window, 2 passes
    N = 23
    all_images = syn.make_images(N, seed=22, size=224)
    ra = t.predict_all_images(all_images)
    for k in ('omegas', 'kps', 'joints', 'omegas_delta', 'cams_delta'):
        out['window_' + k] = np.asarray(ra[k])
    out['window_verts'] = np.asarray(ra['verts'])[:, VERT_IDS]
    tf.reset_default_graph()
    # hallucinator mode (tester.py:189-190), small batch
    OmegasPred.omega_instances[:] = []
    th = Tester(config(1, 4, 'hal'))
    rh = th.predict(images[:1, :4])
    out['hal_omegas'] = np.asarray(rh['omegas'])
    out['hal_omegas_delta'] = np.asarray(rh['omegas_delta'])
    out['hal_kps'] = np.asarray(rh['kps'])
    OmegasPred.omega_instances[:] = []
    tf.reset_default_graph()


def gen_tester_three_deltas(out, syn, ckpt, smpl, tmp):
    """Tester with three delta heads given in UNSORTED order (config.delta_t_values = ['10', '-5', '5']): the reference stacks the
    `_delta` outputs in ascending delta_t order (`sorted(self.omegas_pred.items())`, tester.py:244) and names the scopes
    `_past5` / `_future5` / `_future10` (models.py:344-347).  B=1, T=4, separate weights (seed 9)."""
    import tensorflow as tf
    from src.evaluation.tester import Tester
    from src.omega import OmegasPred
    tf.reset_default_graph()
    OmegasPred.omega_instances[:] = []
    w = syn.make_synthetic_weights(seed=9, delta_t_values=(-5, 5, 10))
    smpl_pkl = os.path.join(tmp, 'neutral_smpl_with_cocoplus_reg.pkl')
    if not os.path.exists(smpl_pkl):
        write_smpl_pickle(smpl, smpl_pkl)
    mp0 = syn.make_mean_param(seed=77)
    np.savez(os.path.join(tmp, 'neutral_smpl_meanwjoints.npz'), pose=mp0[0, 3:75], shape=mp0[0, 75:])
    smpl_vars, _ = smpl_checkpoint_vars(smpl)
    tensors = {k: np.ascontiguousarray(v, np.float32) for k, v in w.items()}
    tensors.update({k: np.ascontiguousarray(v, np.float32) for k, v in smpl_vars.items()})
    prefix = os.path.join(tmp, 'model3.ckpt-3')
    ckpt.save_checkpoint(prefix, tensors)
    cfg = types.SimpleNamespace(load_path=prefix, batch_size=1, sequence_length=4, pred_mode='pred', num_conv_layers=3,
                                delta_t_values=['10', '-5', '5'], smpl_model_path=smpl_pkl, num_kps=25)
    t = Tester(cfg)
    images = syn.make_images(4, seed=23, size=224).reshape(1, 4, 224, 224, 3)
    r = t.predict(images)
    assert np.asarray(r['omegas_delta']).shape == (1, 4, 3, 85)
    out['three_omegas'] = np.asarray(r['omegas'])
    out['three_omegas_delta'] = np.asarray(r['omegas_delta'])
    out['three_kps_delta'] = np.asarray(r['kps_delta'])
    out['three_verts_delta'] = np.asarray(r['verts_delta'])[:, :, :, VERT_IDS]
    out['three_var_names'] = np.array(sorted(v.op_name for v in t.encoder_vars))
    OmegasPred.omega_instances[:] = []
    tf.reset_default_graph()


def gen_feature_extractor(out, syn, ckpt, weights, tmp):
    """resnet_extractor.py:13-98: placeholder of batch_size frames, Saver() over every variable of the graph, zero-padded last batch."""
    import tensorflow as tf
    from src.datasets.resnet_extractor import FeatureExtractor
    tf.reset_default_graph()
    prefix = os.path.join(tmp, 'resnet.ckpt-7')
    ckpt.save_checkpoint(prefix, {k: np.ascontiguousarray(v, np.float32) for k, v in weights.items() if k.startswith('resnet_v2_50/')})
    fe = FeatureExtractor(prefix, img_size=64, batch_size=4)
    frames = syn.make_images(6, seed=61, size=64)                      # 6 frames, batch 4 -> second batch is 2 frames + 2 zero frames
    out['fe_phis'] = np.asarray(fe.compute_all_phis(frames))
    assert out['fe_phis'].shape == (6, 2048)
    out['fe_restored_var_names'] = np.array(sorted(fe.saver.restored))
    tf.reset_default_graph()


def gen_process_image(out, tmp):
    import cv2
    from src.evaluation.run_video import process_image
    pg = _by_path('_preproc_cases', os.path.join(ROOT, 'tests', 'golden', 'preproc_cases.py'))
    out['pi_cases'] = np.array(pg.CASES, np.float64)
    for i, (H, W, cx, cy, s) in enumerate(pg.CASES):
        path = os.path.join(tmp, 'frame_%d.png' % i)
        cv2.imwrite(path, cv2.cvtColor(pg.frame(i, H, W), cv2.COLOR_RGB2BGR))          # lossless; imread gives the frame back
        r = process_image(path, np.array([cx, cy, s], np.float64))
        assert r['image'].shape == (224, 224, 3), r['image'].shape
        out['pi_img_%d' % i] = r['image'][::7, ::7].astype(np.float32)
        out['pi_meta_%d' % i] = np.array(list(r['center']) + list(r['start_pt']) + list(r['im_shape']), np.int64)


def gen_eval_util(out):
    from src.evaluation import eval_util as E
    rng = np.random.RandomState(51)
    gt = rng.normal(0, 0.3, size=(30, 14, 3))
    pr = gt + rng.normal(0, 0.02, size=gt.shape)
    vis = rng.rand(30) > 0.2
    out['ev_gt'], out['ev_pr'], out['ev_vis'] = gt, pr, vis
    out['ev_accel'] = E.compute_accel(gt)
    out['ev_error_accel'] = E.compute_error_accel(gt, pr)
    out['ev_error_accel_vis'] = E.compute_error_accel(gt, pr, vis)
    e, pa = E.compute_error_3d(gt, pr)
    out['ev_mpjpe'], out['ev_pampjpe'] = np.asarray(e), np.asarray(pa)
    out['ev_similarity'] = E.compute_similarity_transform(pr[0], gt[0])
    out['ev_align_pelvis'] = E.align_by_pelvis(gt[0])
    vg = rng.normal(0, 0.3, size=(4, 200, 3))
    vp = vg + rng.normal(0, 0.01, size=vg.shape)
    out['ev_vg'], out['ev_vp'] = vg, vp
    out['ev_error_verts'] = np.asarray(E.compute_error_verts(vg, vp))
    kg = np.concatenate([rng.rand(6, 19, 2) * 2 - 1, (rng.rand(6, 19, 1) > 0.3).astype(np.float64)], axis=2)
    kp = kg[:, :, :2] + rng.normal(0, 0.03, size=(6, 19, 2))
    out['ev_kg'], out['ev_kp'] = kg, kp
    ek, epa, pck = E.compute_error_kp(kg, kp)
    out['ev_error_kp'], out['ev_error_kp_pa'], out['ev_pck'] = np.asarray(ek, np.float64), np.asarray(epa, np.float64), np.asarray(pck, np.float64)
    aligned, cam = E.compute_opt_cam_with_vis(got=kp[0], want=kg[0, :, :2], vis=kg[0, :, 2].astype(bool))
    out['ev_optcam_aligned'], out['ev_optcam_cam'] = np.asarray(aligned), np.asarray(cam)
    aa = rng.normal(0, 0.7, size=72)
    out['ev_aa'] = aa
    Rm = E.axis_angle_to_rot_mat(aa)
    out['ev_aa2rot'] = np.asarray(Rm)
    out['ev_rot2aa'] = np.asarray(E.rot_mat_to_axis_angle(Rm))


def gen_sweeps(out, syn, tmp):
    """Wider sweeps than the fixture above, stored in ref_sweeps_v1.npz; their inputs come from sweep_cases.py."""
    import cv2
    import tensorflow as tf
    from src import models
    from src.evaluation import eval_util as E
    from src.evaluation.run_video import process_image
    from src.evaluation.tester import Tester
    from src.tf_smpl.batch_smpl import SMPL
    from src.tf_smpl.projection import batch_orth_proj_idrot
    sc = _by_path('_sweep_cases', os.path.join(ROOT, 'tests', 'golden', 'sweep_cases.py'))
    # eval_util.py metrics; per-case results of equal shape are stacked along a first axis of cases
    cases = {}
    for i, (gt, pr, vis, kg, kp) in enumerate(sc.eval_sweep()):
        e, pa = E.compute_error_3d(gt, pr)
        ek, epa, pck = E.compute_error_kp(kg, kp)
        for key, a in (('e', e), ('pa', pa), ('sim', E.compute_similarity_transform(pr[0], gt[0])), ('ek', ek), ('epa', epa), ('pck', pck),
                       ('verts', E.compute_error_verts(gt, pr))):
            cases.setdefault('ev_' + key, []).append(np.asarray(a, np.float64))
        out['ev_acc_%d' % i] = np.asarray(E.compute_error_accel(gt, pr, vis))       # length = number of visible frame triples
    out.update((k, np.stack(v)) for k, v in cases.items())
    # tester.py:260-312 sliding window, `predict` replaced by a probe returning the frame ids it was shown
    for ci, (N, B, T, L) in enumerate(sc.SLIDING_CASES):
        t = Tester.__new__(Tester)
        t.batch_size, t.sequence_length, t.img_size, t.fov = B, T, 2, L * 4 + 1
        t.predict = lambda images: {'ids': np.asarray(images)[:, :, 0, 0, 0].copy(), 'two': np.asarray(images)[:, :, :, 0, 0] * 2.0}
        r = t.predict_all_images(sc.sliding_frames(N, np.float64))
        out['sw_ids_%d' % ci], out['sw_two_%d' % ci] = np.asarray(r['ids']), np.asarray(r['two'])
    # models.py with 2 temporal blocks, B=3, T=7, delta heads (-3, +3)
    tf.reset_default_graph()
    w, x, om0 = sc.other_config_inputs(syn)
    y = models.get_temporal_encoder()(is_training=False, net=tf.constant(x), num_conv_layers=2)
    om, deltas = models.batch_pred_omega(input_features=y, batch_size=3, is_training=False, num_output=85, omega_mean=tf.constant(om0),
                                         sequence_length=7, scope='single_view_ief', predict_delta_keys=[3, 0, -3],
                                         use_delta_from_pred=True, use_optcam=True)
    for v in tf.global_variables():
        v.load(w[v.op_name])
    r = tf.Session().run({'strips': y, 'omega': om, 'dm3': deltas[-3], 'dp3': deltas[3]})
    out['mo_strips'], out['mo_strips_proj'] = r['strips'][..., ::16], sc.checksum(r['strips'], lead=2)
    out['mo_omega'], out['mo_dm3'], out['mo_dp3'] = r['omega'], r['dm3'], r['dp3']
    out['mo_names'] = np.array(sorted(v.op_name for v in tf.global_variables()))
    tf.reset_default_graph()
    # SMPL / batch_lbs with large rotations and the dense-weight 19-keypoint model
    pkl = os.path.join(tmp, 'smpl_dense.pkl')
    write_smpl_pickle(sc.smpl_sweep_model(syn), pkl)
    beta, theta, cam = sc.smpl_sweep_inputs()
    s = SMPL(pkl)
    v, j, R = s(tf.constant(beta), tf.constant(theta), get_skin=True)
    k = batch_orth_proj_idrot(j, tf.constant(cam))
    r = tf.Session().run({'verts': v, 'joints': j, 'Rs': R, 'Jtr': s.J_transformed, 'kps': k})
    out['sm_verts'], out['sm_verts_proj'] = r['verts'][:, sc.VERT_IDS], sc.checksum(r['verts'])
    out['sm_joints'], out['sm_Rs'], out['sm_Jtr'], out['sm_kps'] = r['joints'], r['Rs'], r['Jtr'], r['kps']
    tf.reset_default_graph()
    # run_video.py:56-107 process_image, frames handed over as (lossless) PNG files through its imread; one row per case
    cases = {}
    for i, (H, W, cx, cy, s, frame) in enumerate(sc.process_image_sweep()):
        path = os.path.join(tmp, 'sweep_%d.png' % i)
        cv2.imwrite(path, cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))
        r = process_image(path, np.array([cx, cy, s], np.float64))
        img = np.asarray(r['image'], np.float64)
        for key, a in (('frame_sum', frame.astype(np.int64).sum()), ('shape', img.shape),
                       ('meta', list(r['center']) + list(r['start_pt']) + list(r['im_shape']))):
            cases.setdefault('pi_' + key, []).append(np.asarray(a, np.int64))
        cases.setdefault('pi_sample', []).append(sc.pixel_sample(img, i))
        cases.setdefault('pi_proj', []).append(sc.checksum(img[None])[0])
    out.update((k, np.stack(v)) for k, v in cases.items())


def main():
    syn, ckpt = setup_paths()
    if sys.argv[1:2] == ['regen']:
        # the fixture's cheap sections (SMPL path, process_image, eval metrics) regenerated in a run of their own
        tmp = tempfile.mkdtemp(prefix='ref_regen_')
        out = {}
        try:
            write_smpl_pickle(syn.make_synthetic_smpl(seed=2), os.path.join(tmp, 'smpl.pkl'))
            gen_smpl(out, syn, os.path.join(tmp, 'smpl.pkl'))
            gen_process_image(out, tmp)
            gen_eval_util(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, 'tests', 'golden', 'ref_exec_regen_v1.npz')
        np.savez_compressed(path, **out)
        print('wrote', path, os.path.getsize(path), 'bytes,', len(out), 'arrays')
        return
    if sys.argv[1:] == ['sweeps']:
        tmp = tempfile.mkdtemp(prefix='ref_sweeps_')
        out = {}
        try:
            gen_sweeps(out, syn, tmp)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        path = os.path.join(ROOT, 'tests', 'golden', 'ref_sweeps_v1.npz')
        np.savez_compressed(path, **out)
        print('wrote', path, os.path.getsize(path), 'bytes,', len(out), 'arrays')
        return
    weights = syn.make_synthetic_weights(seed=1, with_hal=True)
    smpl = syn.make_synthetic_smpl(seed=2)
    tmp = tempfile.mkdtemp(prefix='ref_exec_')
    out = {'vert_ids': VERT_IDS}
    path = os.path.join(ROOT, 'tests', 'golden', 'ref_exec_v1.npz')
    only = os.environ.get('HD_REF_EXEC_ONLY')           # e.g. "feature_extractor": re-run one cheap section, keep the rest of the file
    if only:
        with np.load(path) as z:
            out = {k: z[k] for k in z.files}
        try:
            {'feature_extractor': lambda: gen_feature_extractor(out, syn, ckpt, weights, tmp),
             'three_deltas': lambda: gen_tester_three_deltas(out, syn, ckpt, smpl, tmp),
             'process_image': lambda: gen_process_image(out, tmp), 'eval_util': lambda: gen_eval_util(out)}[only]()
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        np.savez_compressed(path, **out)
        print('updated section', only, 'of', path, os.path.getsize(path), 'bytes,', len(out), 'arrays')
        return
    try:
        smpl_pkl = os.path.join(tmp, 'smpl.pkl')
        write_smpl_pickle(smpl, smpl_pkl)
        write_smpl_pickle(smpl, os.path.join(tmp, 'neutral_smpl_with_cocoplus_reg.pkl'))
        gen_smpl(out, syn, smpl_pkl)
        print('smpl done', flush=True)
        gen_models(out, syn, weights)
        print('models done', flush=True)
        gen_tester(out, syn, ckpt, weights, smpl, tmp)
        print('tester done', flush=True)
        gen_tester_three_deltas(out, syn, ckpt, smpl, tmp)
        gen_feature_extractor(out, syn, ckpt, weights, tmp)
        gen_process_image(out, tmp)
        gen_eval_util(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes,', len(out), 'arrays')


if __name__ == '__main__':
    main()
