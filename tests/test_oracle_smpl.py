"""CPU: the SMPL oracle (oracle/smpl_ref.py) against analytic known-answers and an independent loop implementation.
The reference ships no tests for this path (SURVEY.md 4), so these pin the restatement itself."""
import numpy as np
import pytest

from oracle import smpl_ref
from human_dynamics_b200 import synthetic


def test_rodrigues_zero_is_identity():
    R = smpl_ref.batch_rodrigues(np.zeros((5, 3), np.float32))
    assert np.array_equal(R, np.tile(np.eye(3, dtype=np.float32), (5, 1, 1)))      # batch_lbs.py:48-59, theta=0 => R=I exactly


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_rodrigues_closed_forms_and_orthonormality(dtype):
    th = np.array([[np.pi / 2, 0, 0], [0, np.pi, 0], [0, 0, -np.pi / 2], [0.3, -0.2, 0.9]], dtype)
    R = smpl_ref.batch_rodrigues(th, dtype)
    tol = 1e-6 if dtype == np.float32 else 1e-7     # the reference's 1e-8 shift perturbs the angle slightly
    assert np.allclose(R[0], [[1, 0, 0], [0, 0, -1], [0, 1, 0]], atol=tol)
    assert np.allclose(R[1], [[-1, 0, 0], [0, 1, 0], [0, 0, -1]], atol=tol)
    assert np.allclose(R[2], [[0, 1, 0], [-1, 0, 0], [0, 0, 1]], atol=tol)
    for r in R:
        assert np.allclose(r @ r.T, np.eye(3), atol=10 * tol)
        assert abs(np.linalg.det(r.astype(np.float64)) - 1) < 10 * tol


def test_rodrigues_matches_scipy():
    from scipy.spatial.transform import Rotation
    th = np.random.RandomState(0).normal(0, 0.7, size=(50, 3))
    assert np.allclose(smpl_ref.batch_rodrigues(th, np.float64), Rotation.from_rotvec(th).as_matrix(), atol=1e-7)


def test_skew_layout():
    S = smpl_ref.batch_skew(np.array([[1., 2., 3.]], np.float32))[0]
    assert np.array_equal(S, np.array([[0, -3, 2], [3, 0, -1], [-2, 1, 0]], np.float32))       # batch_lbs.py:24-36


def _fk_loops(Rs, Js, parents):
    """Independent per-sample FK with explicit 4x4 chains."""
    N = Rs.shape[0]
    newJ = np.zeros((N, 24, 3)); A = np.zeros((N, 24, 4, 4))
    for n in range(N):
        G = []
        for i in range(24):
            T = np.eye(4); T[:3, :3] = Rs[n, i]
            T[:3, 3] = Js[n, i] if i == 0 else Js[n, i] - Js[n, parents[i]]
            G.append(T if i == 0 else G[parents[i]] @ T)
        for i in range(24):
            newJ[n, i] = G[i][:3, 3]
            A[n, i] = G[i]
            A[n, i, :3, 3] -= G[i][:3, :3] @ Js[n, i]
    return newJ, A


def test_global_rigid_vs_loops_and_zero_pose():
    rng = np.random.RandomState(1)
    parents = synthetic.SMPL_PARENTS
    Rs = smpl_ref.batch_rodrigues(rng.normal(0, 0.5, size=(3 * 24, 3)), np.float64).reshape(3, 24, 3, 3)
    Js = rng.normal(0, 0.3, size=(3, 24, 3))
    nj, A = smpl_ref.batch_global_rigid_transformation(Rs, Js, parents, dtype=np.float64)
    nj2, A2 = _fk_loops(Rs, Js, parents)
    assert np.allclose(nj, nj2, atol=1e-12) and np.allclose(A, A2, atol=1e-12)
    assert np.allclose(A[:, :, 3], [0, 0, 0, 1])                                   # batch_lbs.py:192: last row [0,0,0,1]
    I = np.tile(np.eye(3), (3, 24, 1, 1))
    nj0, A0 = smpl_ref.batch_global_rigid_transformation(I, Js, parents, dtype=np.float64)
    assert np.allclose(nj0, Js, atol=1e-12)                                         # identity pose: joints stay, A = [I|0]
    assert np.allclose(A0, np.tile(np.eye(4), (3, 24, 1, 1)), atol=1e-12)
    njr, _ = smpl_ref.batch_global_rigid_transformation(Rs, Js, parents, rotate_base=True, dtype=np.float64)
    assert np.allclose(njr[:, 0], Js[:, 0])                                         # base flip leaves the root joint in place


def test_smpl_zero_pose_and_regressors(smpl_model):
    """BASELINE config 1: batch 4, theta = 0  =>  verts = v_shaped (rows of W sum to 1), joints = verts . regressor."""
    beta, theta = synthetic.make_smpl_inputs(4, seed=0, zero_pose=True)
    s = smpl_ref.SMPLRef(smpl_model, dtype=np.float64)
    verts, joints, Rs = s(beta, theta, get_skin=True)
    v_shaped = (beta.astype(np.float64) @ s.shapedirs).reshape(4, -1, 3) + s.v_template
    assert np.allclose(verts, v_shaped, atol=1e-12)
    assert np.allclose(Rs, np.tile(np.eye(3), (4, 24, 1, 1)), atol=1e-15)      # exact in float32 (test_rodrigues_zero_is_identity)
    assert np.allclose(joints, np.einsum('nvc,vk->nkc', verts, s.joint_regressor), atol=1e-12)
    assert np.allclose(s.J_transformed, np.einsum('nvc,vj->njc', v_shaped, s.J_regressor), atol=1e-12)
    assert joints.shape == (4, 25, 3)
    assert smpl_ref.SMPLRef(smpl_model, joint_type='lsp')(beta, theta).shape == (4, 14, 3)    # batch_smpl.py:81-82
    with pytest.raises(ValueError):
        smpl_ref.SMPLRef(smpl_model, joint_type='coco')


def test_smpl_root_rotation_equivariance(smpl_model):
    beta, theta = synthetic.make_smpl_inputs(3, seed=1)
    s = smpl_ref.SMPLRef(smpl_model, dtype=np.float64)
    v1, _, _ = s(beta, theta, get_skin=True)
    t0 = theta.copy(); t0[:, :3] = 0
    v0, _, _ = s(beta, t0, get_skin=True)
    J0 = s.J_transformed[:, 0:1]
    R0 = smpl_ref.batch_rodrigues(theta[:, :3], np.float64)
    assert np.allclose(np.einsum('nij,nvj->nvi', R0, v0 - J0) + J0, v1, atol=1e-9)


def test_smpl_f32_close_to_f64(smpl_model):
    beta, theta = synthetic.make_smpl_inputs(8, seed=2)
    v32, j32, _ = smpl_ref.SMPLRef(smpl_model, dtype=np.float32)(beta, theta, get_skin=True)
    v64, j64, _ = smpl_ref.SMPLRef(smpl_model, dtype=np.float64)(beta, theta, get_skin=True)
    assert np.abs(v32 - v64).max() / np.abs(v64).max() < 1e-5


def test_projection_formula():
    X = np.random.RandomState(0).normal(size=(4, 7, 3)).astype(np.float32)
    cam = np.array([[2.0, 0.5, -0.25]] * 4, np.float32)
    out = smpl_ref.batch_orth_proj_idrot(X, cam)
    assert out.shape == (4, 7, 2)
    assert np.allclose(out, 2.0 * (X[:, :, :2] + np.array([0.5, -0.25], np.float32)), atol=1e-6)   # projection.py:25-29


def test_face_table_is_bit_exact_fixture():
    """smpl_faces.npy is passed through unchanged (north_star: bit-exact face indexing): the table this repo ships is byte for
    byte the reference's src/tf_smpl/smpl_faces.npy, whose full sha256 is pinned here (SURVEY.md row 21)."""
    import hashlib, os
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'src', 'tf_smpl', 'smpl_faces.npy')
    f = np.load(p)
    assert f.shape == (13776, 3) and f.dtype == np.uint32 and f.min() == 0 and f.max() == 6889
    assert hashlib.sha256(open(p, 'rb').read()).hexdigest() == '51fc11ebadb0487d74bef220c4eea43f014609249f0121413c1fc629d859fecb'


def test_rot2aa_inverts_rodrigues():
    """batch_rot2aa (batch_lbs.py:63-105) recovers the axis-angle vector for angles in (0, pi); identity -> 0."""
    from oracle import smpl_ref
    rng = np.random.RandomState(0)
    axis = rng.normal(size=(64, 3)); axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    ang = rng.uniform(0.05, 3.0, size=(64, 1))
    th = axis * ang
    R = smpl_ref.batch_rodrigues(th, np.float64)
    assert np.allclose(smpl_ref.batch_rot2aa(R, np.float64), th, atol=1e-6)
    assert np.allclose(smpl_ref.batch_rot2aa(np.eye(3)[None], np.float64), 0.0)
