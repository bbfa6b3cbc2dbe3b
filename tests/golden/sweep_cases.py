"""Seeded inputs of the reference sweeps shared by make_ref_exec_golden.py (which runs them through the reference's own source and
stores the outputs in ref_sweeps_v1.npz) and tests/test_ref_exec.py (which runs them through this repo and compares).  Plus the
two helpers that shrink a large output for storage: a fixed sample and float64 projection checksums every element contributes to."""
import numpy as np

VERT_IDS = np.arange(0, 6890, 106)          # 65 sampled vertices of the SMPL sweep


def checksum(a, lead=1, k=4, seed=0):
    """float64 projections of each of the first `lead` axes' entries onto k fixed seeded random vectors: every element counts."""
    a = np.asarray(a, np.float64)
    flat = a.reshape(a.shape[:lead] + (-1,))
    return flat @ np.random.RandomState(seed).normal(size=(flat.shape[-1], k))


def eval_sweep():
    """24 cases: mirrored predictions (every 3rd) and sparse visibility (every 4th / 5th)."""
    rng = np.random.RandomState(99)
    cases = []
    for i in range(24):
        gt = rng.normal(0, 0.4, size=(12, 14, 3))
        pr = gt + rng.normal(0, 0.05, size=gt.shape)
        if i % 3 == 0:
            pr[..., 0] *= -1.0
        vis = rng.rand(12) > (0.6 if i % 4 == 0 else 0.1)
        kg = np.concatenate([rng.rand(5, 19, 2) * 2 - 1, (rng.rand(5, 19, 1) > (0.75 if i % 5 == 0 else 0.2)).astype(np.float64)], axis=2)
        kp = kg[:, :, :2] + rng.normal(0, 0.05, size=(5, 19, 2))
        cases.append((gt, pr, vis, kg, kp))
    return cases


# (N frames, B, T, num_conv_layers): ragged tails, N < one window, exact multiples, minimal T = fov
SLIDING_CASES = [(23, 2, 20, 3), (3, 1, 20, 3), (16, 2, 20, 3), (17, 2, 20, 3), (1, 4, 20, 3), (40, 1, 13, 3), (9, 3, 12, 2), (30, 2, 9, 2),
                 (5, 2, 6, 1)]


def sliding_frames(N, dtype):
    """Frame k is filled with k + 1, so the probe `predict` can report which frames it was shown."""
    return np.tile((np.arange(N, dtype=dtype) + 1.0).reshape(N, 1, 1, 1), (1, 2, 2, 3))


def other_config_inputs(syn):
    """num_conv_layers=2, B=3, T=7, delta heads (-3, +3), weights seed 31."""
    w = syn.make_synthetic_weights(seed=31, num_conv_layers=2, delta_t_values=(-3, 3))
    x = np.random.RandomState(32).normal(0, 1, size=(3, 7, 2048)).astype(np.float32)
    om0 = np.tile(np.asarray(w['mean_param'], np.float32).reshape(1, 85), (21, 1))
    return w, x, om0


def smpl_sweep_model(syn):
    return syn.make_synthetic_smpl(seed=7, dense_weights=True, num_kps=19)


def smpl_sweep_inputs():
    """48 poses with LARGE rotations (theta ~ N(0, 1), beta ~ N(0, 2)); pose 1 has the mean pose's root rotation."""
    rng = np.random.RandomState(2718)
    beta = rng.normal(0, 2.0, size=(48, 10)).astype(np.float32)
    theta = rng.normal(0, 1.0, size=(48, 72)).astype(np.float32)
    theta[1, :3] = [np.pi, 0, 0]
    cam = rng.normal(0, 1, size=(48, 3)).astype(np.float32)
    return beta, theta, cam


def process_image_sweep():
    """40 random (frame size, bbox, frame) cases: yields (H, W, cx, cy, s, uint8 frame)."""
    rng = np.random.RandomState(314)
    for _ in range(40):
        H, W = int(rng.randint(60, 400)), int(rng.randint(60, 400))
        s = float(rng.uniform(0.4, 1.8))
        cx, cy = float(rng.uniform(0, W)), float(rng.uniform(0, H))
        frame = rng.randint(0, 256, size=(H, W, 3)).astype(np.uint8)
        yield H, W, cx, cy, s, frame


def pixel_sample(img, i, n=32):
    """n fixed seeded pixels (all channels) of crop i."""
    img = np.asarray(img, np.float64)
    flat = img.reshape(-1, img.shape[-1])
    return flat[np.sort(np.random.RandomState(i).choice(flat.shape[0], n, replace=False))]
