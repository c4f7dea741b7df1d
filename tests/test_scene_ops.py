"""Scene preprocessing on the device (SURVEY.md 8f rank 3; reference lstm/lstm.py:16-22, lstm/utils.py:10-51,
augmentation.py:65-68): the per-scene NumPy functions of this package are pinned to the reference's on the CPU; the batched
CUDA passes (csrc/scene_ops.cu) must reproduce the per-scene host chain BIT FOR BIT (float64 arithmetic in the
reference's order, one rounding to float32)."""
import math

import numpy as np
import pytest
import torch

from trajnetplusplusbaselines_b200.lstm.lstm import center_scene, drop_distant, inverse_scene, theta_rotation


def _scenes(sizes, seed=0, T=21):
    rng = np.random.RandomState(seed)
    out = []
    for n in sizes:
        xy = rng.randn(n, 2) * 4.0 + rng.randn(2) * 30.0
        xy = xy[None] + np.cumsum(rng.randn(T, n, 2) * 0.3, axis=0)
        if n > 1:
            late = rng.rand(n) < 0.2
            late[0] = False
            xy[:3, late] = np.nan                      # late entries
            gone = rng.rand(n) < 0.1
            gone[0] = False
            xy[6:, gone] = np.nan                      # early exits
        if n > 3:
            xy[:, 2] += 40.0                           # far away in every frame: dropped by drop_distant
            xy[:, 3] = np.nan                          # never present: nanmin is NaN -> dropped
        out.append(xy)
    return out


def _host_chain(xy, r, normalize, obs_length, theta):
    """What lstm/trainer.py:107-116 does to one scene."""
    mask = np.ones(xy.shape[1], dtype=bool)
    if r is not None:
        with np.errstate(all='ignore'):
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                xy, mask = drop_distant(xy, r)
    rotation, center = 0.0, np.zeros(2)
    if normalize:
        xy, rotation, center = center_scene(xy, obs_length)
    if theta is not None:
        xy = theta_rotation(xy, theta)                 # random_rotation with a given angle (lstm/utils.py:10-17)
    return torch.Tensor(xy).numpy(), mask, rotation, center


def test_scene_frames_match_center_scene():
    from trajnetplusplusbaselines_b200.lstm.scene_ops import _frame_table, scene_frames
    scenes = _scenes([1, 2, 5, 17, 40], seed=3)
    split = np.concatenate([[0], np.cumsum([s.shape[1] for s in scenes])])
    center, rotation = scene_frames(np.concatenate(scenes, axis=1), split, obs_length=9)
    for i, xy in enumerate(scenes):
        _, rot, cen = center_scene(xy, 9)
        assert rot == rotation[i] and np.array_equal(cen, center[i])
    table = _frame_table(center, rotation)
    assert table[2, 2] == math.cos(rotation[2]) and table[2, 3] == math.sin(rotation[2])


def test_host_functions_match_reference():
    """Against the outputs of the reference's drop_distant / center_scene / theta_rotation / inverse_scene on the same
    scenes (tests/golden/reference_golden.npz, oracle/make_reference_golden.py)."""
    from oracle.make_reference_golden import GOLDEN, SCENE_SIZES
    ref = np.load(GOLDEN)
    import warnings
    for i, xy in enumerate(_scenes(SCENE_SIZES, seed=5)):
        key = "scene_ops/%d/" % i
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            a, ma = drop_distant(xy)
        b, mb = ref[key + "drop_distant"], ref[key + "drop_distant_mask"]
        assert np.array_equal(ma, mb) and np.array_equal(a, b, equal_nan=True)
        c, rot, cen = center_scene(xy, 9)
        d, rot_r, cen_r = ref[key + "center_scene"], ref[key + "rotation"], ref[key + "center"]
        assert rot == rot_r and np.array_equal(cen, cen_r) and np.array_equal(c, d, equal_nan=True)
        assert np.array_equal(theta_rotation(xy, 1.234), ref[key + "theta_rotation"], equal_nan=True)
        pred = c.astype(np.float32)
        assert np.array_equal(inverse_scene(pred, rot, cen), ref[key + "inverse_scene"], equal_nan=True)


CASES = [
    dict(r=6.0, normalize=True, aug=True),
    dict(r=6.0, normalize=False, aug=False),
    dict(r=None, normalize=True, aug=False),
    dict(r=None, normalize=False, aug=True),
    dict(r=2.5, normalize=True, aug=True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_cuda_preprocess_matches_host_chain_bitwise(case):
    from trajnetplusplusbaselines_b200 import _lib
    from trajnetplusplusbaselines_b200.lstm.scene_ops import preprocess_scenes
    sizes = [1, 2, 20, 7, 129, 300, 3, 64, 128, 5]        # > 128 tracks: several chunks of the block scan
    scenes = _scenes(sizes, seed=11)
    rng = np.random.RandomState(4)
    thetas = rng.rand(len(scenes)) * 2.0 * math.pi if case["aug"] else None
    before = _lib.load().tb2_launch_count()
    xy_dev, split, keep, rotation, center = preprocess_scenes(scenes, device="cuda", r=case["r"], normalize_scene=case["normalize"],
                                                              obs_length=9, thetas=thetas)
    assert _lib.load().tb2_launch_count() > before
    got = xy_dev.cpu().numpy()
    assert got.dtype == np.float32
    off = 0
    new_split = [0]
    for i, xy in enumerate(scenes):
        ref, mask, rot, cen = _host_chain(xy, case["r"], case["normalize"], 9, None if thetas is None else thetas[i])
        n_in, n_out = xy.shape[1], ref.shape[1]
        assert np.array_equal(keep[off:off + n_in], mask), i
        lo = int(split[i])
        assert int(split[i + 1]) - lo == n_out, i
        assert np.array_equal(got[:, lo:lo + n_out], ref, equal_nan=True), i          # bit for bit
        if case["normalize"]:
            assert rotation[i] == rot and np.array_equal(center[i], cen)
        off += n_in
        new_split.append(new_split[-1] + n_out)
    assert split.tolist() == new_split and got.shape[1] == new_split[-1]


@pytest.mark.gpu
def test_cuda_inverse_matches_host_bitwise():
    from trajnetplusplusbaselines_b200.lstm.scene_ops import inverse_scenes
    sizes = [1, 6, 20, 150]
    rng = np.random.RandomState(2)
    split = np.concatenate([[0], np.cumsum(sizes)])
    pred = (rng.randn(19, split[-1], 2) * 5).astype(np.float32)
    pred[3:, 4] = np.nan
    rotation = rng.rand(len(sizes)) * 6.0 - 3.0
    center = rng.randn(len(sizes), 2) * 20.0
    got = inverse_scenes(torch.from_numpy(pred).cuda(), split, rotation, center)
    assert got.dtype == np.float64
    for i in range(len(sizes)):
        ref = inverse_scene(pred[:, split[i]:split[i + 1]], rotation[i], center[i])
        assert np.array_equal(got[:, split[i]:split[i + 1]], ref, equal_nan=True), i


@pytest.mark.gpu
def test_predict_batch_normalized_equals_single_calls():
    """predict_batch(normalize_scene=True) centres / rotates / inverts every scene on the device; the per-scene call does it
    on the host like the reference (lstm/lstm.py:292-304): same float32 inputs, same predictions."""
    from types import SimpleNamespace
    from oracle import lstm_oracle as O
    from trajnetplusplusbaselines_b200.data import TrackRow
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling, LSTMPredictor
    kind = "directional"
    W = O.random_weights(kind, seed=12)
    model = LSTM(pool=GridBasedPooling(**O.MODEL_SPECS[kind]))
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in W.items()})
    predictor = LSTMPredictor(model.cuda().eval())
    rng = np.random.RandomState(9)
    scenes = []
    for n in (3, 1, 6, 4):
        start = rng.randn(n, 2) * 2.0 + 10.0
        vel = rng.randn(n, 2) * 0.3
        scenes.append([[TrackRow(f, 10 + p, float(start[p, 0] + vel[p, 0] * f), float(start[p, 1] + vel[p, 1] * f))
                        for f in range(1 if p % 3 != 2 else 4, 10)] for p in range(n)])
    args = SimpleNamespace(normalize_scene=True)
    singles = [predictor(p, np.zeros((len(p), 2)), n_predict=12, obs_length=9, modes=1, args=args) for p in scenes]
    batched = predictor.predict_batch(scenes, n_predict=12, obs_length=9, args=args)
    for s_out, b_out in zip(singles, batched):
        assert s_out[0][0].dtype == b_out[0][0].dtype == np.float64
        assert np.array_equal(s_out[0][0], b_out[0][0], equal_nan=True)
        assert np.array_equal(s_out[0][1], b_out[0][1], equal_nan=True)
