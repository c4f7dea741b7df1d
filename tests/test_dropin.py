"""Drop-in proof (INTEGRATION.md section 1): this package's classes do what the UNMODIFIED reference's code does with
its own classes, on the same inputs.  The reference's results are stored in tests/golden/reference_golden.npz
(oracle/make_reference_golden.py runs the reference's Trainer and predict_scene once):

  * one `Trainer.train_batch` (reference lstm/trainer.py:229-269) of
    `trajnetplusplusbaselines_b200.lstm.{LSTM, GridBasedPooling, PredictionLoss}` on the GPU against the same step of
    the reference's model on the CPU: loss and the parameters after the optimizer step.
  * `predict_scene` (reference lstm/trajnet_evaluator.py:15-19: preprocess_test, then the predictor) with this
    package's `LSTMPredictor` against the reference's predictor.
"""
import argparse

import numpy as np
import pytest
import torch

from oracle import lstm_oracle as O
from oracle.make_reference_golden import GOLDEN, SGD_LR, paths_from_xy, sample_index


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


def _model(kind, seed):
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling
    spec = O.MODEL_SPECS[kind]
    mine = LSTM(pool=GridBasedPooling(**spec) if spec is not None else None)
    mine.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in O.random_weights(kind, seed=seed).items()}, strict=True)
    return mine.cuda()


def _train_batch(model, criterion, optimizer, scene, goals, split, obs_length=9, pred_length=12):
    """One training step as Trainer.train_batch takes it: teacher-forced forward, loss on the last pred_length outputs
    (positions of the primary tracks passed for the collision term) x batch size, backward, optimizer step."""
    batch_size = len(split) - 1
    rel, pos = model(scene[:obs_length], goals, split, scene[obs_length:-1])
    targets = scene[obs_length:] - scene[obs_length - 1:-1]
    primary = scene[-pred_length:].clone()
    primary[:, split[:-1]] = pos[-pred_length:, split[:-1]]
    loss = criterion(rel[-pred_length:], targets, split, primary) * batch_size
    optimizer.zero_grad()
    loss.backward()
    optimizer.step()
    return loss.item()


def _step_names(ref, kind):
    prefix = "trainer/%s/step/" % kind
    return list(dict.fromkeys(k[len(prefix):].rsplit("/", 1)[0] for k in ref.files if k.startswith(prefix)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["vanilla", "directional", "social_small"])
def test_reference_trainer_drives_b200_model(kind, ref):
    from trajnetplusplusbaselines_b200 import _lib
    from trajnetplusplusbaselines_b200.lstm import PredictionLoss
    model = _model(kind, seed=11)
    model.train()
    xy, bs = O.synthetic_scenes(10, 7, seed=17, ragged=True, nan_tracks=True)
    scene = torch.from_numpy(xy).cuda()
    goals = torch.zeros(xy.shape[1], 2).cuda()
    split = torch.from_numpy(bs).cuda()
    # plain SGD: the parameter update is proportional to the gradient, so the comparison after the step is a
    # comparison of the whole backward pass (Adam's first step is +-lr whatever the magnitude)
    before = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    launches = _lib.load().tb2_launch_count()
    loss_ref = float(ref["trainer/%s/loss_sgd" % kind])
    loss_b200 = _train_batch(model, PredictionLoss(), torch.optim.SGD(model.parameters(), lr=SGD_LR), scene, goals, split)
    assert _lib.load().tb2_launch_count() > launches + 20        # forward, loss and backward kernels of this library ran
    assert abs(loss_b200 - loss_ref) <= 1e-4 * max(1.0, abs(loss_ref)), (loss_b200, loss_ref)
    sd_b200 = model.state_dict()
    assert _step_names(ref, kind) == list(sd_b200.keys())
    worst = 0.0
    for k in sd_b200:
        step_b200 = (sd_b200[k].cpu() - before[k]).numpy().reshape(-1)
        key = "trainer/%s/step/%s/" % (kind, k)
        if key + "full" in ref.files:
            step_ref = ref[key + "full"].reshape(-1)
            scale = max(float(np.abs(step_ref).max()), 1e-6 * SGD_LR)
        else:                                     # large tensor: seeded sample, plus max |.|, sum and sum |.| of all of it
            amax, total, abs_total = ref[key + "stats"]
            scale = max(float(amax), 1e-6 * SGD_LR)
            assert abs(step_b200.sum(dtype=np.float64) - total) <= 1e-3 * scale * step_b200.size, k
            assert abs(np.abs(step_b200).sum(dtype=np.float64) - abs_total) <= 1e-3 * scale * step_b200.size, k
            step_b200, step_ref = step_b200[sample_index(step_b200.size)], ref[key + "samples"]
        worst = max(worst, float(np.abs(step_b200 - step_ref).max()) / scale)
    assert worst < 1e-3, worst            # update of every parameter tensor within 0.1 % of its largest entry

    # default optimizer of the reference Trainer (Adam + weight decay) on the stepped model: runs and tracks the loss
    adam = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4)
    l2 = _train_batch(model, PredictionLoss(), adam, scene, goals, split)
    l2_ref = float(ref["trainer/%s/loss_adam" % kind])
    assert abs(l2 - l2_ref) <= 2e-3 * max(1.0, abs(l2_ref)), (l2, l2_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["vanilla", "directional", "social"])
def test_reference_predict_scene_drives_b200_predictor(kind, ref):
    from trajnetplusplusbaselines_b200.data import preprocess_test
    from trajnetplusplusbaselines_b200.lstm import LSTMPredictor
    model = _model(kind, seed=4)
    xy, _ = O.synthetic_scenes(1, 6, seed=23)
    paths = paths_from_xy(xy.astype(np.float64), late={4})        # pedestrian 4 is dropped by preprocess_test
    goal = np.zeros((len(paths), 2))

    def predict_scene(args):
        return LSTMPredictor(model)(preprocess_test(paths, args.obs_length), goal, n_predict=args.pred_length,
                                    obs_length=args.obs_length, modes=args.modes, args=args)

    args = argparse.Namespace(obs_length=9, pred_length=12, modes=1, normalize_scene=False)
    out = predict_scene(args)
    assert list(out.keys()) == [0]
    prim, neigh = out[0]
    prim_ref, neigh_ref = ref["predict/%s/plain/primary" % kind], ref["predict/%s/plain/neighbours" % kind]
    assert prim.shape == prim_ref.shape == (12, 2) and neigh.shape == neigh_ref.shape
    assert np.abs(prim - prim_ref).max() < 1e-4
    assert (np.isnan(neigh) == np.isnan(neigh_ref)).all()
    assert np.nanmax(np.abs(neigh - neigh_ref)) < 1e-4
    # normalize_scene=True goes through center_scene / inverse_scene on both sides
    args.normalize_scene = True
    out = predict_scene(args)
    assert np.abs(out[0][0] - ref["predict/%s/normalized/primary" % kind]).max() < 1e-4
