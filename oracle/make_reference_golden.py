"""Golden vectors for the tests that compare with the UNMODIFIED reference run live: the reference is run
once here on exactly the inputs those tests build, and its outputs are stored so the tests need no copy of it.

    python -m oracle.make_reference_golden  -> tests/golden/reference_golden.npz   (model / scene-function outputs)
                                            -> tests/golden/data_block_sample.npz  (sample of the reference's DATA_BLOCK)

Large parameter updates are stored as a seeded sample plus max |.|, sum and sum |.| (see `summarize`).
TEST INFRASTRUCTURE.
"""
import argparse
import glob
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import lstm_oracle as O           # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_golden.npz")
DATA_BLOCK_SAMPLE = os.path.join(ROOT, "tests", "golden", "data_block_sample.npz")

FORWARD_KINDS = ["vanilla", "directional", "social_small", "occupancy_front", "directional_const"]
FORWARD_VARIANTS = ["plain", "ragged_nan"]
SGAN_KINDS = ["vanilla", "occupancy", "social_small"]
TRAINER_KINDS = ["vanilla", "directional", "social_small"]
PREDICT_KINDS = ["vanilla", "directional", "social"]
SCENE_SIZES = [1, 4, 9, 33]
SGD_LR = 0.05

FULL_LIMIT = 2048
N_SAMPLES = 256
SCENES_PER_TRAIN_FILE = 40            # DATA_BLOCK training files: the 40 scenes that end first, with their frames


def summarize(name, a, out):
    """Tensors up to FULL_LIMIT entries in full; larger ones as N_SAMPLES seeded entries, max |.|, sum, sum |.|."""
    a = np.asarray(a, dtype=np.float32)
    if a.size <= FULL_LIMIT:
        out[name + "/full"] = a
        return
    out[name + "/samples"] = a.reshape(-1)[sample_index(a.size)]
    out[name + "/stats"] = np.array([np.abs(a).max(), a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64)])


def positions_from_normals(observed, rel):
    """The positions LSTM.forward returns beside its normals (reference lstm/lstm.py:226-255): the mean offset added to
    the current observation, then to the previous prediction, in float32.  Stored forward cases keep `rel` only;
    main() checks that this rebuilds the reference's positions bit for bit."""
    pos = np.empty(rel.shape[:2] + (2,), dtype=np.float32)
    n_obs = observed.shape[0] - 1
    pos[:n_obs] = observed[1:] + rel[:n_obs, :, :2]
    for t in range(n_obs, rel.shape[0]):
        pos[t] = pos[t - 1] + rel[t, :, :2]
    return pos


def sample_index(size):
    return np.random.RandomState(2024).randint(0, size, size=N_SAMPLES)


def paths_from_xy(xy, late=(), first_frame=100, step=10):
    """TrackRow paths of one scene; pedestrians in `late` enter after the observation period."""
    from trajnetplusplusbaselines_b200.data import TrackRow
    paths = []
    for p in range(xy.shape[1]):
        rows = []
        for t in range(xy.shape[0]):
            if p in late and t < 10:
                continue
            rows.append(TrackRow(first_frame + step * t, 7 + p, float(xy[t, p, 0]), float(xy[t, p, 1])))
        paths.append(rows)
    return paths


def scene_ops_scenes():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_scene_ops import _scenes
    return _scenes(SCENE_SIZES, seed=5)


def oracle_cases(out):
    import torch
    from oracle import sgan_oracle as SO
    from oracle.make_golden import build_reference_model
    import trajnetbaselines.sgan.sgan as ref_sgan
    import trajnetbaselines.vae.vae as ref_vae
    from trajnetbaselines.lstm.gridbased_pooling import GridBasedPooling
    for kind in FORWARD_KINDS:
        for variant in FORWARD_VARIANTS:
            ragged = variant == "ragged_nan"
            xy, bs = O.synthetic_scenes(7, 9, seed=123, ragged=ragged, nan_tracks=ragged)
            model = build_reference_model(kind, O.random_weights(kind, seed=5))
            with torch.no_grad():
                rel, pred = model(torch.from_numpy(xy[:9]), torch.zeros(xy.shape[1], 2), torch.from_numpy(bs), n_predict=12)
            assert np.array_equal(positions_from_normals(xy[:9], rel.numpy()), pred.numpy(), equal_nan=True)
            out["forward/%s/%s/rel" % (kind, variant)] = rel.numpy()

    xy, bs = O.synthetic_scenes(4, 8, seed=7)
    model = build_reference_model("social", O.random_weights("social", seed=3))
    with torch.no_grad():
        _, pred = model(torch.from_numpy(xy[:9]), torch.zeros(xy.shape[1], 2), torch.from_numpy(bs), n_predict=12)
    out["social_full/pred"] = pred.numpy()

    noise = np.linspace(-1.5, 1.5, 8).astype(np.float32)
    ref_sgan.get_noise = lambda shape, noise_type, device: torch.from_numpy(noise.copy())
    for kind in SGAN_KINDS:
        xy, bs = O.synthetic_scenes(5, 6, seed=321, ragged=True, nan_tracks=True)
        spec = O.MODEL_SPECS[kind]
        Wg, Wd = SO.sgan_weights(kind, 9)
        gen = ref_sgan.LSTMGenerator(pool=GridBasedPooling(**spec) if spec else None)
        dis = ref_sgan.LSTMDiscriminator(pool=GridBasedPooling(**spec) if spec else None)
        for module, W in ((gen, Wg), (dis, Wd)):
            sd = module.state_dict()
            sd.update({k: torch.from_numpy(v.copy()) for k, v in W.items() if k in sd})
            module.load_state_dict(sd)
        scene, split = torch.from_numpy(xy), torch.from_numpy(bs)
        goals = torch.zeros(xy.shape[1], 2)
        with torch.no_grad():
            rel, pred = gen(scene[:9], goals, split, n_predict=12)
            scores = dis(scene[:9], scene[9:21], goals, split)
        out["sgan/%s/rel" % kind] = rel.numpy()
        out["sgan/%s/pred" % kind] = pred.numpy()
        out["sgan/%s/scores" % kind] = scores.numpy()

    xy, bs = O.synthetic_scenes(4, 5, seed=654, nan_tracks=True)
    W = SO.vae_weights("vanilla", 5)
    model = ref_vae.VAE(num_modes=1)
    sd = model.state_dict()
    sd.update({k: torch.from_numpy(v.copy()) for k, v in W.items() if k in sd})
    model.load_state_dict(sd)
    model.eval()
    z = (np.random.RandomState(3).standard_normal((xy.shape[1], 128)) * 1.6).astype(np.float32)
    ref_vae.sample_multivariate_distribution = lambda mean, var_log: torch.from_numpy(z.copy())
    with torch.no_grad():
        rel_list, pred_list, _, _ = model(torch.from_numpy(xy[:9]), torch.zeros(xy.shape[1], 2), torch.from_numpy(bs),
                                          n_predict=12)
    out["vae/rel"] = rel_list[0].numpy()
    out["vae/pred"] = pred_list[0].numpy()


def scene_ops_cases(out):
    from trajnetbaselines import augmentation
    from trajnetbaselines.lstm import lstm as ref_lstm
    from trajnetbaselines.lstm import utils as ref_utils
    for i, xy in enumerate(scene_ops_scenes()):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            b, mb = ref_lstm.drop_distant(xy)
        d, rot_r, cen_r = ref_utils.center_scene(xy, 9)
        key = "scene_ops/%d/" % i
        out[key + "drop_distant"], out[key + "drop_distant_mask"] = b, mb
        out[key + "center_scene"], out[key + "rotation"], out[key + "center"] = d, np.float64(rot_r), cen_r
        out[key + "theta_rotation"] = ref_utils.theta_rotation(xy, 1.234)
        out[key + "inverse_scene"] = augmentation.inverse_scene(d.astype(np.float32), rot_r, cen_r)


def dropin_cases(out):
    import torch
    from oracle.make_golden import build_reference_model
    from trajnetbaselines.lstm import trainer as ref_trainer
    from trajnetbaselines.lstm import trajnet_evaluator as ref_eval
    from trajnetbaselines.lstm.loss import PredictionLoss as RefLoss
    from trajnetbaselines.lstm.lstm import LSTMPredictor as RefPredictor
    for kind in TRAINER_KINDS:
        ref_model = build_reference_model(kind, O.random_weights(kind, seed=11))
        ref_model.train()
        xy, bs = O.synthetic_scenes(10, 7, seed=17, ragged=True, nan_tracks=True)
        B = len(bs) - 1
        scene, goals, split = torch.from_numpy(xy), torch.zeros(xy.shape[1], 2), torch.from_numpy(bs)
        t_ref = ref_trainer.Trainer(model=ref_model, criterion=RefLoss(), optimizer=torch.optim.SGD(ref_model.parameters(), lr=SGD_LR),
                                    device=torch.device("cpu"), batch_size=B, augment=False)
        before = {k: v.detach().clone() for k, v in ref_model.state_dict().items()}
        out["trainer/%s/loss_sgd" % kind] = np.float64(t_ref.train_batch(scene, goals, split))
        for k, v in ref_model.state_dict().items():
            summarize("trainer/%s/step/%s" % (kind, k), (v - before[k]).numpy(), out)
        t_def = ref_trainer.Trainer(model=ref_model, criterion=RefLoss(), device=torch.device("cpu"), batch_size=B, augment=False)
        out["trainer/%s/loss_adam" % kind] = np.float64(t_def.train_batch(scene, goals, split))

    for kind in PREDICT_KINDS:
        ref_model = build_reference_model(kind, O.random_weights(kind, seed=4))
        xy, _ = O.synthetic_scenes(1, 6, seed=23)
        paths = paths_from_xy(xy.astype(np.float64), late={4})
        goal = np.zeros((len(paths), 2))
        for normalize in (False, True):
            args = argparse.Namespace(obs_length=9, pred_length=12, modes=1, normalize_scene=normalize)
            prim, neigh = ref_eval.predict_scene(RefPredictor(ref_model), "m", paths, goal, args)[0]
            key = "predict/%s/%s/" % (kind, "normalized" if normalize else "plain")
            out[key + "primary"], out[key + "neighbours"] = prim, neigh


def data_block_sample(root):
    """The reference's DATA_BLOCK: small files whole; of each training file the lines of the scenes that end within its
    SCENES_PER_TRAIN_FILE scenes that end first and every track row up to that frame, in file order."""
    import json
    out = {}
    base = os.path.join(root, "DATA_BLOCK")
    for fn in sorted(glob.glob(os.path.join(base, "**", "*.ndjson"), recursive=True)):
        lines = open(fn, "rb").read().splitlines(keepends=True)
        rel = os.path.relpath(fn, base)
        if os.sep + "train" + os.sep not in os.sep + rel:
            out[rel] = np.frombuffer(b"".join(lines), dtype=np.uint8)
            continue
        recs = [json.loads(ln) for ln in lines]
        ends = sorted(r["scene"]["e"] for r in recs if "scene" in r)
        last = ends[SCENES_PER_TRAIN_FILE - 1]
        keep = [ln for ln, r in zip(lines, recs)
                if ("track" in r and r["track"]["f"] <= last) or ("scene" in r and r["scene"]["e"] <= last)]
        out[rel] = np.frombuffer(b"".join(keep), dtype=np.uint8)
    return out


def main():
    from oracle.ref_shim import import_reference, reference_root
    import_reference()
    out = {}
    oracle_cases(out)
    scene_ops_cases(out)
    dropin_cases(out)
    np.savez_compressed(GOLDEN, **out)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")
    np.savez_compressed(DATA_BLOCK_SAMPLE, **data_block_sample(reference_root()))
    print("wrote", DATA_BLOCK_SAMPLE, os.path.getsize(DATA_BLOCK_SAMPLE), "bytes")


if __name__ == "__main__":
    main()
