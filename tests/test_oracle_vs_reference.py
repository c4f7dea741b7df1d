"""Oracle vs the UNMODIFIED reference on the same inputs: the reference's outputs are stored in
tests/golden/reference_golden.npz (oracle/make_reference_golden.py)."""
import numpy as np
import pytest

from oracle import lstm_oracle as O
from oracle.make_reference_golden import GOLDEN, positions_from_normals


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


@pytest.mark.parametrize("kind", ["vanilla", "directional", "social_small", "occupancy_front", "directional_const"])
@pytest.mark.parametrize("variant", ["plain", "ragged_nan"])
def test_forward_live(kind, variant, ref):
    ragged = variant == "ragged_nan"
    xy, bs = O.synthetic_scenes(7, 9, seed=123, ragged=ragged, nan_tracks=ragged)
    W = O.random_weights(kind, seed=5)
    rel = ref["forward/%s/%s/rel" % (kind, variant)]
    pred = positions_from_normals(xy[:9], rel)
    rel_o, pred_o = O.forward(W, O.pool_config(kind), xy[:9], bs, n_predict=12)
    assert (np.isnan(rel) == np.isnan(rel_o)).all()
    assert np.nanmax(np.abs(rel - rel_o)) < 2e-5
    assert np.nanmax(np.abs(pred - pred_o)) < 2e-5


def test_social_full_config_live(ref):
    xy, bs = O.synthetic_scenes(4, 8, seed=7)
    W = O.random_weights("social", seed=3)
    rel_o, pred_o = O.forward(W, O.pool_config("social"), xy[:9], bs, n_predict=12)
    assert np.nanmax(np.abs(ref["social_full/pred"] - pred_o)) < 2e-5


@pytest.mark.parametrize("kind", ["vanilla", "occupancy", "social_small"])
def test_sgan_generator_and_discriminator_live(kind, ref):
    """oracle/sgan_oracle.py vs the reference's LSTMGenerator / LSTMDiscriminator (noise fixed)."""
    from oracle import sgan_oracle as SO
    noise = np.linspace(-1.5, 1.5, 8).astype(np.float32)
    xy, bs = O.synthetic_scenes(5, 6, seed=321, ragged=True, nan_tracks=True)
    Wg, Wd = SO.sgan_weights(kind, 9)
    rel, pred, scores = (ref["sgan/%s/%s" % (kind, name)] for name in ("rel", "pred", "scores"))
    rel_o, pred_o = SO.generator_forward(Wg, O.pool_config(kind), xy[:9], bs, n_predict=12, noise=noise)
    assert (np.isnan(pred) == np.isnan(pred_o)).all()
    assert np.nanmax(np.abs(pred - pred_o)) < 2e-5
    assert np.nanmax(np.abs(rel - rel_o)) < 2e-5
    assert np.abs(scores - SO.discriminator_forward(Wd, O.pool_config(kind), xy[:9], xy[9:21], bs)).max() < 2e-5


def test_vae_test_time_live(ref):
    from oracle import sgan_oracle as SO
    xy, bs = O.synthetic_scenes(4, 5, seed=654, nan_tracks=True)
    W = SO.vae_weights("vanilla", 5)
    z = (np.random.RandomState(3).standard_normal((xy.shape[1], 128)) * 1.6).astype(np.float32)
    rel_o, pred_o = SO.vae_forward(W, None, xy[:9], bs, n_predict=12, z=z)
    assert np.nanmax(np.abs(ref["vae/pred"] - pred_o)) < 2e-5
    assert np.nanmax(np.abs(ref["vae/rel"] - rel_o)) < 2e-5
