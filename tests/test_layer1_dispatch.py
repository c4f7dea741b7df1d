"""The first Linear of the social grid embedding has two tcgen05 kernels: the CTA-pair kernel that runs by default
and round 1's sparse_layer1_tc, which TB2_SPARSE=tc forces.  Both form the same products in the same order per
output column, so their outputs must agree bit for bit (DESIGN.md section 2), at the BASELINE batch size."""
import ctypes
import json

import numpy as np
import pytest
import torch

from oracle import lstm_oracle as O

pytestmark = pytest.mark.gpu

# one_layer embedding: the pool output IS the first Linear's output
SOCIAL_L1 = dict(type_="social", hidden_dim=128, cell_side=0.6, n=16, out_dim=1024,
                 embedding_arch="one_layer", latent_dim=16)


def _padded_inputs(ragged):
    """256 scenes x 20 pedestrians (ragged: 2..20 pedestrians, tracks entering / leaving) as the padded
    [B, Nmax, .] tensors the pool plug takes."""
    xy, bs = O.synthetic_scenes(256, 20, n_frames=4, seed=7, ragged=ragged, nan_tracks=ragged)
    h = (np.random.RandomState(11).randn(xy.shape[1], 128) * 0.5).astype(np.float32)
    sizes = np.diff(bs)

    def pad(a):
        out = np.full((len(sizes), int(sizes.max())) + a.shape[1:], np.nan, dtype=np.float32)
        for b in range(len(sizes)):
            out[b, :sizes[b]] = a[bs[b]:bs[b + 1]]
        return torch.from_numpy(out).cuda()

    return pad(h), pad(xy[2]), pad(xy[3])


def _pool(kind, monkeypatch):
    from trajnetplusplusbaselines_b200.lstm import GridBasedPooling
    monkeypatch.setitem(O.MODEL_SPECS, "social_l1", SOCIAL_L1)
    W = O.random_weights(kind, seed=21)
    pool = GridBasedPooling(**O.MODEL_SPECS[kind])
    pool.load_state_dict({k[len("pool."):]: torch.from_numpy(v.copy()) for k, v in W.items() if k.startswith("pool.")},
                         strict=True)
    return pool.cuda()


def _run_profiled(pool, inputs):
    """The pool output and the names of the library kernels the call launched."""
    from trajnetplusplusbaselines_b200 import _lib
    lib = _lib.load()
    lib.tb2_profile_begin()
    out = pool(*inputs).cpu().numpy()
    buf = ctypes.create_string_buffer(1 << 16)
    _lib.check(lib.tb2_profile_end(buf, len(buf)))
    return out, set(json.loads(buf.value.decode()))


@pytest.mark.parametrize("ragged", [False, True], ids=["regular", "ragged_nan"])
@pytest.mark.parametrize("kind", ["social_l1", "social"])
def test_pair_kernel_equals_round1_kernel(kind, ragged, monkeypatch):
    pool = _pool(kind, monkeypatch)
    inputs = _padded_inputs(ragged)
    monkeypatch.delenv("TB2_SPARSE", raising=False)
    out, kernels = _run_profiled(pool, inputs)
    assert "sparse_layer1_pair_ts" in kernels and "sparse_layer1_tc" not in kernels, kernels
    monkeypatch.setenv("TB2_SPARSE", "tc")
    ref, kernels_tc = _run_profiled(pool, inputs)
    assert "sparse_layer1_tc" in kernels_tc and "sparse_layer1_pair_ts" not in kernels_tc, kernels_tc
    assert np.array_equal(out, ref, equal_nan=True)
