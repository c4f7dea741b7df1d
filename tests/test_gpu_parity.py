"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the committed reference
fixtures.  Run on the B200 box: `pytest -m gpu`.

Bars (BASELINE.json north_star): grid cell indices bit-exact; predicted positions within 1e-4 m
(ADE/FDE vs the reference), tolerance written at each assert.
"""
import os

import numpy as np
import pytest
import torch

from oracle import lstm_oracle as O
from oracle.make_golden import CASES

pytestmark = pytest.mark.gpu

TOL_POS = 1e-4      # metres, north_star: "within 1e-4 m on ADE/FDE"
TOL_STEP = 2e-5     # single teacher-forced step / short chains (fp32, different summation order)


def build_model(kind, W, device="cuda"):
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling
    spec = O.MODEL_SPECS[kind]
    pool = GridBasedPooling(**spec) if spec is not None else None
    model = LSTM(pool=pool)
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in W.items()}, strict=True)
    return model.to(device).eval()


def report(line):
    """Parity numbers of passing tests are kept (gpurun_out/parity_report.txt) for profiles/."""
    import os
    print(line)
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(d, exist_ok=True)
    tag = "[no-tc] " if os.environ.get("TB2_DISABLE_TC") == "1" else ""
    with open(os.path.join(d, "parity_report.txt"), "a") as f:
        f.write(tag + line + "\n")


def maxdiff(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    assert a.shape == b.shape, (a.shape, b.shape)
    assert (np.isnan(a) == np.isnan(b)).all(), "NaN pattern differs"
    return float(np.nanmax(np.abs(a - b))) if a.size else 0.0


# ---------------------------------------------------------------------------------------------
# grid cell indices: bit-exact
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["social", "directional", "occupancy_front"])
def test_grid_indices_match_reference_fixture(golden, kind):
    from trajnetplusplusbaselines_b200.engine import SceneLayout
    obs = golden["cells_%s/obs" % kind]                      # [B, N, 2]
    B, N, _ = obs.shape
    model = build_model(kind, O.random_weights(kind, seed=0))
    handle = model._engine()
    layout = SceneLayout(range(0, B * N + 1, N))
    cells, flags = handle.grid_indices(layout, torch.from_numpy(obs.reshape(B * N, 2)).cuda())
    assert np.array_equal(flags.cpu().numpy().astype(bool).reshape(B, N, N - 1), golden["cells_%s/in_range" % kind])
    assert np.array_equal(cells.cpu().numpy().reshape(B, N, N - 1), golden["cells_%s/cells" % kind])


@pytest.mark.parametrize("kind,seed", [("social", 0), ("directional", 1), ("occupancy_front", 2)])
def test_grid_indices_boundary_sweep_bit_exact(kind, seed):
    """20k pairs snapped onto / one ulp around cell edges, ragged scenes: int equality vs oracle."""
    from trajnetplusplusbaselines_b200.engine import SceneLayout
    cfg = O.pool_config(kind)
    rng = np.random.RandomState(seed)
    B, N = 64, 18
    sizes = rng.randint(2, N + 1, size=B)
    sizes[0] = N
    obs = np.full((B, N, 2), np.nan, dtype=np.float32)
    side = np.float32(cfg.cell_side)
    for b in range(B):
        pts = (rng.randn(sizes[b], 2) * 2.0).astype(np.float32)
        for j in range(1, sizes[b]):
            r = rng.rand()
            if r < 0.6:       # on a cell edge relative to ped 0, +- one ulp
                k = rng.randint(-cfg.n // 2 - 1, cfg.n // 2 + 2, size=2).astype(np.float32)
                edge = pts[0] + k * side
                pts[j] = np.nextafter(edge, edge + rng.choice([-1.0, 0.0, 1.0], size=2).astype(np.float32))
            if r > 0.95:
                pts[j] = np.nan
        obs[b, :sizes[b]] = pts
    cells_o, inr_o = O.grid_cells(obs, cfg)                 # padded [B, N, N-1]
    offs = np.concatenate([[0], np.cumsum(sizes)])
    flat = np.concatenate([obs[b, :sizes[b]] for b in range(B)]).astype(np.float32)
    model = build_model(kind, O.random_weights(kind, seed=0))
    layout = SceneLayout(offs.tolist())
    cells, flags = model._engine().grid_indices(layout, torch.from_numpy(flat).cuda())
    cells = cells.cpu().numpy()
    flags = flags.cpu().numpy().astype(bool)
    for b in range(B):
        s, e = offs[b], offs[b + 1]
        assert np.array_equal(flags[s:e], inr_o[b, :sizes[b]]), b
        assert np.array_equal(cells[s:e], cells_o[b, :sizes[b]].astype(np.int32)), b


# ---------------------------------------------------------------------------------------------
# pool plug
# ---------------------------------------------------------------------------------------------
def test_pool_plug_reference_golden_vectors(golden):
    """GridBasedPooling(embedding_arch='None') raw grids: adapted reference tests (SURVEY section 4)
    at pool_size = blur_size = 1 (the only values the reference CLI can produce)."""
    from trajnetplusplusbaselines_b200.lstm import GridBasedPooling
    nan = float("nan")
    pool = GridBasedPooling(n=2, cell_side=2.0, embedding_arch='None').cuda()
    o = torch.tensor([[[0., 0.], [-1., -1.]]])
    g = pool(torch.zeros(1, 2, 128), o, o)
    assert np.array_equal(g.cpu().numpy(), golden["sec4/simple_grid_ps1"])
    assert np.array_equal(g.cpu().numpy(), np.array([[1, 0, 0, 0], [0, 0, 0, 1]], dtype=np.float32))
    o = torch.tensor([[[0., 0.], [nan, nan]]])
    g = pool(torch.zeros(1, 2, 128), o, o)
    assert np.array_equal(g.cpu().numpy(), golden["sec4/nan"])
    pool = GridBasedPooling(n=2, cell_side=2.0, embedding_arch='None', type_='directional').cuda()
    o1 = torch.tensor([[[0., 0.], [-1., -1.]]])
    o2 = torch.tensor([[[0.1, 0.1], [-1.1, -1.1]]])
    g = pool(torch.zeros(1, 2, 128), o1, o2)
    assert np.allclose(g.cpu().numpy(), golden["sec4/directional_ps1"], atol=1e-7)
    assert g.shape == (2, 8)


@pytest.mark.parametrize("kind", ["occupancy", "directional", "social", "social_small",
                                  "directional_const", "occupancy_front"])
def test_pool_forward_matches_oracle(kind):
    from trajnetplusplusbaselines_b200.lstm import GridBasedPooling
    cfg = O.pool_config(kind)
    W = O.random_weights(kind, seed=21)
    rng = np.random.RandomState(5)
    B, N = 9, 11
    obs2 = (rng.randn(B, N, 2) * 2.0).astype(np.float32)
    obs1 = obs2 - (rng.randn(B, N, 2) * 0.3).astype(np.float32)
    hid = (rng.randn(B, N, 128) * 0.5).astype(np.float32)
    obs2[1, 4:] = np.nan          # padded scene
    obs1[1, 4:] = np.nan
    hid[1, 4:] = np.nan
    obs1[2, 3] = np.nan           # present now, absent before (velocity NaN -> 0 payload)
    obs2[3, 5] = np.nan           # absent now
    ref = O.pool_forward(cfg, W, hid, obs1, obs2)
    pool = GridBasedPooling(**O.MODEL_SPECS[kind])
    sd = {k[len("pool."):]: torch.from_numpy(v.copy()) for k, v in W.items() if k.startswith("pool.")}
    pool.load_state_dict(sd, strict=True)
    pool = pool.cuda()
    out = pool(torch.from_numpy(hid).cuda(), torch.from_numpy(obs1).cuda(), torch.from_numpy(obs2).cuda())
    assert out.shape == ref.shape
    assert maxdiff(out, ref) < TOL_STEP


# ---------------------------------------------------------------------------------------------
# step and sequence
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["vanilla", "directional", "social_small", "social"])
def test_single_step_matches_oracle(kind):
    W = O.random_weights(kind, seed=31)
    cfg = O.pool_config(kind)
    xy, bs = O.synthetic_scenes(12, 10, seed=3, ragged=True, nan_tracks=True)
    M = xy.shape[1]
    rng = np.random.RandomState(0)
    h = (rng.randn(M, 128) * 0.3).astype(np.float32)
    c = (rng.randn(M, 128) * 0.3).astype(np.float32)
    model = build_model(kind, W)
    for phase, lstm in (("encoder", model.encoder), ("decoder", model.decoder)):
        h_o, c_o, n_o = O.step(W, cfg, phase, h, c, xy[2], xy[3], bs)
        (h_g, c_g), n_g = model.step(lstm, (torch.from_numpy(h).cuda(), torch.from_numpy(c).cuda()),
                                     torch.from_numpy(xy[2]), torch.from_numpy(xy[3]), None, torch.from_numpy(bs))
        assert maxdiff(n_g, n_o) < TOL_STEP
        assert maxdiff(h_g, h_o) < TOL_STEP
        assert maxdiff(c_g, c_o) < TOL_STEP


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_forward_matches_reference_fixture(golden, case):
    name, kind, B, N, ragged, nan_tracks, dseed, wseed, wscale = case
    xy, bs = O.synthetic_scenes(B, N, seed=dseed, ragged=ragged, nan_tracks=nan_tracks)
    W = O.random_weights(kind, seed=wseed, scale=wscale)
    model = build_model(kind, W)
    M = xy.shape[1]
    with torch.no_grad():
        rel_f, pred_f = model(torch.from_numpy(xy[:9]), torch.zeros(M, 2), torch.from_numpy(bs), n_predict=12)
        rel_t, pred_t = model(torch.from_numpy(xy[:9]), torch.zeros(M, 2), torch.from_numpy(bs),
                              prediction_truth=torch.from_numpy(xy[9:20]).clone())
    assert rel_f.device.type == "cpu"          # outputs follow the input device (predictor calls .numpy())
    assert maxdiff(pred_t, golden[name + "/pred_teacher"]) < TOL_POS
    assert maxdiff(rel_t, golden[name + "/rel_teacher"]) < TOL_POS
    assert maxdiff(pred_f, golden[name + "/pred_free"]) < TOL_POS
    assert maxdiff(rel_f, golden[name + "/rel_free"]) < TOL_POS


@pytest.mark.parametrize("kind", ["vanilla", "occupancy", "directional", "social"])
def test_baseline_config_ade_fde_vs_oracle(kind):
    """BASELINE configs (N = 20, T = 9 + 12) at a batch the oracle finishes in seconds.  Gate on
    ADE / FDE of the primaries vs the oracle, mean over scenes <= 1e-4 m; cell flips (chaotic
    bin changes in a free-running rollout, SURVEY.md section 7) are reported, not hidden."""
    B, N = 48, 20
    xy, bs = O.synthetic_scenes(B, N, seed=100 + len(kind))
    W = O.random_weights(kind, seed=41)
    model = build_model(kind, W)
    M = xy.shape[1]
    with torch.no_grad():
        _, pred = model(torch.from_numpy(xy[:9]).cuda(), torch.zeros(M, 2), torch.from_numpy(bs), n_predict=12)
        _, pred_tf = model(torch.from_numpy(xy[:9]).cuda(), torch.zeros(M, 2), torch.from_numpy(bs),
                           prediction_truth=torch.from_numpy(xy[9:20]).cuda())
    assert pred.device.type == "cuda"
    _, pred_o = O.forward(W, O.pool_config(kind), xy[:9], bs, n_predict=12)
    _, pred_tf_o = O.forward(W, O.pool_config(kind), xy[:9], bs, prediction_truth=xy[9:20])
    pred = pred.cpu().numpy()
    prim = bs[:-1]
    ades, fdes = [], []
    for p in prim:
        a, f = O.ade_fde(pred[-12:, p], pred_o[-12:, p])
        ades.append(a)
        fdes.append(f)
    flips = int((np.array(fdes) > 1e-3).sum())
    report("%s: ADE mean %.3e max %.3e  FDE mean %.3e max %.3e  scenes with FDE>1e-3: %d/%d" %
           (kind, np.mean(ades), np.max(ades), np.mean(fdes), np.max(fdes), flips, B))
    # teacher-forced: neighbours follow the truth, only the primaries feed predictions back.  A
    # primary whose fed-back position sits within float rounding of a cell edge can land in the
    # other cell (SURVEY.md section 7 "chaotic sensitivity"); such scenes are counted, not hidden.
    d_tf = np.abs(pred_tf.cpu().numpy() - pred_tf_o)
    assert (np.isnan(d_tf) == np.isnan(pred_tf_o)).all()
    bad_tf = int((np.nanmax(d_tf, axis=(0, 2)) > TOL_POS).sum())
    report("%s: teacher-forced tracks off by > 1e-4 m: %d/%d, median %.2e, max %.2e" %
           (kind, bad_tf, M, np.nanmedian(d_tf), np.nanmax(d_tf)))
    assert bad_tf <= max(1, M // 100)
    assert np.nanmedian(d_tf) < 1e-6
    assert np.median(ades) < TOL_POS and np.median(fdes) < TOL_POS
    assert np.mean(ades) < TOL_POS and np.mean(fdes) < TOL_POS


def test_obs_length_two_and_short_horizon():
    """len(observed) == 2 seeds `positions` with observed[-1] (lstm.py:222-223)."""
    kind = "directional"
    xy, bs = O.synthetic_scenes(5, 6, seed=9)
    W = O.random_weights(kind, seed=2)
    model = build_model(kind, W)
    M = xy.shape[1]
    with torch.no_grad():
        rel, pred = model(torch.from_numpy(xy[7:9]), torch.zeros(M, 2), torch.from_numpy(bs), n_predict=4)
    rel_o, pred_o = O.forward(W, O.pool_config(kind), xy[7:9], bs, n_predict=4)
    assert maxdiff(rel, rel_o) < TOL_STEP * 5
    assert maxdiff(pred, pred_o) < TOL_STEP * 5
    assert pred.shape[0] == rel.shape[0] + 1


def test_single_pedestrian_scenes():
    """Nmax == 1: constant grid (gridbased_pooling.py:252-253)."""
    kind = "social_small"
    xy, bs = O.synthetic_scenes(1, 1, seed=4)
    W = O.random_weights(kind, seed=2)
    model = build_model(kind, W)
    with torch.no_grad():
        rel, pred = model(torch.from_numpy(xy[:9]), torch.zeros(1, 2), torch.from_numpy(bs), n_predict=12)
    rel_o, pred_o = O.forward(W, O.pool_config(kind), xy[:9], bs, n_predict=12)
    assert maxdiff(pred, pred_o) < TOL_POS


def test_full_size_properties_social():
    """BASELINE full size (B = 256, N = 20): size-independent properties instead of the oracle.
    (1) scenes are independent: the batched result equals per-shard results bit-for-bit
        (this is also what the multi-GPU sharding relies on);
    (2) determinism across repeated runs (the scatter is last-writer-wins, never atomic-add);
    (3) tracks absent at the last observed frame stay NaN for the whole free-running rollout
        (lstm.py:158)."""
    kind = "social"
    B, N = 256, 20
    xy, bs = O.synthetic_scenes(B, N, seed=77, nan_tracks=True)
    W = O.random_weights(kind, seed=8)
    model = build_model(kind, W)
    M = xy.shape[1]
    obs = torch.from_numpy(xy[:9]).cuda()
    with torch.no_grad():
        rel, pred = model(obs, torch.zeros(M, 2), torch.from_numpy(bs), n_predict=12)
        rel2, pred2 = model(obs, torch.zeros(M, 2), torch.from_numpy(bs), n_predict=12)
        half = B // 2
        cut = int(bs[half])
        rel_a, pred_a = model(obs[:, :cut].contiguous(), torch.zeros(cut, 2), torch.from_numpy(bs[:half + 1]), n_predict=12)
        rel_b, pred_b = model(obs[:, cut:].contiguous(), torch.zeros(M - cut, 2),
                              torch.from_numpy(bs[half:] - cut), n_predict=12)
    assert torch.equal(torch.nan_to_num(pred, nan=-1.0), torch.nan_to_num(pred2, nan=-1.0))
    both = torch.cat([pred_a, pred_b], dim=1)
    assert torch.equal(torch.nan_to_num(pred, nan=-1.0), torch.nan_to_num(both, nan=-1.0))
    gone = np.isnan(xy[8, :, 0])                 # absent at the last observed frame
    assert gone.any()
    assert torch.isnan(pred[7:, torch.from_numpy(gone).cuda()]).all()    # from encoder step (7, 8) onwards
    always = ~np.isnan(xy[:9, :, 0]).any(axis=0)
    assert not torch.isnan(pred[:, torch.from_numpy(always).cuda()]).any()
    # sanity vs the oracle on a 16-scene slice of the same batch (scene independence makes this valid)
    k = 16
    cutk = int(bs[k])
    _, pred_o = O.forward(W, O.pool_config(kind), xy[:9, :cutk], bs[:k + 1], n_predict=12)
    d = np.abs(pred[:, :cutk].cpu().numpy() - pred_o)
    assert (np.isnan(d) == np.isnan(pred_o)).all()
    assert np.nanmedian(d) < TOL_POS


def test_full_size_social_vs_oracle():
    """BASELINE configs[2] at its FULL size (256 scenes x 20 pedestrians, T = 9 + 12) against the numpy oracle:
    every track of every scene, not a slice.  Gate: ADE / FDE of the primaries and the worst track within
    1e-4 m; tracks that land in a different grid cell than the oracle (a boundary hit within float
    rounding) would show up as outliers and are counted."""
    kind = "social"
    B, N = 256, 20
    xy, bs = O.synthetic_scenes(B, N, seed=41, nan_tracks=True)
    W = O.random_weights(kind, seed=8)
    model = build_model(kind, W)
    M = xy.shape[1]
    with torch.no_grad():
        rel, pred = model(torch.from_numpy(xy[:9]).cuda(), torch.zeros(M, 2), torch.from_numpy(bs), n_predict=12)
    rel_o, pred_o = O.forward(W, O.pool_config(kind), xy[:9], bs, n_predict=12)
    pred = pred.cpu().numpy()
    assert (np.isnan(pred) == np.isnan(pred_o)).all()
    d = np.where(np.isnan(pred_o), 0.0, np.abs(pred - pred_o))
    per_track = d.max(axis=(0, 2))
    outliers = int((per_track > 1e-4).sum())
    prim = bs[:-1]
    err = np.linalg.norm((pred - pred_o)[-12:, prim], axis=2)          # [12, B] displacement error vs the oracle
    ade, fde = float(err.mean()), float(err[-1].mean())
    print("full-size social vs oracle: max %.2e m, tracks beyond 1e-4 m: %d of %d, ADE diff %.2e, FDE diff %.2e"
          % (float(d.max()), outliers, M, ade, fde))
    assert outliers == 0
    assert ade < 1e-4 and fde < 1e-4 and float(err.max()) < 1e-4


def test_predictor_boundary_roundtrip(tmp_path):
    """LSTMPredictor.__call__ / save / load (lstm.py:266-313) on the collision-test style scene."""
    from types import SimpleNamespace
    from trajnetplusplusbaselines_b200.data import TrackRow
    from trajnetplusplusbaselines_b200.lstm import LSTMPredictor
    kind = "directional"
    W = O.random_weights(kind, seed=12)
    model = build_model(kind, W)
    paths = [[TrackRow(f, 1, 0.1, 6.2 - 0.4 * (f - 1)) for f in range(1, 10)],
             [TrackRow(f, 2, 0.0, -6.2 + 0.4 * (f - 1)) for f in range(1, 10)],
             [TrackRow(f, 3, 1.0 + 0.1 * f, 2.0) for f in range(4, 10)]]
    predictor = LSTMPredictor(model)
    args = SimpleNamespace(normalize_scene=False)
    out = predictor(paths, np.zeros((3, 2)), n_predict=12, obs_length=9, modes=1, args=args)
    prim, neigh = out[0]
    assert prim.shape == (12, 2) and neigh.shape == (12, 2, 2)
    xy = np.full((9, 3, 2), np.nan, dtype=np.float32)
    for p, path in enumerate(paths):
        for r in path:
            xy[r.frame - 1, p] = (r.x, r.y)
    _, pred_o = O.forward(W, O.pool_config(kind), xy, [0, 3], n_predict=12)
    assert np.nanmax(np.abs(prim - pred_o[-12:, 0])) < TOL_POS
    # batched evaluator path: three scenes in one forward, each bit-identical to its single call
    paths_b = [[TrackRow(f, 7, 1.0 + 0.2 * f, -1.0) for f in range(1, 10)],
               [TrackRow(f, 8, 1.5, -2.0 + 0.3 * f) for f in range(1, 10)]]
    singles = [predictor(p, np.zeros((len(p), 2)), n_predict=12, obs_length=9, modes=1, args=args) for p in (paths, paths_b, paths)]
    batched = predictor.predict_batch([paths, paths_b, paths], n_predict=12, obs_length=9, args=args)
    for s_out, b_out in zip(singles, batched):
        assert np.array_equal(s_out[0][0], b_out[0][0]) and np.array_equal(s_out[0][1], b_out[0][1])
    fn = str(tmp_path / "model.pkl")
    predictor.save({"epoch": 1, "state_dict": model.state_dict()}, fn)
    again = LSTMPredictor.load(fn)
    out2 = again(paths, np.zeros((3, 2)), n_predict=12, obs_length=9, modes=1, args=args)
    assert np.array_equal(out2[0][0], prim)


def _large_scenes(sizes, seed=0):
    rng = np.random.RandomState(seed)
    xs = []
    for n in sizes:
        p0 = rng.randn(n, 2) * 3.0
        xs.append(p0[None] + np.cumsum(rng.randn(21, n, 2) * 0.3, axis=0))
    xy = np.concatenate(xs, axis=1).astype(np.float32)
    xy[:4, 5] = np.nan                      # a late entry and an early exit inside the big scene
    xy[12:, 7] = np.nan
    return xy, np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["social", "directional"])
def test_large_scenes_take_the_fallback_kernels(kind):
    """Scenes far beyond the BASELINE size (90 and 40 pedestrians next to a 3-pedestrian one): the
    grouping / shared-memory budgets of the tensor-core kernels no longer fit and the warp-level /
    FFMA kernels take over; results still match the oracle within the 1e-4 m gate."""
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling
    xy, bs = _large_scenes([90, 3, 40])
    W = O.random_weights(kind, seed=4)
    rel_o, pred_o = O.forward(W, O.pool_config(kind), xy[:9], bs, n_predict=12)
    model = LSTM(pool=GridBasedPooling(**O.MODEL_SPECS[kind]))
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in W.items()})
    model = model.cuda().eval()
    with torch.no_grad():
        rel, pred = model(torch.from_numpy(xy[:9]), torch.zeros(xy.shape[1], 2), torch.from_numpy(bs), n_predict=12)
    rel, pred = rel.numpy(), pred.numpy()
    assert (np.isnan(pred) == np.isnan(pred_o)).all()
    assert np.nanmax(np.abs(pred - pred_o)) < 1e-4
    assert np.nanmax(np.abs(rel - rel_o)) < 1e-4


@pytest.mark.gpu
def test_evaluate_file_batched_equals_per_scene(tmp_path):
    """ndjson -> chunks of scenes through one forward each -> ndjson; same numbers as calling the
    predictor scene by scene like lstm/trajnet_evaluator.py:15-19."""
    import types
    from trajnetplusplusbaselines_b200.data import SceneRow, TrackRow, read_ndjson_scenes, trajnet_line
    from trajnetplusplusbaselines_b200.evaluator import evaluate_file, load_test_scenes
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling, LSTMPredictor
    # ragged scenes: predict_batch uses the per-scene layout (tb2_layout_set_padding(0)), so the padded slots
    # of a batched reference call (which clobber grid cell 0, gridbased_pooling.py:281-293) do not appear
    xy, bs = O.synthetic_scenes(12, 6, seed=31, ragged=True)
    infile, outfile = os.path.join(tmp_path, "in.ndjson"), os.path.join(tmp_path, "out.ndjson")
    with open(infile, "w") as f:
        for b in range(len(bs) - 1):
            f0 = 1000 * b                  # scenes are told apart by their frame range, as in DATA_BLOCK
            f.write(trajnet_line(SceneRow(b, 100 * b, f0, f0 + 200, 2.5, 0)) + "\n")
            for p in range(bs[b], bs[b + 1]):
                for t in range(21):
                    f.write(trajnet_line(TrackRow(f0 + 10 * t, 100 * b + int(p - bs[b]), float(xy[t, p, 0]),
                                                  float(xy[t, p, 1]))) + "\n")
    W = O.random_weights("directional", seed=8)
    model = LSTM(pool=GridBasedPooling(**O.MODEL_SPECS["directional"]))
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in W.items()})
    predictor = LSTMPredictor(model.cuda())
    args = types.SimpleNamespace(normalize_scene=False)
    assert evaluate_file(predictor, infile, outfile, chunk=5, args=args) == len(bs) - 1
    got = {sid: paths for sid, paths in read_ndjson_scenes(outfile)}
    for _, sid, paths in load_test_scenes(infile):
        single = predictor(paths, np.zeros((len(paths), 2)), n_predict=12, obs_length=9, args=args)[0]
        assert np.allclose([[r.x, r.y] for r in got[sid][0]], np.round(single[0], 2), atol=0.011)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["social", "occupancy"])
def test_per_scene_layout_equals_single_scene_calls(kind):
    """Ragged batch with tb2_layout_set_padding(0) == every scene forwarded alone, bit for bit; with the
    default (trainer) padding the small scenes see the padded slots, as in the reference's batched call."""
    from trajnetplusplusbaselines_b200.lstm import LSTM, GridBasedPooling
    xy, bs = O.synthetic_scenes(10, 9, seed=77, ragged=True, nan_tracks=True)
    xy[:, :, :] = xy * 1.6                 # spread: more neighbours out of range / in the corner cell
    W = O.random_weights(kind, seed=12)
    model = LSTM(pool=GridBasedPooling(**O.MODEL_SPECS[kind]))
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in W.items()})
    model = model.cuda().eval()
    obs = torch.from_numpy(xy[:9]).cuda()
    with torch.no_grad():
        _, batched = model._forward_nograd(obs, torch.from_numpy(bs), None, 12, pad_to_batch_max=False)
        batched = batched.cpu().numpy()
        for b in range(len(bs) - 1):
            sl = slice(int(bs[b]), int(bs[b + 1]))
            _, single = model(obs[:, sl].contiguous(), torch.zeros(sl.stop - sl.start, 2),
                              torch.tensor([0, sl.stop - sl.start]), n_predict=12)
            a, c = batched[:, sl], single.cpu().numpy()
            assert (np.isnan(a) == np.isnan(c)).all()
            assert np.array_equal(np.nan_to_num(a), np.nan_to_num(c)), b
    # and the oracle agrees scene by scene
    b = int(np.argmin(np.diff(bs)))
    sl = slice(int(bs[b]), int(bs[b + 1]))
    _, pred_o = O.forward(W, O.pool_config(kind), xy[:9, sl], np.array([0, sl.stop - sl.start]), n_predict=12)
    assert np.nanmax(np.abs(batched[:, sl] - pred_o)) < 1e-4
