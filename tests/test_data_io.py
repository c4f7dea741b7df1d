"""ndjson boundary (SURVEY.md 8f rank 1): reader / writer either side of the batched predictor."""
import json
import os

import numpy as np
import pytest

from trajnetplusplusbaselines_b200.data import (SceneRow, TrackRow, paths_to_xy, preprocess_test,
                                                read_ndjson_scenes, trajnet_line, write_predictions)


def _scene(scene_id, n_peds, start, rng):
    paths = []
    for p in range(n_peds):
        x0 = rng.randn(2)
        paths.append([TrackRow(start + 10 * t, 100 * scene_id + p, float(x0[0] + 0.1 * t), float(x0[1] - 0.05 * t))
                      for t in range(21)])
    return paths


def test_writer_matches_data_block_line_format():
    # the two record kinds exactly as they appear in the reference's DATA_BLOCK/*.ndjson
    assert json.loads(trajnet_line(SceneRow(3, 7, 10, 210, 2.5, 0))) == \
        {"scene": {"id": 3, "p": 7, "s": 10, "e": 210, "fps": 2.5, "tag": 0}}
    assert json.loads(trajnet_line(TrackRow(10, 7, 1.23456, -2.5))) == {"track": {"f": 10, "p": 7, "x": 1.23, "y": -2.5}}
    assert json.loads(trajnet_line(TrackRow(10, 7, 1.0, 2.0, 0, 3)))["track"]["prediction_number"] == 0


def test_write_then_read_round_trip(tmp_path):
    rng = np.random.RandomState(0)
    scenes = [("file", sid, _scene(sid, n, 1000 * sid, rng)) for sid, n in ((1, 3), (2, 1), (5, 4))]
    preds = []
    for _, _, paths in scenes:
        K = len(paths) - 1
        prim = rng.randn(12, 2)
        neigh = rng.randn(12, K, 2) if K else []
        preds.append({0: [prim, neigh]})
    fn = os.path.join(tmp_path, "pred.ndjson")
    write_predictions(preds, scenes, fn, obs_length=9, pred_length=12)
    got = {sid: paths for sid, paths in read_ndjson_scenes(fn)}
    assert sorted(got) == [1, 2, 5]
    for (_, sid, paths), pred in zip(scenes, preds):
        back = got[sid]
        assert back[0][0].pedestrian == paths[0][0].pedestrian            # primary first
        assert len(back) == len(paths)
        assert [r.frame for r in back[0]] == [paths[0][8].frame + 10 * (k + 1) for k in range(12)]
        assert np.allclose([[r.x, r.y] for r in back[0]], np.round(pred[0][0], 2))
        by_id = {p[0].pedestrian: p for p in back[1:]}
        for n, path in enumerate(paths[1:]):
            assert np.allclose([[r.x, r.y] for r in by_id[path[0].pedestrian]], np.round(pred[0][1][:, n], 2))


def test_preprocess_test_drops_late_tracks():
    rng = np.random.RandomState(1)
    paths = _scene(1, 3, 0, rng)
    paths[2] = [r for r in paths[2] if r.frame >= 100]        # appears after the 9 observed frames
    out = preprocess_test(paths, 9)
    assert len(out) == 2 and all(r.frame <= 80 for p in out for r in p)
    assert paths_to_xy(out).shape == (9, 2, 2)


class _ConstantVelocity:
    """Stand-in with the reference's predictor call signature (CPU, no CUDA)."""

    def __call__(self, paths, scene_goal, n_predict=12, modes=1, predict_all=True, obs_length=9, start_length=0,
                 args=None):
        xy = paths_to_xy(paths)
        v = xy[obs_length - 1] - xy[obs_length - 2]
        pred = xy[obs_length - 1][None] + np.arange(1, n_predict + 1)[:, None, None] * v[None]
        return {0: [pred[:, 0], pred[:, 1:]]}


def test_evaluate_file_ndjson_in_ndjson_out(tmp_path):
    """load_test_scenes -> predict_scenes -> write_predictions on a file written in the DATA_BLOCK format."""
    from trajnetplusplusbaselines_b200.evaluator import evaluate_file, load_test_scenes
    rng = np.random.RandomState(2)
    infile, outfile = os.path.join(tmp_path, "in.ndjson"), os.path.join(tmp_path, "out.ndjson")
    truth = {}
    with open(infile, "w") as f:
        for sid, n in ((0, 3), (1, 2)):
            paths = _scene(sid, n, 5000 * sid, rng)
            late = [TrackRow(5000 * sid + 10 * t, 100 * sid + 50, 0.0, 0.1 * t) for t in range(12, 21)]   # enters after obs
            f.write(trajnet_line(SceneRow(sid, paths[0][0].pedestrian, paths[0][0].frame, paths[0][-1].frame, 2.5, 0)) + "\n")
            for p in paths + [late]:
                for r in p:
                    f.write(trajnet_line(r) + "\n")
            truth[sid] = paths
    scenes = load_test_scenes(infile, obs_length=9)
    assert [len(paths) for _, _, paths in scenes] == [3, 2]              # the late track is dropped
    assert all(len(p) == 9 for _, _, paths in scenes for p in paths)     # only the observed frames remain
    assert evaluate_file(_ConstantVelocity(), infile, outfile) == 2
    got = {sid: paths for sid, paths in read_ndjson_scenes(outfile)}
    for sid, paths in truth.items():
        xy = paths_to_xy(paths)
        v = xy[8, 0] - xy[7, 0]
        want = np.round(xy[8, 0][None] + np.arange(1, 13)[:, None] * v[None], 2)
        # the ndjson rows carry two decimals: compare in hundredths; a value within float rounding of x.xx5 may
        # round the other way, those entries are counted
        units = np.rint(np.abs(np.array([[r.x, r.y] for r in got[sid][0]]) - want) * 100).astype(int)
        assert units.max() <= 1 and int((units > 0).sum()) <= 1, units


def test_get_predictions_writes_one_file_per_dataset(tmp_path):
    """Directory layout of lstm/trajnet_evaluator.get_predictions: <root>/test/*.ndjson ->
    <root>/test_pred/<model>_modes<k>/<dataset>.ndjson; an existing model folder is skipped."""
    import types
    from trajnetplusplusbaselines_b200.evaluator import get_predictions
    rng = np.random.RandomState(4)
    test_dir = os.path.join(tmp_path, "test")
    os.makedirs(test_dir)
    for name, sids in (("a.ndjson", (0, 1)), ("b.ndjson", (2,))):
        with open(os.path.join(test_dir, name), "w") as f:
            for sid in sids:
                paths = _scene(sid, 3, 3000 * sid, rng)
                f.write(trajnet_line(SceneRow(sid, paths[0][0].pedestrian, paths[0][0].frame, paths[0][-1].frame, 2.5, 0)) + "\n")
                for p in paths:
                    for r in p:
                        f.write(trajnet_line(r) + "\n")
    args = types.SimpleNamespace(path=os.path.join(tmp_path, "test_pred") + os.sep, output=["models/cv.pkl"], modes=1,
                                 obs_length=9, pred_length=12, chunk=2, normalize_scene=False)
    os.makedirs(args.path)
    assert get_predictions(args, load_predictor=lambda fn: _ConstantVelocity()) == {"cv_modes1": 3}
    out_dir = os.path.join(args.path, "cv_modes1")
    assert sorted(os.listdir(out_dir)) == ["a.ndjson", "b.ndjson"]
    assert len(list(read_ndjson_scenes(os.path.join(out_dir, "a.ndjson")))) == 2
    assert get_predictions(args, load_predictor=lambda fn: _ConstantVelocity()) == {}      # skipped: already there


def test_fast_writer_is_byte_identical_to_the_line_writer(tmp_path):
    """write_predictions formats track rows directly; the text must equal trajnet_line row by row, also for
    negative zero, integral values, rounding ties and NaN neighbours."""
    rng = np.random.RandomState(7)
    scenes = [("f", 3, _scene(3, 4, 700, rng))]
    prim = rng.randn(12, 2) * 30
    prim[0] = (-0.0, 2.0)
    prim[1] = (0.125, -0.375)
    prim[2] = (1e-9, 123456.789)
    neigh = rng.randn(12, 3, 2)
    neigh[5:, 1] = np.nan
    fn = os.path.join(tmp_path, "p.ndjson")
    write_predictions([{0: [prim, neigh]}], scenes, fn)
    lines = open(fn).read().splitlines()
    first = scenes[0][2][0][8].frame + 10
    want = [trajnet_line(SceneRow(3, scenes[0][2][0][0].pedestrian, 700, 700 + 200, 2.5, 0))]
    want += [trajnet_line(TrackRow(first + 10 * i, scenes[0][2][0][0].pedestrian, prim[i, 0], prim[i, 1], 0, 3)) for i in range(12)]
    for n in range(3):
        want += [trajnet_line(TrackRow(first + 10 * j, scenes[0][2][n + 1][0].pedestrian, neigh[j, n, 0], neigh[j, n, 1], 0, 3))
                 for j in range(12)]
    assert lines == want


def test_paths_to_xy_contract():
    """trajnetplusplustools.Reader.paths_to_xy semantics: frames = sorted set of the primary's frames, pedestrians
    without a row in those frames are dropped, rows outside them ignored; rows may be plain objects with attributes."""
    import types
    from trajnetplusplusbaselines_b200.data import TrackRow, paths_to_xy
    primary = [TrackRow(30, 1, 3.0, 3.5), TrackRow(10, 1, 1.0, 1.5), TrackRow(20, 1, 2.0, 2.5)]     # unsorted on purpose
    other = [TrackRow(20, 2, 7.0, 7.5), TrackRow(40, 2, 9.0, 9.5)]                                  # frame 40 is outside
    ghost = [TrackRow(50, 3, 0.0, 0.0)]                                                            # never inside: dropped
    xy = paths_to_xy([primary, other, ghost])
    assert xy.shape == (3, 2, 2) and xy.dtype == np.float64 and xy.flags["C_CONTIGUOUS"]
    assert xy[:, 0].tolist() == [[1.0, 1.5], [2.0, 2.5], [3.0, 3.5]]
    assert np.isnan(xy[0, 1]).all() and xy[1, 1].tolist() == [7.0, 7.5] and np.isnan(xy[2, 1]).all()
    rows = [[types.SimpleNamespace(frame=r.frame, pedestrian=r.pedestrian, x=r.x, y=r.y) for r in path]
            for path in (primary, other, ghost)]
    assert np.array_equal(np.isnan(paths_to_xy(rows)), np.isnan(xy)) and np.nanmax(np.abs(paths_to_xy(rows) - xy)) == 0.0


# --------------------------------------------------------------------------------------------------------------
# Column pipeline (native ndjson passes, data.load_test_scenes_xy / write_predictions_xy) against the row pipeline,
# which is the definition: equal arrays, equal metadata, byte-identical output files.
# --------------------------------------------------------------------------------------------------------------
def _rows_reference(filename, obs_length=9):
    from trajnetplusplusbaselines_b200.data import _scene_meta_from_paths
    out = []
    for sid, paths in read_ndjson_scenes(filename):
        paths = preprocess_test(paths, obs_length)
        out.append((paths_to_xy(paths), _scene_meta_from_paths(sid, paths, obs_length), paths))
    return out


def _assert_pipelines_agree(filename, obs_length=9, expect_native=True):
    from trajnetplusplusbaselines_b200.data import load_test_scenes_xy, parse_ndjson_columns
    assert (parse_ndjson_columns(filename) is not None) == expect_native
    cols = load_test_scenes_xy(filename, obs_length)
    rows = _rows_reference(filename, obs_length)
    assert len(cols) == len(rows)
    for (xy_c, meta_c), (xy_r, meta_r, _) in zip(cols, rows):
        assert xy_c.dtype == xy_r.dtype == np.float64 and xy_c.shape == xy_r.shape
        assert np.array_equal(xy_c, xy_r, equal_nan=True)
        assert meta_c == meta_r and all(type(v) is int for v in meta_c[:5]) and all(type(v) is int for v in meta_c.neigh_ids)
    return cols, rows


def _tricky_file(filename, seed=0):
    """Overlapping scenes that share tracks (sliding windows), late / leaving / off-grid pedestrians, a scene without its
    primary, shuffled keys, integer and exponent coordinates, NaN literals, blank lines, CRLF."""
    rng = np.random.RandomState(seed)
    lines = []
    peds = {}
    for p in range(14):
        t0, t1 = sorted(rng.choice(60, 2, replace=False))
        if p < 3:
            t0, t1 = 0, 59
        peds[p] = (t0, max(t1, t0 + 1))
    for t in range(60):
        for p, (t0, t1) in peds.items():
            if t0 <= t <= t1:
                x, y = rng.randn() * 4, rng.randn() * 4
                style = rng.randint(6)
                if style == 0:
                    lines.append('{"track": {"p": %d, "y": %r, "x": %r, "f": %d}}' % (p, y, x, 10 * t))           # shuffled keys
                elif style == 1:
                    lines.append('{"track":{"f":%d,"p":%d,"x":%d,"y":%.3e}}' % (10 * t, p, int(x), y))           # int / exponent, no spaces
                elif style == 2:
                    lines.append('  {"track": {"f": %d, "p": %d, "x": %r, "y": %r, "prediction_number": 0, "scene_id": 3}}  ' % (10 * t, p, x, y))
                else:
                    lines.append(trajnet_line(TrackRow(10 * t, p, x, y)))
        if t == 20:
            lines.append('{"track": {"f": 205, "p": 77, "x": 1.0, "y": 2.0}}')         # only between the primary's frames
            lines.append('{"track": {"f": 200, "p": 5, "x": NaN, "y": -Infinity}}')    # json.loads accepts these
            lines.append('')
    sid = 0
    for start in range(0, 40, 4):
        long_enough = [p for p, (t0, t1) in peds.items() if p >= 3 and t0 <= start and t1 >= start + 9]
        for primary in [0, 1, 2] + long_enough[:2]:
            lines.insert(rng.randint(len(lines)), trajnet_line(SceneRow(sid, primary, 10 * start, 10 * (start + 20), 2.5, 0)))
            sid += 1
    lines.append('{"scene": {"id": 999, "p": 4242, "s": 0, "e": 100, "fps": 2.5, "tag": [3, [2], {"k": "v"}]}}')   # primary has no rows; nested tag as in DATA_BLOCK
    with open(filename, "w", newline="") as f:
        f.write("\r\n".join(lines) + "\n")


def test_column_pipeline_equals_row_pipeline(tmp_path):
    from trajnetplusplusbaselines_b200.data import write_predictions_xy
    fn = os.path.join(tmp_path, "tricky.ndjson")
    rng = np.random.RandomState(5)
    for seed in range(4):
        _tricky_file(fn, seed)
        cols, rows = _assert_pipelines_agree(fn)
        assert len(cols) >= 30 and any(xy.shape[1] - 1 != len(m.neigh_ids) for xy, m in cols)     # incl. a dropped pedestrian
        preds = []
        for xy, meta in cols:
            k = xy.shape[1] - 1
            prim = rng.randn(12, 2) * 50
            neigh = rng.randn(12, k, 2) * 50
            if k:
                neigh[rng.randint(12):, rng.randint(k)] = np.nan                     # a neighbour that vanished
            preds.append({0: [prim, neigh if k else []]})
        a, b = os.path.join(tmp_path, "a.ndjson"), os.path.join(tmp_path, "b.ndjson")
        for fn_out in (a, b):
            if os.path.exists(fn_out):
                os.remove(fn_out)
        write_predictions(preds, [("f", m.scene_id, paths) for _, m, paths in rows], a)
        write_predictions_xy(preds, [m for _, m in cols], b)
        assert open(a, "rb").read() == open(b, "rb").read()


def test_native_parser_refuses_what_it_is_not_sure_about(tmp_path):
    """Anything outside the plain format sends the WHOLE file through json.loads: same results either way."""
    from trajnetplusplusbaselines_b200.data import load_test_scenes_xy, parse_ndjson_columns
    rng = np.random.RandomState(1)
    base = [trajnet_line(SceneRow(0, 1, 0, 200, 2.5, 0))]
    for p in (1, 2):
        base += [trajnet_line(TrackRow(10 * t, p, rng.randn(), rng.randn())) for t in range(21)]
    odd_lines = [
        '{"scene": {"id": 5, "p": 1, "s": 0, "e": 200, "fps": 2.5, "tag": "a\\"b"}}',     # escape in a string
        '{"scene": {"id": 5, "p": 1, "s": 0, "e": 200, "fps": 2.5, "tag": [1, "a\\b"]}}',  # escape inside a nested value
        '{"track": {"f": 10.0, "p": 2, "x": 0.5, "y": 0.5}}',                              # float frame stays a float in Python
        '{"track": {"f": 10, "p": 2, "x": 0.5, "y": 0.5}, "extra": 1}',                    # a second top-level key
        '{"info": {"a": 1}}',                                                              # unknown record type
        '{"track": {"f": 123456789012345678901234567890, "p": 2, "x": 0.5, "y": 0.5}}',    # beyond int64
    ]
    fn = os.path.join(tmp_path, "odd.ndjson")
    for odd in odd_lines:
        with open(fn, "w") as f:
            f.write("\n".join(base + [odd]) + "\n")
        assert parse_ndjson_columns(fn) is None, odd
        _assert_pipelines_agree(fn, expect_native=False)
    with open(fn, "w") as f:                                                               # a missing field raises in both
        f.write("\n".join(base + ['{"track": {"f": 10, "p": 2, "x": 0.5}}']) + "\n")
    assert parse_ndjson_columns(fn) is None
    with pytest.raises(KeyError):
        load_test_scenes_xy(fn)
    with open(fn, "w") as f:                                                               # a nested value where a number belongs
        f.write("\n".join(base + ['{"track": {"f": 10, "p": 2, "x": [0.5], "y": 0.5}}']) + "\n")
    assert parse_ndjson_columns(fn) is None
    with pytest.raises(ValueError):
        load_test_scenes_xy(fn)
    with open(fn, "w") as f:                                                               # the primary leaves before obs_length rows
        f.write("\n".join([base[0]] + base[1:6] + base[22:]) + "\n")
    assert parse_ndjson_columns(fn) is not None
    with pytest.raises(IndexError):
        load_test_scenes_xy(fn)
    with pytest.raises(IndexError):
        _rows_reference(fn)
    with open(fn, "w") as f:                                                               # empty file
        pass
    assert load_test_scenes_xy(fn) == []


def test_native_writer_formats_like_json_dumps(tmp_path):
    """Coordinates: round(v, 2) printed like repr -- rounding ties of the binary value, negative zero, integral values,
    NaN / infinities, large and tiny magnitudes; 200 k random values."""
    from trajnetplusplusbaselines_b200.data import SceneMeta, write_predictions_xy
    rng = np.random.RandomState(3)
    special = np.array([0.0, -0.0, 0.005, -0.005, 0.015, 0.025, 1.005, 2.675, 1.0, -1.0, 10.0, 100.5, 0.1, 0.01, -0.01, 0.004999,
                        1e-9, -1e-9, 123456.785, 99999999.995, 1e12 + 0.125, -8.5e14, np.nan, np.inf, -np.inf, 0.994999, 0.995,
                        1.999, 9.995, 9.994999999999999])
    vals = np.concatenate([special, rng.randn(100000) * 30, np.round(rng.randn(50000) * 30, 3), rng.randint(-5000, 5000, 50000) / 200.0,
                           rng.randn(2000) * 1e9])
    vals = vals[:len(vals) // 24 * 24].reshape(-1, 12, 2)                # scenes of 12 frames, primary only
    preds = [{0: [v, []]} for v in vals]
    rows = [("f", i, [[TrackRow(10 * t, 7 + i, 0.0, 0.0) for t in range(9)]]) for i in range(len(vals))]
    metas = [SceneMeta(i, 7 + i, 0, 10, 80, []) for i in range(len(vals))]
    a, b = os.path.join(tmp_path, "a.ndjson"), os.path.join(tmp_path, "b.ndjson")
    write_predictions(preds, rows, a)
    write_predictions_xy(preds, metas, b)
    ta, tb = open(a, "rb").read(), open(b, "rb").read()
    if ta != tb:
        for la, lb in zip(ta.split(b"\n"), tb.split(b"\n")):
            assert la == lb
    assert ta == tb
    with pytest.raises(RuntimeError):                                   # finite and >= 1e15: repr() would use an exponent
        write_predictions_xy([{0: [np.full((12, 2), 3e15), []]}], metas[:1], b)


class _ArrayConstantVelocity(_ConstantVelocity):
    """The stand-in with the array entry point: evaluate_file takes the column pipeline for it."""

    def predict_batch_xy(self, xys, scene_goals=None, n_predict=12, obs_length=9, start_length=0, args=None):
        out = []
        for xy in xys:
            v = xy[obs_length - 1] - xy[obs_length - 2]
            pred = xy[obs_length - 1][None] + np.arange(1, n_predict + 1)[:, None, None] * v[None]
            out.append({0: [pred[:, 0], pred[:, 1:]]})
        return out


def test_evaluate_file_column_pipeline_writes_the_same_file(tmp_path):
    from trajnetplusplusbaselines_b200.evaluator import evaluate_file
    fn = os.path.join(tmp_path, "in.ndjson")
    rng = np.random.RandomState(8)
    with open(fn, "w") as f:
        for sid, n in enumerate((3, 1, 7, 2, 5)):
            paths = _scene(sid, n, 4000 * sid, rng)
            late = [TrackRow(4000 * sid + 10 * t, 100 * sid + 60, 0.3, 0.1 * t) for t in range(5, 21)]     # enters mid-observation
            f.write(trajnet_line(SceneRow(sid, paths[0][0].pedestrian, paths[0][0].frame, paths[0][-1].frame, 2.5, 0)) + "\n")
            for p in paths + [late]:
                for r in p:
                    f.write(trajnet_line(r) + "\n")
    a, b, c = (os.path.join(tmp_path, name) for name in ("rows.ndjson", "cols.ndjson", "cols_sharded.ndjson"))
    assert evaluate_file(_ConstantVelocity(), fn, a) == 5
    assert evaluate_file(_ArrayConstantVelocity(), fn, b, chunk=2) == 5
    assert open(a, "rb").read() == open(b, "rb").read()
    for rank in (1, 0):
        evaluate_file(_ArrayConstantVelocity(), fn, c, chunk=2, rank=rank, world_size=2)
    assert open(c, "rb").read() == open(a, "rb").read()


def _data_block_files(tmp_path, subdir=""):
    """The sample of every ndjson file the reference ships in DATA_BLOCK (tests/golden/data_block_sample.npz, made by
    oracle/make_reference_golden.py), written back as files."""
    from oracle.make_reference_golden import DATA_BLOCK_SAMPLE
    files = []
    with np.load(DATA_BLOCK_SAMPLE) as sample:
        for name in sorted(sample.files):
            if name.startswith(subdir):
                fn = os.path.join(tmp_path, name.replace("/", "__"))
                sample[name].tofile(fn)
                files.append(fn)
    return files


def test_column_pipeline_on_the_reference_data_block(tmp_path):
    """Every ndjson file the reference ships (DATA_BLOCK): the native parser takes it and both pipelines agree."""
    files = _data_block_files(tmp_path)
    assert len(files) == 9
    for fn in files:
        try:
            rows = _rows_reference(fn)
        except IndexError:
            continue                        # training files hold scenes shorter than the test protocol assumes
        _assert_pipelines_agree(fn)
        assert rows


def test_native_parser_reads_numbers_like_float(tmp_path):
    """Coordinates bit for bit as json.loads reads them: the exact-division fast path (short decimals) and the strtod path
    (long mantissas, exponents, subnormals) against float(str)."""
    import random
    from trajnetplusplusbaselines_b200.data import parse_ndjson_columns
    rng = random.Random(5)
    lits = []
    for _ in range(60000):
        k = rng.randint(0, 22)
        digits = str(rng.randint(0, 10 ** rng.randint(1, 15)))
        sign = '-' if rng.random() < 0.3 else ''
        if k == 0:
            lits.append(sign + digits + '.0')
        else:
            digits = digits.rjust(k + 1, '0')
            lits.append(sign + digits[:-k] + '.' + digits[-k:])
    lits += [repr(rng.gauss(0, 1) * 10 ** rng.randint(-8, 8)) for _ in range(40000)]
    lits += ['0.0', '-0.0', '0.10', '0.000000000000000000001', '123456789012345.67', '1234567890123456.7', '0.30000000000000004',
             '1e5', '1.5e-7', '-2.5E+3', '5e-324', '1.7976931348623157e308', '0.000', '100000000000000.0', '99999999999999.99', '7']
    fn = os.path.join(tmp_path, "numbers.ndjson")
    with open(fn, "w") as f:
        for i in range(0, len(lits) - 1, 2):
            f.write('{"track": {"f": %d, "p": 1, "x": %s, "y": %s}}\n' % (i, lits[i], lits[i + 1]))
    cols = parse_ndjson_columns(fn)
    assert cols is not None and len(cols['x']) == len(lits) // 2
    want_x = np.array([float(lits[2 * i]) for i in range(len(cols['x']))])
    want_y = np.array([float(lits[2 * i + 1]) for i in range(len(cols['y']))])
    assert np.array_equal(cols['x'].view(np.int64), want_x.view(np.int64))
    assert np.array_equal(cols['y'].view(np.int64), want_y.view(np.int64))


def _assert_whole_scenes_agree(filename):
    from trajnetplusplusbaselines_b200.data import load_scenes_xy
    cols = load_scenes_xy(filename)
    rows = [(sid, paths_to_xy(paths)) for sid, paths in read_ndjson_scenes(filename)]
    assert len(cols) == len(rows)
    for (sid_c, xy_c), (sid_r, xy_r) in zip(cols, rows):
        assert sid_c == sid_r and xy_c.shape == xy_r.shape and np.array_equal(xy_c, xy_r, equal_nan=True)
    return len(cols)


def test_whole_scene_loader_equals_paths_to_xy(tmp_path):
    """load_scenes_xy (training files: every scene over its whole frame range) == paths_to_xy of the row reader."""
    fn = os.path.join(tmp_path, "tricky.ndjson")
    for seed in range(3):
        _tricky_file(fn, seed)
        assert _assert_whole_scenes_agree(fn) >= 30


def test_whole_scene_loader_on_the_reference_training_files(tmp_path):
    files = _data_block_files(tmp_path, "trajdata/train/")
    assert len(files) == 7
    assert sum(_assert_whole_scenes_agree(fn) for fn in files) == 292        # every scene of the sample


def test_native_format_reports_the_size_it_needs():
    """tb2_ndjson_format: the byte count is returned whatever the capacity; nothing is written past it."""
    import ctypes
    from trajnetplusplusbaselines_b200 import _lib
    lib = _lib.load()
    i64 = lambda *v: np.array(v, dtype=np.int64)
    sid, sped, ss, se, nrows = i64(3), i64(12), i64(100), i64(300), i64(2)
    fr, pd, md = i64(190, 200), i64(12, 12), i64(0, 0)
    x, y = np.array([1.005, -0.0]), np.array([np.nan, 2.5])
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)
    args = (1, ptr(sid), ptr(sped), ptr(ss), ptr(se), ptr(nrows), ptr(fr), ptr(pd), ptr(x), ptr(y), ptr(md))
    need = lib.tb2_ndjson_format(*args, ctypes.c_void_p(0), 0)
    want = ('{"scene": {"id": 3, "p": 12, "s": 100, "e": 300, "fps": 2.5, "tag": 0}}\n'
            '{"track": {"f": 190, "p": 12, "x": 1.0, "y": NaN, "prediction_number": 0, "scene_id": 3}}\n'
            '{"track": {"f": 200, "p": 12, "x": -0.0, "y": 2.5, "prediction_number": 0, "scene_id": 3}}\n')
    assert need == len(want)
    buf = ctypes.create_string_buffer(need + 8)
    buf.raw = b"#" * (need + 8)
    assert lib.tb2_ndjson_format(*args, ctypes.cast(buf, ctypes.c_void_p), need) == need
    assert buf.raw[:need].decode() == want and buf.raw[need:] == b"#" * 8
    small = ctypes.create_string_buffer(b"#" * 40, 40)
    assert lib.tb2_ndjson_format(*args, ctypes.cast(small, ctypes.c_void_p), 40) == need      # too small: size only
    assert small.raw == b"#" * 40
