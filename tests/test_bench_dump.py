"""CPU: bench.py --dump-outputs writes what a pipeline step returned, as float arrays that are equal for equal results."""
import os

import numpy as np

import bench
import adas_b200  # noqa: F401
from adas_b200 import _capi
from adas_b200.pipeline import StepResult


def _step(seed, B=6, max_det=300, max_pts=81):
    rng = np.random.default_rng(seed)
    counts = np.array([0, 3, 300, 7, 1, 12][:B], np.int32)
    npts = rng.integers(0, max_pts + 1, (B, 4)).astype(np.int32)
    # rows past the counts are unset memory in a real step: fill them with noise that must not reach the files
    y = (rng.standard_normal((B, max_det, 4)).astype(np.float32), rng.random((B, max_det)).astype(np.float32),
         rng.integers(-99, 99, (B, max_det)).astype(np.int32), rng.integers(-99, 99, (B, max_det)).astype(np.int32), counts,
         rng.integers(0, 500, B).astype(np.int32))
    u = (rng.integers(-9, 2000, (B, 4, max_pts, 2)).astype(np.int32), npts, rng.integers(0, 2, (B, 4)).astype(np.uint8), None)
    r = StepResult(y, u)
    r.tracks = []
    for b in range(B):
        t = np.zeros(int(counts[b]) % 5, _capi.TRACK_DTYPE)
        t["track_id"] = np.arange(len(t)) + 10 * b
        t["tlwh"] = rng.random((len(t), 4))
        r.tracks.append(t)
    return r


def _clean(r, b):
    n, k = int(r.counts[b]), r.lane_npts[b]
    return (r.boxes[b, :n], r.scores[b, :n], r.class_ids[b, :n], r.cand_index[b, :n], [r.lane_pts[b, l, :k[l]] for l in range(4)])


def test_dump_is_float_masked_and_complete(tmp_path):
    r = _step(0)
    out = bench.dump_outputs(r, str(tmp_path / "d"))
    files = sorted(os.listdir(tmp_path / "d"))
    assert files == sorted(n + ".npy" for n in out)
    for name in out:
        a = np.load(tmp_path / "d" / (name + ".npy"))
        assert a.dtype in (np.float32, np.float64), name
        assert np.array_equal(a, out[name])
    assert np.array_equal(out["frame_index"], np.arange(6))
    assert np.array_equal(out["det_counts"], r.counts) and np.array_equal(out["lane_npts"], r.lane_npts)
    for b in range(6):
        n = int(r.counts[b])
        boxes, scores, cls, cand, lanes = _clean(r, b)
        assert np.array_equal(out["det_boxes"][b, :n], boxes) and not out["det_boxes"][b, n:].any()
        assert np.array_equal(out["det_scores"][b, :n], scores) and np.array_equal(out["det_class_ids"][b, :n], cls)
        assert np.array_equal(out["det_cand_index"][b, :n], cand) and (out["det_cand_index"][b, n:] == -1).all()
        for l in range(4):
            k = int(r.lane_npts[b, l])
            assert np.array_equal(out["lane_pts"][b, l, :k], lanes[l]) and not out["lane_pts"][b, l, k:].any()
    assert out["tracks"].shape == (sum(len(t) for t in r.tracks), 27)
    assert np.array_equal(out["track_counts"], [len(t) for t in r.tracks])
    assert np.array_equal(out["tracks"][:, 0], np.concatenate([t["track_id"] for t in r.tracks]))


def test_dump_depends_only_on_the_results(tmp_path):
    """Two steps with equal results but different unset memory give identical files."""
    a, b = _step(0), _step(1)
    for k in range(6):
        n = int(a.counts[k])
        b.boxes[k, :n], b.scores[k, :n], b.class_ids[k, :n], b.cand_index[k, :n] = a.boxes[k, :n], a.scores[k, :n], a.class_ids[k, :n], a.cand_index[k, :n]
    b.n_candidates[:], b.lane_status[:], b.lane_npts[:], b.tracks = a.n_candidates, a.lane_status, a.lane_npts, a.tracks
    for k in range(6):
        for l in range(4):
            m = int(a.lane_npts[k, l])
            b.lane_pts[k, l, :m] = a.lane_pts[k, l, :m]
    da, db = bench.dump_outputs(a, str(tmp_path / "a")), bench.dump_outputs(b, str(tmp_path / "b"))
    for name in da:
        assert np.array_equal(da[name], db[name]), name


def test_dump_of_a_large_step_is_a_fixed_sample_under_the_limit(tmp_path):
    r = _step(2)
    full = sum(a.nbytes for a in bench.dump_outputs(r, str(tmp_path / "full")).values())
    limit = full // 3
    s1 = bench.dump_outputs(r, str(tmp_path / "s1"), limit=limit)
    s2 = bench.dump_outputs(r, str(tmp_path / "s2"), limit=limit)
    assert sum(a.nbytes for a in s1.values()) <= limit
    keep = s1["frame_index"].astype(int)
    assert 1 <= len(keep) < 6 and np.array_equal(keep, np.sort(keep)) and np.array_equal(keep, s2["frame_index"])
    assert np.array_equal(s1["det_counts"], r.counts[keep])
    assert bench.DUMP_LIMIT == 64 << 20
