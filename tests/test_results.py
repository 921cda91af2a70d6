"""CPU suite: the vectorised pose back-projection / COCO rows (SURVEY.md 8f-2) against the
loop restatement of the reference (oracle)."""
import numpy as np
import pytest

from offsetguided_b200 import results
from oracle import ref_oracle as ro


def _batch(seed=0):
    rng = np.random.RandomState(seed)
    poses, metas = [], []
    for i, m in enumerate((3, 0, 5, 1)):
        p = np.zeros((m, 17, 6), np.float32)
        if m:
            p[..., 0:2] = rng.uniform(0, 640, size=(m, 17, 2))
            p[..., 2] = rng.uniform(0.05, 1, size=(m, 17))
            p[..., 3] = 4
            p[..., 4] = rng.uniform(0, 1, size=(m, 17))
            p[..., 5] = rng.randint(1, 10 ** 6, size=(m, 17))
            p[rng.uniform(size=(m, 17)) < 0.3] = 0          # unset keypoints
        poses.append(p)
        metas.append({'offset': np.array([-rng.randint(0, 90), -rng.randint(0, 60)], dtype=np.float64),
                      'scale': np.array([rng.uniform(0.5, 1.5)] * 2), 'hflip': False,
                      'width_height': (640, 480), 'image_id': 1000 + i})
    return poses, metas


def test_rows_equal_loop_restatement():
    poses, metas = _batch()
    rows, ids, proj = results.coco_results(poses, metas)
    ref_rows, ref_ids = ro.coco_result_rows(poses, metas)
    assert ids == ref_ids and len(rows) == len(ref_rows) == 3 + 1 + 5 + 1
    for a, b in zip(rows, ref_rows):
        assert a['image_id'] == b['image_id'] and a['category_id'] == 1
        assert a['keypoints'] == b['keypoints']
        assert a['score'] == b['score']
    for p, q, m in zip(proj, poses, metas):
        assert p.dtype == np.float32 and p.shape == q.shape


def test_inputs_are_not_mutated_and_hflip_raises():
    poses, metas = _batch(1)
    keep = [p.copy() for p in poses]
    results.coco_results(poses, metas)
    for a, b in zip(poses, keep):
        assert np.array_equal(a, b)
    metas[0]['hflip'] = True
    with pytest.raises(Exception):
        results.annotations_inverse(poses[0], metas[0])


def test_annotations_inverse_equals_restatement():
    """Bit-exact against the oracle's copy of the four in-place updates of the reference's
    transforms/preprocess.py:33-63, with equal and with unequal x / y scales."""
    poses, metas = _batch(2)
    rng = np.random.RandomState(3)
    for m in list(metas):
        metas.append(dict(m, scale=rng.uniform(0.5, 1.5, size=2)))
    for p, m in zip(poses + poses, metas):
        assert np.array_equal(results.annotations_inverse(p, m), ro.annotations_inverse(p, m))
