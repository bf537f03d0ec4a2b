"""CPU restatement of the reference's StVD INPUT point discard — TEST INFRASTRUCTURE (see oracle/__init__.py).

Follows `DatasetTemplate.partition` (pcdet/datasets/dataset.py:120-166) and `DatasetTemplate.input_point_discard`
(:168-189) statement by statement; pinned against the reference's own methods by `oracle/make_golden.py`
(tests/golden/stvd_input.npz).  `rng` is the numpy generator the permutations are drawn from (the reference uses the
global `np.random`)."""
from __future__ import annotations

import numpy as np


def partition(points, num=10, max_dis=60, rate=0.2):
    """-> (parts far->near, position, distant_points_num_acc)   (dataset.py:120-166)"""
    parts = []
    inter = max_dis / num
    n_all = points.shape[0]
    acc = 0
    position = num - 1
    distant_acc = 0
    x = points[:, 0]
    f32 = np.float32                             # a float32 array against a python float compares in float32, the edge
    for it in range(num):                        # (a float64 product) rounded once — numpy 1.x and 2.x alike
        i = num - it - 1
        if i == num - 1:
            mask = x >= f32(inter * i)           # :137 last bin is open-ended
        else:
            mask = (x >= f32(inter * i)) & (x < f32(inter * (i + 1)))          # :150-152
        this = points[mask]
        acc += this.shape[0]
        sampled_sum = acc + i * this.shape[0]
        if sampled_sum / n_all < rate:           # :144,157 (ZeroDivisionError on an empty cloud, like the reference)
            position = i
            distant_acc = acc
        parts.append(this)
    if position <= 0:
        position = 0
    return parts, position, distant_acc


def plan(counts_far_to_near, n_all, bin_num, rate, rng=np.random):
    """The host-side half shared with the product (`virconv_b200/preprocess.py` re-implements it; this copy is the
    checker): from the bin sizes alone decide `position`, `per_bin` and draw the permutations.  -> list of
    (bin id, None | array of kept in-bin ranks) in output (far -> near) order."""
    retain = 1 - rate
    num = bin_num
    acc, position, distant_acc = 0, num - 1, 0
    for it in range(num):
        i = num - it - 1
        cnt = counts_far_to_near[it]
        acc += cnt
        if (acc + i * cnt) / n_all < retain:
            position = i
            distant_acc = acc
    position = max(position, 0)
    out_n = int(n_all * retain)
    per_bin = int((out_n - distant_acc) / (position + 0.0001))
    segs = []
    for it in range(num):
        i = num - it - 1
        cnt = counts_far_to_near[it]
        sel = None
        if it >= num - position and cnt > per_bin:
            sel = rng.permutation(cnt)[:per_bin]
        segs.append((i, sel))
    return segs


def input_point_discard(points, bin_num=2, rate=0.8, rng=np.random):
    """(dataset.py:168-189)"""
    retain = 1 - rate
    parts, pos, distant_acc = partition(points, num=bin_num, rate=retain)
    out_n = int(points.shape[0] * retain)
    per_bin = int((out_n - distant_acc) / (pos + 0.0001))
    for i in range(len(parts) - pos, len(parts)):
        if parts[i].shape[0] > per_bin:
            rands = rng.permutation(parts[i].shape[0])
            parts[i] = parts[i][rands[:per_bin]]
    return np.concatenate(parts)


def golden_cases(g):
    """The cases of tests/golden/stvd_input.npz (oracle/make_golden.py): each input cloud is stored once
    ('<cloud>:points'), each case names its cloud ('<case>:cloud') and gives its output as rows of it ('<case>:out_rows').
    -> [(case name, points, bin_num, rate, seed, expected output)]"""
    out = []
    for name in sorted(k[:-len(':cloud')] for k in g.files if k.endswith(':cloud')):
        pts = g[f'{g[name + ":cloud"]}:points']
        bn, seed = (int(v) for v in g[f'{name}:meta'])
        out.append((name, pts, bn, float(g[f'{name}:rate']), seed, pts[g[f'{name}:out_rows']]))
    return out
