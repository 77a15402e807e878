"""The non-finite rule of the reference-parity select, top-k and no-repeat paths, pinned on the CPU oracle before any
kernel is held to it (include/pcv_b200.h, DESIGN.md section 2):

- greedy select equals torch.max(dim=1) on +-inf scores, +inf ties and signed-zero ties: same index, same value;
- a NaN score never wins: it counts as -inf, and a row with no score above -inf returns its first index with value
  -inf.  torch.max would return the NaN; matching that would put a NaN test into every hot loop;
- top-k lists only scores above -inf, best first, ties by ascending index; the rest of the window is -1 / -inf;
- no-repeat: a slot takes its best untaken item above -inf; a slot with none keeps its plain arg-max."""
import numpy as np
import torch

import oracle

NAN, INF = np.float32(np.nan), np.float32(np.inf)


def _select_row(scores):
    """Scores s_j = 1 * w_j: a [N, 1] table and the query [[1]], so every score is exactly the table entry."""
    W = np.asarray(scores, np.float32).reshape(-1, 1)
    i, v = oracle.score_select(W, np.ones((1, 1), np.float32))
    return int(i[0]), float(v[0])


ORDERED_ROWS = [
    [-INF, 1.0, INF, 2.0, INF],
    [-INF, -INF, -INF],
    [3.0, -INF, 3.0],
    [-0.0, 0.0, -1.0],
    [0.0, -0.0],
    [-INF, -3.0e38, -INF],
    [INF],
    [1.0, INF, INF, INF],
]


def test_select_matches_torch_max_on_ordered_scores():
    for row in ORDERED_ROWS:
        tv, ti = torch.max(torch.tensor([row], dtype=torch.float32), dim=1)
        i, v = _select_row(row)
        assert i == int(ti[0]) and v == float(tv[0]), row


NAN_ROWS = [
    ([NAN], 0),
    ([NAN, NAN, NAN], 0),
    ([NAN, 1.0, NAN], 1),
    ([NAN, -INF, NAN], 0),
    ([-INF, NAN, -INF], 0),
    ([NAN, INF, 5.0], 1),
    ([2.0, NAN, 2.0], 0),
    ([-5.0, NAN, -7.0], 0),
]


def test_select_nan_never_wins():
    for row, want in NAN_ROWS:
        i, v = _select_row(row)
        assert i == want, row
        x = torch.tensor([row], dtype=torch.float32)
        tv, ti = torch.max(torch.nan_to_num(x, nan=-np.inf, posinf=np.inf, neginf=-np.inf), dim=1)
        assert i == int(ti[0]) and v == float(tv[0]), row     # the rule: NaN counts as -inf
        if not np.isfinite(v):
            assert v == -np.inf or v == np.inf
        if np.isnan(row).any():
            assert np.isnan(float(torch.max(x)))               # torch.max itself returns the NaN


def test_select_nan_query_rows():
    rng = np.random.default_rng(3)
    W = rng.standard_normal((50, 8)).astype(np.float32)
    Q = rng.standard_normal((4, 8)).astype(np.float32)
    Q[0] = np.nan
    Q[1, 3] = np.nan
    Q[2] = 0.0
    i, v = oracle.score_select(W, Q)
    assert list(i[:2]) == [0, 0] and list(v[:2]) == [-np.inf, -np.inf]
    assert i[2] == 0 and v[2] == 0.0                           # all-zero scores: a tie, the lowest index


def _topk_reference(p, k):
    """torch: stable descending sort of the scores with NaN -> -inf; entries at -inf become -1 / -inf."""
    x = torch.nan_to_num(torch.tensor(p), nan=-np.inf, posinf=np.inf, neginf=-np.inf)
    v, i = torch.sort(x, dim=1, descending=True, stable=True)
    v, i = v[:, :k], i[:, :k]
    i = torch.where(v > -np.inf, i, torch.full_like(i, -1))
    return i.numpy(), v.numpy()


def test_topk_rule():
    rng = np.random.default_rng(5)
    N, D, k = 30, 4, 12
    W = rng.standard_normal((N, D)).astype(np.float32)
    W[3] = np.nan
    W[7, 1] = np.nan
    W[10:16] = 0.0
    W[10:16, 0] = -np.inf
    Q = rng.standard_normal((6, D)).astype(np.float32)
    Q[0, 0] = 2.0                  # -inf on items 10..15
    Q[1, 0] = -2.0                 # +inf on items 10..15: six ties
    Q[2] = np.nan
    Q[3] = 0.0
    Q[4, 0] = 0.0                  # 0 * -inf: NaN on items 10..15
    oi, ov = oracle.score_topk(W, Q, k)
    ti, tv = _topk_reference(oracle.score_logits(W, Q), k)
    assert np.array_equal(oi, ti) and np.array_equal(ov, tv)
    assert np.all(oi[2] == -1) and np.all(ov[2] == -np.inf)
    assert list(oi[1, :6]) == list(range(10, 16))
    # a finite table: the order torch.topk's documented ties give
    Wf = rng.standard_normal((40, D)).astype(np.float32)
    Wf[9] = Wf[2]
    Qf = rng.standard_normal((5, D)).astype(np.float32)
    fi, fv = oracle.score_topk(Wf, Qf, 10)
    ti, tv = _topk_reference(oracle.score_logits(Wf, Qf), 10)
    assert np.array_equal(fi, ti) and np.array_equal(fv, tv)


def test_no_repeat_rule():
    N, D, L = 6, 1, 3
    W = np.array([[1.0], [NAN], [3.0], [-INF], [2.0], [NAN]], np.float32)
    Q = np.array([[1.0], [1.0], [1.0],        # slate 0: 2, 4, 0 (the NaN and -inf items never enter)
                  [NAN], [1.0], [NAN],        # slate 1: two slots with no orderable score keep index 0 / -inf
                  [-1.0], [-1.0], [-1.0]],    # slate 2: scores -1, NaN, -3, +inf, -2: 3, then 0, then 4
                 np.float32)
    items, vals = oracle.slate_no_repeat(W, Q, L)
    assert list(items) == [2, 4, 0, 0, 2, 0, 3, 0, 4]
    assert list(vals[:3]) == [3.0, 2.0, 1.0]
    assert vals[3] == -np.inf and vals[5] == -np.inf
    # a slot whose orderable items are all taken keeps its plain arg-max (a repeat)
    W2 = np.array([[1.0], [-INF], [NAN]], np.float32)
    items, vals = oracle.slate_no_repeat(W2, np.ones((2, 1), np.float32), 2)
    assert list(items) == [0, 0] and list(vals) == [1.0, 1.0]
