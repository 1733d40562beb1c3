"""Tests of the dense tensor-core retrieval (pc_score_topk_dense, csrc/score.cu) and CatalogIndex.topk_dense.

The kernel's exactness rests on a guard band rather than on exact arithmetic: kernel 1 keeps the best KP = 8 TF32
scores of every (row, unit, 32-column chunk) list, kernel 2 re-scores them in float64 and flags a row unless the exact
k-th score is above tau + 2 eps (tau: the weakest kept score of any full list, eps = 2^-9 |q| max_norm).  So:

* the candidate lists kernel 1 leaves in the workspace are checked against the three claims the guard relies on
  (TF32 error within the budget, tau bounds every dropped product, the type filter passes every eligible product);
* constructed rows in which TF32 reverses the exact order near the k-th place must be flagged, and rows whose margin
  is wide must come back unflagged and exact (both checked on the host first, in a TF32 emulation of the pipeline);
* every row the raw kernel leaves unflagged equals the exact top-k bit for bit (oracle/retrieval.py for small shapes,
  the exact segmented path for large ones), over dims, k, catalog and row counts, units and index bases;
* CatalogIndex.topk_dense equals CatalogIndex.topk bit for bit for every row type.

In the raw kernel (and in oracle.retrieval.masked_topk) a negative row type means "no restriction"; CatalogIndex.topk
and topk_dense give such rows, and row types past num_types, no product."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import retrieval as oret
from test_gpu_parity import dev

KP, CHUNKS, BN = 8, 4, 128          # score.cu: candidates per list, 32-column chunks per tile, products per tile
PC_OK, PC_ERR_INVALID, PC_ERR_WORKSPACE, PC_ERR_UNSUPPORTED = 0, 1, 3, 4


# --------------------------------------------------------------------------- host model of the kernel pair

def _tf32(x: np.ndarray, mode: str) -> np.ndarray:
    """float32 -> the TF32 value the tensor core reads: the low 13 mantissa bits cleared ("trunc") or rounded to
    nearest ("rn", ties away; no constructed value is a tie)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32)
    if mode == "rn":
        u = u + np.uint32(0x1000)
    return (u & np.uint32(0xFFFFE000)).view(np.float32)


def _eps(q: np.ndarray, max_norm: float) -> np.ndarray:
    return np.ldexp(np.sqrt((q.astype(np.float64) ** 2).sum(1)) * np.float64(np.float32(max_norm)), -9)


def _max_norm(cat: np.ndarray) -> float:
    return float(np.float32(np.sqrt((cat.astype(np.float64) ** 2).sum(1)).max()))


def _emulate(q, cat, k, type_id, row_type, units, mode, guard=2.0):
    """(scores, indices, flags) of pc_score_topk_dense when the tensor core reads TF32 inputs rounded by `mode` and
    accumulates exactly (true for the constructed data below, whose products and sums need few bits).  `guard` is the
    multiple of eps of the guard band (2 in score.cu)."""
    p = cat.shape[0]
    n_tiles = -(-p // BN)
    tpu = -(-n_tiles // units)
    exact = oret.scores_fp64(q, cat)
    approx = (_tf32(q, mode).astype(np.float64) @ _tf32(cat, mode).astype(np.float64).T).astype(np.float32)
    eps = _eps(q, _max_norm(cat))
    region = (np.arange(p) // BN // tpu) * CHUNKS + (np.arange(p) % BN) // 32
    out_s = np.full((q.shape[0], k), -np.inf)
    out_i = np.full((q.shape[0], k), -1, np.int64)
    flags = np.zeros(q.shape[0], np.int32)
    for r in range(q.shape[0]):
        ok = np.ones(p, bool) if row_type is None or row_type[r] < 0 else type_id == row_type[r]
        cand, tau = [], -np.inf
        for g in np.unique(region[ok]):
            members = np.nonzero(ok & (region == g))[0]
            kept = members[np.lexsort((members, -approx[r, members]))][:KP]
            cand += kept.tolist()
            if kept.size == KP:
                tau = max(tau, float(approx[r, kept[-1]]))
        cand = np.array(cand, np.int64)
        top = cand[np.lexsort((cand, -exact[r, cand]))][:k]
        out_s[r, :top.size], out_i[r, :top.size] = exact[r, top], top
        if tau > -np.inf:
            flags[r] = int(top.size < k or not out_s[r, k - 1] - tau > guard * eps[r])
    return out_s, out_i, flags


def _f32(bits: int) -> np.float32:
    return np.array([bits], np.uint32).view(np.float32)[0]


HALF = 64                                # dims 0..63 carry the TF32-lossy pattern, dims 64..127 exact values
BETA = _f32(0x3F800000 | 0x0FFF)         # 1 + 4095 * 2^-23: both TF32 roundings give 1.0
UP = _f32(0x3F800000 | 0x1001)           # 1 + 4097 * 2^-23: truncation gives 1.0, round-to-nearest 1 + 2^-10
L1_AT = [32, 33, 34, 64, 65, 66, 96, 97, 98, 160, 192, 224, 288, 320, 352, 416]   # chunks 1-3, at most 6 per chunk
H_AT, WIDE_H_AT, PROBE_B_AT, PROBE_A_AT = 20, 148, (256, 257), 300


def _heavy():
    """Catalog, types and four rows (units = 1, k <= 16) built so that every score is a short sum of TF32-exact terms:

    row 0, type 0, adversarial: 8 fill products L2 (p 0-7, chunk 0) score s2 = 64 + 4/1024 exactly in TF32 and fill
      chunk 0's list, so tau = s2.  16 products L1 in chunks 1-3 score s1 = 64 + 55/1024 (= s2 + 0.28 eps).  The heavy
      product H (p 20, chunk 0) has the 0x0FFF pattern in the lossy half, where q has it too: exact s1 + 0.05 eps, TF32
      64 < s2, so kernel 1 drops it.  The exact top-k holds H; the candidates do not: the row must be flagged.
    row 1, type 1, wide margin: the same layout at s2' = 60 + 1/256 and s1' = 60.5 (= s2' + 2.8 eps), with a dropped
      product H' whose exact score is below s1': the row is provably exact and must not be flagged.
    rows 2 and 3, types 2 and 3: probes whose TF32 score is 64 under truncation and 64 + 2^-4 under round-to-nearest,
      for the catalog operand (row 2: product 256 has the 0x1001 pattern) and the query operand (row 3).
    Every other product is small Gaussian filler of type 9, and no norm exceeds L1's (eps is the same for all rows)."""
    rng = np.random.default_rng(5)
    p = 5 * BN
    cat = (rng.normal(size=(p, 128)) * 0.3).astype(np.float32)
    tid = np.full(p, 9, np.int32)

    def put(at, lossy, exact_dims, last, t):
        cat[at] = 0.0
        cat[at, :HALF] = lossy
        cat[at, HALF:] = exact_dims
        cat[at, 127] = last
        tid[at] = t

    put(np.arange(8), 0.0, 1.0, 1 + 4 / 1024, 0)                       # L2
    put(L1_AT, 0.0, 1.0, 1 + 55 / 1024, 0)                             # L1
    put(H_AT, BETA, 0.0, 0.0, 0)                                       # H
    put(BN + np.arange(8), 0.0, 0.9375, 0.9375 + 1 / 256, 1)           # L2'
    put([a + 3 for a in L1_AT], 0.0, 0.9375, 1.4375, 1)                # L1'
    put(WIDE_H_AT, _f32(0x3F700000 | 0x0FFF), 0.0, 0.0, 1)             # H': 0.9375 + 4095 * 2^-24
    put(PROBE_B_AT[0], UP, 0.0, 0.0, 2)
    put(PROBE_B_AT[1], BETA, 0.0, 0.0, 2)
    put(PROBE_A_AT, 1.0, 0.0, 0.0, 3)
    q = np.ones((4, 128), np.float32)
    q[:3, :HALF] = BETA
    q[3, :HALF] = UP
    return cat, tid, q, np.arange(4, dtype=np.int32)


def test_heavy_construction_defeats_a_narrow_guard_under_both_tf32_roundings():
    """Host check of _heavy(), before any device run: under truncation and under round-to-nearest the dense pipeline
    drops H, flags row 0, proves row 1; with a 0.25 eps guard band row 0 comes back unflagged and wrong."""
    cat, tid, q, rt = _heavy()
    eps = _eps(q, _max_norm(cat))
    exact = oret.scores_fp64(q, cat)
    s1, s2, h = exact[0, L1_AT[0]], exact[0, 0], exact[0, H_AT]
    assert 0.25 * eps[0] < s1 - s2 < 0.5 * eps[0] and s1 < h
    assert exact[1, L1_AT[0] + 3] - exact[1, BN] > 2 * eps[1] and exact[1, WIDE_H_AT] < exact[1, L1_AT[0] + 3]
    for k in (10, 16):
        ref_s, ref_i = oret.masked_topk(q, cat, k, rt, tid)
        assert ref_i[0, 0] == H_AT and set(ref_i[0, 1:]) <= set(L1_AT)
        for mode in ("trunc", "rn"):
            approx = (_tf32(q, mode).astype(np.float64) @ _tf32(cat, mode).astype(np.float64).T)
            assert approx[0, H_AT] < approx[0, :8].min() and approx[1, WIDE_H_AT] < approx[1, BN:BN + 8].min()
            s, i, f = _emulate(q, cat, k, tid, rt, 1, mode)
            assert f.tolist() == [1, 0, 0, 0], (mode, f)
            assert H_AT not in i[0]
            assert np.array_equal(i[1:], ref_i[1:]) and np.array_equal(s[1:], ref_s[1:])
            s, i, f = _emulate(q, cat, k, tid, rt, 1, mode, guard=0.25)
            assert f[0] == 0 and not np.array_equal(i[0], ref_i[0])
        probe = {m: (_tf32(q, m).astype(np.float64) @ _tf32(cat, m).astype(np.float64).T) for m in ("trunc", "rn")}
        assert probe["trunc"][2, PROBE_B_AT[0]] == 64.0 and probe["rn"][2, PROBE_B_AT[0]] == 64.0625
        assert probe["trunc"][3, PROBE_A_AT] == 64.0 and probe["rn"][3, PROBE_A_AT] == 64.0625


def _capacity_data():
    """2,048 products (16 tiles), dim 64.  Type 0: 20 members, all in chunk 0 (p % 128 < 32) of tiles 0-9; type 1: 5
    members; type 2: none; the rest types 4-9.  Rows: type 0 (x3), 1, 2, 0 with a zero query, -1 with a zero query."""
    rng = np.random.default_rng(21)
    p = 16 * BN
    cat = rng.normal(size=(p, 64)).astype(np.float32)
    tid = rng.integers(4, 10, p).astype(np.int32)
    crowd = np.array([t * BN + j for t in range(10) for j in (3, 17)])
    tid[crowd] = 0
    tid[[40, 300, 700, 1100, 2000]] = 1
    q = rng.normal(size=(7, 64)).astype(np.float32)
    q[5:] = 0.0
    return cat, tid, q, np.array([0, 0, 0, 1, 2, 0, -1], np.int32), crowd


def test_capacity_constructions_on_the_host():
    cat, tid, q, rt, crowd = _capacity_data()
    assert np.all(crowd % BN < 32) and np.sum(tid == 0) == 20 and np.sum(tid == 1) == 5 and np.sum(tid == 2) == 0
    # with one unit chunk 0's list holds 8 of type 0's 20 members: rows of type 0 must be flagged for any k > 8
    for mode in ("trunc", "rn"):
        for k in (9, 16):
            _, _, f = _emulate(q, cat, k, tid, rt, 1, mode)
            assert f[:3].tolist() == [1, 1, 1] and f[3:5].tolist() == [0, 0] and f[5:].tolist() == [1, 1]


# --------------------------------------------------------------------------- refusals (no device)

PTR = ctypes.c_void_p(1 << 20)           # non-null and 16-byte aligned; never dereferenced: each refusal precedes any CUDA call


def _refusal(**over):
    from pcompanion_b200 import _lib
    a = dict(q=PTR, rows=256, dim=128, catalog=PTR, products=1000, type_id=None, row_type=None, k=10, units=2,
             index_base=0, max_norm=1.0, out_s=PTR, out_i=PTR, flags=PTR, ws=PTR,
             ws_bytes=_lib.LIB.pc_score_topk_workspace_bytes(256, 2), stream=None)
    a.update(over)
    rc = _lib.LIB.pc_score_topk_dense(*a.values())
    return rc, (_lib.LIB.pc_last_error() or b"").decode()


@pytest.mark.parametrize("over, code", [
    (dict(k=0), PC_ERR_UNSUPPORTED), (dict(k=17), PC_ERR_UNSUPPORTED),
    (dict(dim=16), PC_ERR_UNSUPPORTED), (dict(dim=48), PC_ERR_UNSUPPORTED), (dict(dim=160), PC_ERR_UNSUPPORTED),
    (dict(units=0), PC_ERR_INVALID), (dict(units=4097), PC_ERR_INVALID),
    (dict(products=0), PC_ERR_UNSUPPORTED), (dict(products=1 << 31), PC_ERR_UNSUPPORTED),
    (dict(ws_bytes=256 * 2 * CHUNKS * KP * 8 - 1), PC_ERR_WORKSPACE),
    (dict(q=ctypes.c_void_p((1 << 20) + 4)), PC_ERR_INVALID),
])
def test_bad_arguments_are_refused_without_a_device(over, code):
    rc, msg = _refusal(**over)
    assert rc == code and "score_topk_dense" in msg, (rc, msg)


def test_workspace_layout_and_zero_rows_without_a_device():
    from pcompanion_b200 import _lib
    # part_s float [rows, units, 4, KP] followed by part_i int32 of the same shape (ScoreParams); the device tests
    # below read the candidate lists through this layout
    assert _lib.LIB.pc_score_topk_workspace_bytes(300, 7) == 300 * 7 * CHUNKS * KP * 8
    assert _refusal(rows=0, ws_bytes=0)[0] == PC_OK


# --------------------------------------------------------------------------- device helpers

def _raw(q, cat, k, type_id=None, row_type=None, units=1, index_base=0):
    """pc_score_topk_dense with a workspace this test owns (filled with -7 first, so an unwritten entry shows).  Returns
    numpy (scores, indices, flags, part_s [R, units, 4, KP], part_i) and the max_norm passed."""
    from pcompanion_b200 import _lib
    rows, dim = q.shape
    max_norm = float(cat.norm(dim=1).max())
    n = rows * units * CHUNKS * KP
    ws = torch.full((2 * n,), -7, dtype=torch.int32, device=q.device)
    s = torch.empty(rows, k, dtype=torch.float64, device=q.device)
    i = torch.empty(rows, k, dtype=torch.int64, device=q.device)
    f = torch.empty(rows, dtype=torch.int32, device=q.device)
    _lib.call("pc_score_topk_dense", _lib.dev(q, torch.float32, "q"), rows, dim, _lib.dev(cat, torch.float32, "catalog"),
              cat.shape[0], _lib.dev(type_id, torch.int32, "type_id"), _lib.dev(row_type, torch.int32, "row_type"), k,
              units, int(index_base), max_norm, _lib.dev(s, torch.float64, "s"), _lib.dev(i, torch.int64, "i"),
              _lib.dev(f, torch.int32, "flags"), _lib.dev(ws, torch.int32, "ws"), ws.numel() * 4, _lib.stream())
    part_s = ws[:n].view(torch.float32).reshape(rows, units, CHUNKS, KP).cpu().numpy()
    part_i = ws[n:].reshape(rows, units, CHUNKS, KP).cpu().numpy()
    return s.cpu().numpy(), i.cpu().numpy(), f.cpu().numpy(), part_s, part_i, max_norm


def _check_lists(q, cat, type_id, row_type, units, part_s, part_i, max_norm, exact=None):
    """The premises of the guard band, for every candidate list kernel 1 wrote.  Returns max |approx - exact| / eps.

    * entries are a prefix of valid candidates, then (-inf, -1); valid ones are sorted by (score desc, index asc);
    * a candidate lies in its unit's tile range and its chunk's 32 columns, and has the row's type;
    * |approx - exact| <= 2 eps for every candidate (the budget the guard uses);
    * a list holds min(KP, eligible products of its (unit, chunk)), and (with `exact`, the [R, P] fp64 scores) no
      eligible product missing from a full list scores above the list's weakest approximate score + 2 eps."""
    p = cat.shape[0]
    n_tiles = -(-p // BN)
    tpu = -(-n_tiles // units)
    valid = part_i >= 0
    assert np.all(valid | (part_i == -1)), "unwritten or corrupt candidate index"
    assert np.all(np.isneginf(part_s[~valid]))
    assert np.all(valid[..., :-1] | ~valid[..., 1:]), "a list is not a prefix"
    pair = valid[..., :-1] & valid[..., 1:]
    a, b = part_s[..., :-1], part_s[..., 1:]
    ordered = (a > b) | ((a == b) & (part_i[..., :-1] < part_i[..., 1:]))
    assert np.all(ordered[pair]), "a list is not sorted by (score desc, index asc)"
    r_, u_, c_, _ = np.nonzero(valid)
    idx = part_i[valid].astype(np.int64)
    assert np.all(idx < p)
    tile = idx // BN
    assert np.all((tile >= u_ * tpu) & (tile < np.minimum((u_ + 1) * tpu, n_tiles))), "candidate outside its unit"
    assert np.all((idx % BN) // 32 == c_), "candidate outside its chunk"
    if type_id is not None and row_type is not None:
        rt = row_type[r_]
        assert np.all((rt < 0) | (type_id[idx] == rt)), "candidate of another type"
    ex = np.einsum("nd,nd->n", q[r_].astype(np.float64), cat[idx].astype(np.float64))
    eps = _eps(q, max_norm)[r_]
    err = np.abs(part_s[valid].astype(np.float64) - ex)
    assert np.all(err <= 2 * eps), f"TF32 error {float((err / np.maximum(eps, 1e-300)).max()):.3f} eps > 2 eps"
    if exact is not None:
        rows = q.shape[0]
        g = (np.arange(p) // BN // tpu) * CHUNKS + (np.arange(p) % BN) // 32
        if type_id is not None and row_type is not None:
            elig = (row_type[:, None] < 0) | (type_id[None, :] == row_type[:, None])
        else:
            elig = np.ones((rows, p), bool)
        count = np.zeros((rows, units * CHUNKS), np.int64)
        np.add.at(count, (np.nonzero(elig)[0], g[np.nonzero(elig)[1]]), 1)
        assert np.array_equal(valid.sum(-1).reshape(rows, -1), np.minimum(count, KP)), "an eligible product was lost"
        last = np.where(valid[..., -1], part_s[..., -1], np.inf).reshape(rows, -1).astype(np.float64)
        kept = np.zeros((rows, p), bool)
        kept[r_, idx] = True
        rr, pp = np.nonzero(elig & ~kept)
        bound = last[rr, g[pp]] + 2 * _eps(q, max_norm)[rr]
        assert np.all(exact[rr, pp] <= bound), "a dropped product scores above tau + 2 eps"
    pos = eps > 0
    return float((err[pos] / eps[pos]).max()) if pos.any() else 0.0


def _oracle_topk(exact, k, row_type=None, type_id=None):
    """oracle.retrieval.masked_topk from its own scores (oret.scores_fp64, computed once per data set)."""
    s = exact
    if row_type is not None and type_id is not None:
        s = np.where((type_id[None, :] == row_type[:, None]) | (row_type[:, None] < 0), exact, -np.inf)
    idx = np.where(np.isneginf(s), -1, np.arange(exact.shape[1], dtype=np.int64)[None, :])
    pad_s, pad_i = np.full((exact.shape[0], k), -np.inf), np.full((exact.shape[0], k), -1, np.int64)
    return oret.merge_topk(np.concatenate([pad_s, s], 1), np.concatenate([pad_i, idx], 1), k)


def _assert_unflagged_exact(s, i, f, ref_s, ref_i, what):
    ok = f == 0
    assert np.all((f == 0) | (f == 1))
    bad = np.nonzero(ok & ~(np.all(i == ref_i, 1) & np.all(s == ref_s, 1)))[0]
    assert bad.size == 0, f"{what}: unflagged rows differ from the exact top-k: {bad[:8].tolist()}"


def _t(x):
    return None if x is None else torch.tensor(x, device=dev())


# --------------------------------------------------------------------------- (a) guard-band premise

@pytest.mark.gpu
def test_candidate_lists_satisfy_the_guard_premise():
    """Gaussian data (unrestricted rows, typed rows, quarters mixing both; 3 units) and the heavy construction.  Prints
    the largest |approx - exact| / eps seen, and whether the tensor core truncates or rounds each TF32 operand."""
    rng = np.random.default_rng(3)
    p, r, t = 20_000, 256, 6
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    tid = rng.integers(0, t, p).astype(np.int32)
    q = rng.normal(size=(r, 128)).astype(np.float32)
    rt = rng.integers(0, t, r).astype(np.int32)
    rt[:64] = -1
    rt[128:160:3] = -1
    s, i, f, ps, pi, mn = _raw(_t(q), _t(cat), 10, _t(tid), _t(rt), units=3)
    exact = oret.scores_fp64(q, cat)
    worst = _check_lists(q, cat, tid, rt, 3, ps, pi, mn, exact)
    ref_s, ref_i = _oracle_topk(exact, 10, rt, tid)
    _assert_unflagged_exact(s, i, f, ref_s, ref_i, "gaussian")
    assert f.sum() < r // 4

    cat, tid, q, rt = _heavy()
    s, i, f, ps, pi, mn = _raw(_t(q), _t(cat), 10, _t(tid), _t(rt), units=1)
    worst_heavy = _check_lists(q, cat, tid, rt, 1, ps, pi, mn, oret.scores_fp64(q, cat))
    got_b = ps[2][pi[2] == PROBE_B_AT[0]]
    got_a = ps[3][pi[3] == PROBE_A_AT]
    mode = {64.0: "truncates", 64.0625: "rounds to nearest"}
    assert got_b.size == 1 and got_a.size == 1 and got_b[0] in mode and got_a[0] in mode, (got_b, got_a)
    print(f"\nmax |approx - exact| / eps: gaussian {worst:.4f}, heavy {worst_heavy:.4f}; TF32 catalog operand "
          f"{mode[float(got_b[0])]}, query operand {mode[float(got_a[0])]}")


# --------------------------------------------------------------------------- (b) adversarial guard-band rows

@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16])
def test_adversarial_row_is_flagged_and_wide_margin_row_is_exact(k):
    from pcompanion_b200 import CatalogIndex
    cat, tid, q, rt = _heavy()
    s, i, f, ps, pi, _ = _raw(_t(q), _t(cat), k, _t(tid), _t(rt), units=1)
    ref_s, ref_i = oret.masked_topk(q, cat, k, rt, tid)
    assert H_AT not in pi[0] and WIDE_H_AT not in pi[1], "kernel 1 kept the product the construction makes it drop"
    assert f.tolist() == [1, 0, 0, 0], f"flags {f.tolist()}: row 0 must be flagged, rows 1-3 proven"
    assert np.array_equal(i[1:], ref_i[1:]) and np.array_equal(s[1:], ref_s[1:])
    index = CatalogIndex(_t(cat), _t(tid), num_types=10)
    ds, di = index.topk_dense(_t(q), k, _t(rt))
    assert np.array_equal(di.cpu().numpy(), ref_i) and np.array_equal(ds.cpu().numpy(), ref_s)


# --------------------------------------------------------------------------- (c) candidate capacity

@pytest.mark.gpu
@pytest.mark.parametrize("k", [9, 16])
def test_candidate_capacity(k):
    """A type whose members share one chunk column range: with one unit a list keeps 8 of them, so the row must be
    flagged; with one unit per tile no list is full and the row is exact.  A type with fewer than k members pads,
    is not flagged and has no full list; an empty type is all padding; zero queries (eps = 0, all scores tie) are
    flagged or exact."""
    from pcompanion_b200 import CatalogIndex
    cat, tid, q, rt, _ = _capacity_data()
    ref_s, ref_i = oret.masked_topk(q, cat, k, rt, tid)
    n_tiles = cat.shape[0] // BN
    for units in (1, n_tiles):
        s, i, f, ps, pi, mn = _raw(_t(q), _t(cat), k, _t(tid), _t(rt), units=units)
        _check_lists(q, cat, tid, rt, units, ps, pi, mn, oret.scores_fp64(q, cat))
        _assert_unflagged_exact(s, i, f, ref_s, ref_i, f"units={units}")
        if units == 1:
            assert f[:3].tolist() == [1, 1, 1], "a row with more eligible products than candidates was not flagged"
        else:
            assert f[:3].tolist() == [0, 0, 0] and not (pi[:3, ..., -1] >= 0).any()
        assert f[3] == 0 and f[4] == 0 and not (pi[3:5, ..., -1] >= 0).any()      # tau = -inf: no full list
        assert np.array_equal(i[3, :5], ref_i[3, :5]) and (i[3, 5:] == -1).all() and np.isneginf(s[3, 5:]).all()
        assert (i[4] == -1).all() and np.isneginf(s[4]).all()
    index = CatalogIndex(_t(cat), _t(tid), num_types=10)
    ds, di = index.topk_dense(_t(q), k, _t(np.maximum(rt, 0)))
    es, ei = index.topk(_t(q), k, _t(np.maximum(rt, 0)))
    assert torch.equal(di, ei) and torch.equal(ds, es)


# --------------------------------------------------------------------------- (d) type filter

N_FILTER_TYPES = 2000


def _filter_data():
    """30,000 products of 2,000 types; 160 rows (five 32-row lane quarters) whose types collide in the 768-bucket
    filter: quarter 0 only typed rows of types t, t + 768, t + 1536 (filtered path), quarter 1 the same with two
    unrestricted rows (unfiltered path), quarter 2 typed rows including types no product has (2304 = 768 * 3 and
    2309, in the buckets of types 0 and 5), quarter 3 typed and negative rows, quarter 4 random types."""
    rng = np.random.default_rng(7)
    p, r = 30_000, 160
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    tid = rng.integers(0, N_FILTER_TYPES, p).astype(np.int32)
    q = rng.normal(size=(r, 128)).astype(np.float32)
    coll = np.array([t + j * 768 for t in (0, 5, 300) for j in range(3)], np.int32)
    rt = rng.integers(0, N_FILTER_TYPES, r).astype(np.int32)
    rt[0:32] = np.resize(coll, 32)
    rt[32:64] = np.resize(coll[::-1], 32)
    rt[[40, 50]] = -1
    rt[64:96] = np.resize(np.append(coll, [2304, 2309, 5000]), 32)
    rt[96:128] = np.resize(np.append(coll, [-1, -5]), 32)
    return cat, tid, q, rt


@pytest.mark.gpu
def test_type_filter_bucket_collisions_and_mixed_quarters():
    cat, tid, q, rt = _filter_data()
    exact = oret.scores_fp64(q, cat)
    qt, ct = _t(q), _t(cat)
    for use_tid, use_rt in ((True, True), (True, False), (False, False), (False, True)):
        t_np, r_np = (tid if use_tid else None), (rt if use_rt else None)
        s, i, f, ps, pi, mn = _raw(qt, ct, 10, _t(t_np), _t(r_np), units=4)
        if use_rt and not use_tid:
            # without type ids every product has type 0: rows of type 0 and unrestricted rows rank everything
            ref_s, ref_i = _oracle_topk(exact, 10, rt, np.zeros_like(tid))
            _check_lists(q, cat, np.zeros_like(tid), rt, 4, ps, pi, mn, exact)
        else:
            ref_s, ref_i = _oracle_topk(exact, 10, r_np, t_np)
            _check_lists(q, cat, t_np, r_np, 4, ps, pi, mn, exact)
        _assert_unflagged_exact(s, i, f, ref_s, ref_i, f"type_id={use_tid} row_type={use_rt}")
        if use_tid and use_rt:
            assert f[rt >= 0].sum() == 0, "a typed row with ~30 eligible products was flagged"
            assert (i[rt >= N_FILTER_TYPES] == -1).all()


# --------------------------------------------------------------------------- (e) shape sweep

N_SWEEP_TYPES = 7
# (dim, k, products, rows, units, index_base); units "t" = one per tile, "t+5" = five empty units more
SWEEP = [
    (32, 1, 1, 1, 1, 0),
    (64, 2, 127, 31, 1, 5_000_000_000),
    (96, 8, 128, 129, 3, 0),
    (128, 9, 129, 31, "t", 5_000_000_000),
    (32, 16, 129, 129, "t+5", 0),
    (128, 16, 1, 4097, 3, 5_000_000_000),
    (64, 9, 100_003, 4097, None, 0),
    (96, 16, 100_003, 129, 3, 5_000_000_000),
    (128, 1, 100_003, 1, 1, 0),
    (32, 8, 100_003, 31, "t+5", 5_000_000_000),
    (128, 2, 100_003, 129, "t", 0),
]


def _reference(q, cat, k, tid, rt, base):
    """Exact top-k with the raw kernel's row-type semantics: the oracle for small shapes, else the exact segmented
    path (CatalogIndex.topk; rows with a negative type ranked against the whole catalog)."""
    if q.shape[0] * cat.shape[0] <= 1 << 21:
        return oret.masked_topk(q, cat, k, rt, tid, index_base=base)
    from pcompanion_b200 import CatalogIndex
    index = CatalogIndex(_t(cat), _t(tid), base, N_SWEEP_TYPES)
    s, i = index.topk(_t(q), k, _t(rt))
    un = torch.tensor(np.nonzero(rt < 0)[0], device=dev())
    if un.numel():
        us, ui = index.topk(_t(q)[un], k)
        s[un], i[un] = us, ui
    return s.cpu().numpy(), i.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("dim, k, p, r, units, base", SWEEP)
def test_shape_sweep_unflagged_rows_are_exact(dim, k, p, r, units, base):
    from pcompanion_b200 import ops
    rng = np.random.default_rng(dim * 7919 + k * 31 + p + r)
    cat = rng.normal(size=(p, dim)).astype(np.float32)
    tid = rng.integers(0, N_SWEEP_TYPES, p).astype(np.int32)
    q = rng.normal(size=(r, dim)).astype(np.float32)
    rt = rng.integers(-1, N_SWEEP_TYPES, r).astype(np.int32)
    n_tiles = -(-p // BN)
    if units is None:
        qt, ct = _t(q), _t(cat)
        s, i, f = (x.cpu().numpy() for x in ops.score_topk_dense(qt, ct, k, _t(tid), _t(rt), base))
        s2, i2, f2 = (x.cpu().numpy() for x in ops.score_topk_dense(qt, ct, k, _t(tid), _t(rt), base))
        assert np.array_equal(s, s2) and np.array_equal(i, i2) and np.array_equal(f, f2), "repeated call differs"
    else:
        units = {"t": n_tiles, "t+5": n_tiles + 5}.get(units, units)
        s, i, f, ps, pi, mn = _raw(_t(q), _t(cat), k, _t(tid), _t(rt), units, base)
        if p * r <= 1 << 21:
            _check_lists(q, cat, tid, rt, units, ps, pi, mn, oret.scores_fp64(q, cat))
    ref_s, ref_i = _reference(q, cat, k, tid, rt, base)
    _assert_unflagged_exact(s, i, f, ref_s, ref_i, f"dim={dim} k={k} P={p} R={r} units={units} base={base}")
    assert (f == 0).any(), "every row flagged: the sweep case checks nothing"


@pytest.mark.gpu
def test_flag_rate_on_c4_like_data():
    """Gaussian catalog of 1,000 types (as bench.py's retrieval leg, at 1/10 of its size), 3,072 typed rows, k = 10,
    automatic units: unflagged rows are exact, and the flag rate is printed.  A list then holds ~19 products of a type,
    and the 10th best of a type's ~1,000 lies far above any list's 8th best, so (almost) no row is flagged."""
    from pcompanion_b200 import CatalogIndex, ops
    g = torch.Generator(device=dev()).manual_seed(4)
    cat = torch.randn(1_000_000, 128, generator=g, device=dev())
    tid = torch.randint(0, 1000, (1_000_000,), generator=g, device=dev(), dtype=torch.int32)
    q = torch.randn(3072, 128, generator=g, device=dev())
    rt = torch.randint(0, 1000, (3072,), generator=g, device=dev(), dtype=torch.int32)
    s, i, f = ops.score_topk_dense(q, cat, 10, tid, rt)
    es, ei = CatalogIndex(cat, tid, num_types=1000).topk(q, 10, rt)
    ok = f == 0
    print(f"\nC4-like flag rate: {int(f.sum())} of {f.numel()} rows")
    assert torch.equal(s[ok], es[ok]) and torch.equal(i[ok], ei[ok])
    assert int(f.sum()) <= f.numel() // 100


# --------------------------------------------------------------------------- (g) CatalogIndex.topk_dense

N_G_TYPES = 8


@pytest.mark.gpu
def test_topk_dense_equals_topk_for_every_row_type():
    """Types: 2 empty, 5 with 6 products (< k), 6 with 12 products in one chunk column range (flagged rows, re-run on
    the exact path).  Row types cover -3..11: negative, empty, small, crowded and past num_types."""
    from pcompanion_b200 import CatalogIndex
    rng = np.random.default_rng(8)
    p, r = 30_000, 200
    cat = rng.normal(size=(p, 128)).astype(np.float32)
    tid = rng.choice(np.array([0, 1, 3, 4, 7], np.int32), p)
    tid[rng.choice(p, 6, replace=False)] = 5
    tid[5:17] = 6
    q = rng.normal(size=(r, 128)).astype(np.float32)
    rt = rng.integers(-3, N_G_TYPES + 4, r).astype(np.int32)
    rt[:15] = np.arange(-3, 12)
    rt[15:40] = 6
    index = CatalogIndex(_t(cat), _t(tid), num_types=N_G_TYPES)
    qt, rtt = _t(q), _t(rt)
    for k in (1, 10, 16):
        es, ei = index.topk(qt, k, rtt)
        ds, di = index.topk_dense(qt, k, rtt)
        assert torch.equal(di, ei) and torch.equal(ds, es), f"k={k}"
        assert (ei[(rtt < 0) | (rtt >= N_G_TYPES)] == -1).all()
        us, ui = index.topk_dense(qt[:40], k)
        es, ei = index.topk(qt[:40], k)
        assert torch.equal(ui, ei) and torch.equal(us, es), f"k={k}, no row types"
    with pytest.raises(RuntimeError, match="k=17"):
        index.topk_dense(qt, 17, rtt)
    with pytest.raises(RuntimeError, match="dim=160"):
        CatalogIndex(_t(rng.normal(size=(1000, 160)).astype(np.float32))).topk_dense(_t(np.ones((4, 160), np.float32)), 10)
    untyped = CatalogIndex(_t(cat))
    with pytest.raises(ValueError, match="built without type ids"):
        untyped.topk_dense(qt, 10, rtt)
    ds, di = untyped.topk_dense(qt[:40], 10)
    es, ei = untyped.topk(qt[:40], 10)
    assert torch.equal(di, ei) and torch.equal(ds, es)
