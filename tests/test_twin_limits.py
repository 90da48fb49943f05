"""The compressed twins at the limits of their encoders: csr-pattern8 (one byte per row) and csr-dict16 (two bytes per
entry).

Each device matrix keeps at most the twins its encoders accept, and the twins decide the kernel: the lean pattern kernel
(csr_pat2_kernel), the table kernel (csr_pattern_kernel), the dictionary kernel or the plain CSR kernels.  The encoders
decide against hard limits: 255 pattern ids (id 255 is the escape), 2048 table entries (a candidate that would overflow
the table is skipped and later, shorter ones still enter), rows of at most 64 entries, pattern 0 by value up to 32
entries and masked only up to 7, the lean kernel for a 5- or 7-entry pattern 0 on at least half the rows, a twin only
when at least 3/4 of the rows are tabulated, at most 2^15 distinct rows, and at most 256 distinct values and 256
distinct offsets for csr-dict16 (the value whose bits are all ones is the device set's empty-slot marker).

The matrices below are built to sit exactly on either side of each limit: a 7-offset band whose first and last H rows
hold only the diagonal, with groups of rows whose diagonal is moved by an exactly representable k * 2^-20 (a pattern
of their own each), longer rows, reordered rows, signed zeros and NaN payloads.  CPU: each generator against the host
encoders (sparsh_pattern_encode, sparsh_dict_encode): the intended pattern, entry, escape and dictionary counts.  GPU:
the device encoders' decisions against the host encoders', every kernel family against the oracle bit for bit (the fused
reductions against an exact sum), and value updates that cross each limit against a fresh upload of the same values."""
import math
from functools import lru_cache

import numpy as np
import pytest
from oracle_bindings import CSR
from test_host_setup import _check_pattern_decode, _dict_encode, _pattern_encode

OMEGA = 0.66667
EPS = 2.0 ** -20  # 6 + k * EPS is exact for every k used here
S1, S2, H = 12, 150, 160  # band offsets; the first and last H rows hold the diagonal alone
P7 = [(-S2, -1.0), (-S1, -1.0), (-1, -1.0), (0, 6.0), (1, -1.0), (S1, -1.0), (S2, -1.0)]
B1 = [(0, 6.0)]
ESC = 255
VALID = 0x80
KIND = {"scalar": 0, "stream": 1, "vector": 2, "dict": 3, "pattern": 4}


def long_row(m, diag):
    """m entries at offsets -(m // 2) .. m - m // 2 - 1: -1 off the diagonal"""
    return [(o, diag if o == 0 else -1.0) for o in range(-(m // 2), m - m // 2)]


def build(n, shapes, groups, seed=1, halo=0, h=H):
    """n rows: shapes[1] on the first h rows (and on the last h rows when halo == 0: square), shapes[0] on every other
    row except the groups, [(shape index, rows, diagonal or None)], which are spread over the interior in a fixed
    shuffled order.  The diagonal of a group replaces the first offset-0 entry of its rows.  Columns: n + halo."""
    lo, hi = h, n - (h if halo == 0 else 0)
    lab = np.full(n, -1, dtype=np.int64)
    sizes = [g[1] for g in groups]
    assert sum(sizes) <= hi - lo, (sum(sizes), hi - lo)
    inner = np.zeros(hi - lo, dtype=np.int64)
    inner[: sum(sizes)] = np.repeat(np.arange(1, len(groups) + 1), sizes)
    lab[lo:hi] = np.random.default_rng(seed).permutation(inner)
    sid = np.where(lab < 0, 1, 0)
    gshape = np.array([0] + [g[0] for g in groups])
    sid[lab > 0] = gshape[lab[lab > 0]]
    lens = np.array([len(s) for s in shapes])
    rp = np.zeros(n + 1, dtype=np.int64)
    rp[1:] = np.cumsum(lens[sid])
    ci, v = np.empty(rp[-1], dtype=np.int64), np.empty(rp[-1])
    dpos = np.full(n, -1, dtype=np.int64)
    for t, s in enumerate(shapes):
        rows = np.flatnonzero(sid == t)
        if rows.size == 0:
            continue
        off = np.array([o for o, _ in s], dtype=np.int64)
        idx = rp[rows][:, None] + np.arange(len(s))[None, :]
        ci[idx] = rows[:, None] + off[None, :]
        v[idx] = np.array([x for _, x in s])
        if 0 in list(off):
            dpos[rows] = rp[rows] + list(off).index(0)
    gdiag = np.array([np.nan] + [np.nan if g[2] is None else g[2] for g in groups])
    moved = lab > 0
    moved[moved] = ~np.isnan(gdiag[lab[moved]])
    assert np.all(dpos[moved] >= 0)
    v[dpos[moved]] = gdiag[lab[moved]]
    assert ci.min() >= 0 and ci.max() < n + halo
    return CSR(n, n + halo, rp, ci, v)


def with_bits(M, pos, bits):
    v = M.val.copy()
    v.view(np.uint64)[pos] = np.asarray(bits, dtype=np.uint64)
    return CSR(M.nrow, M.ncol, M.rowptr, M.colindex, v)


# ---------------------------------------------------------------------------------------------------------- cases
# Each case: the matrix and what the host encoders must make of it.  "pat": (patterns, table entries, escape rows)
# without a smoothing diagonal; (0, 0, nrow) when the encoder declines.  "dict": (values, offsets) or None.
# "kind": the family choose_kernel picks before any twin.
def patterns_case(total):
    """pattern 0, the boundary row and 298 groups of 299 .. 2 rows; the groups after the first total - 2 keep
    pattern 0's diagonal (they are pattern 0 rows): every variant has the same sparsity"""
    sizes = [300 - k for k in range(1, 299)]
    groups = [(0, s, 6.0 + k * EPS if k <= total - 2 else 6.0) for k, s in enumerate(sizes, 1)]
    M = build(160000, [P7, B1], groups, seed=2)
    tab = min(total, 255)
    esc = sum(sizes[tab - 2: total - 2])
    values = 2 + min(total - 2, 298)
    return M, dict(pat=(tab, 8 + 7 * (tab - 2), esc), dict=(values, 7) if values <= 256 else None, kind="stream")


def candidates_case(distinct, n=140320):
    """pattern 0, the boundary row and distinct - 2 rows of pattern 0's structure with distinct diagonals; past 2^15
    distinct rows neither encoder tabulates anything"""
    u = distinct - 2
    M = build(n, [P7, B1], [(0, 1, 6.0 + k * EPS) for k in range(1, u + 1)], seed=3)
    pat = (255, 8 + 7 * 253, u - 253) if distinct <= 1 << 15 else (0, 0, n)
    return M, dict(pat=pat, dict=None, kind="stream")


def table_case(full):
    """4 groups of 64-entry rows, one of 48, 248 of pattern 0's structure: 255 patterns and exactly 2048 entries; with
    full=False all but 20 of the short groups are pattern 0 rows (27 patterns), same sparsity"""
    shapes = [P7, B1, long_row(64, 64.0), long_row(48, 48.0)]
    groups = [(2, 301 - k, 64.0 + k * EPS) for k in range(1, 5)] + [(3, 296, 48.0 + EPS)]
    groups += [(0, 296 - k, 6.0 + k * EPS if full or k <= 20 else 6.0) for k in range(1, 249)]
    M = build(120000, shapes, groups, seed=4)
    pat = (255, 2048, 0) if full else (27, 8 + 4 * 64 + 48 + 20 * 7, 0)
    return M, dict(pat=pat, dict=(255 if full else 27, 66), kind="stream")


def entries_exact_case(last):
    """31 groups of 64-entry rows and one of `last` entries: 8 + 31 * 64 + 56 = 2048 fills the table exactly; with
    57 entries the last group is skipped"""
    shapes = [P7, B1, long_row(64, 64.0), long_row(last, float(last))]
    groups = [(2, 121 - k, 64.0 + k * EPS) for k in range(1, 32)] + [(3, 60, float(last) + EPS)]
    M = build(40000, shapes, groups, seed=5)
    pat = (34, 2048, 0) if last == 56 else (33, 1992, 60)
    return M, dict(pat=pat, dict=(34, 66), kind="stream")


def entries_skip_case(merged):
    """33 groups of 64-entry rows, then 8 short groups: the 32nd and 33rd long patterns would overflow the table and are
    skipped, the short ones after them still fill it to 2048.  merged: the last two long groups take the values of two
    others (same sparsity), so every long pattern fits"""
    shapes = [P7, B1, long_row(64, 64.0)]
    ks = list(range(1, 34))
    if merged:
        ks[31], ks[32] = 30, 31
    groups = [(2, 121 - i, 64.0 + k * EPS) for i, k in enumerate(ks, 1)] + [(0, 81 - i, 6.0 + i * EPS) for i in range(1, 9)]
    M = build(40000, shapes, groups, seed=6)
    pat = (41, 2048, 0) if merged else (41, 2048, (121 - 32) + (121 - 33))
    return M, dict(pat=pat, dict=(41 if merged else 43, 66), kind="stream")


def row_length_case(m):
    M = build(20000, [P7, B1, long_row(m, float(m))], [(2, 400, None)], seed=7)
    pat = (3, 8 + m, 0) if m <= 64 else (2, 8, 400)
    return M, dict(pat=pat, dict=(3, 2 + m), kind="stream")


def len0_case(length):
    """a band whose every row has `length` entries (constant values), the first and last 16 rows the diagonal alone"""
    p = long_row(length, float(length))
    b = [(0, float(length))]
    M = build(8192, [p, b], [], seed=8, h=16)
    pat = (1, 1, 0) if length == 1 else (2, length + 1, 0)
    return M, dict(pat=pat, dict=(1 if length == 1 else 2, length), kind="scalar" if length <= 2 else "stream")


def cover_half_case(minus):
    """pattern 0 on exactly n/2 rows (minus=1: one row fewer, which joins another group)"""
    n = 20000
    p0 = n // 2 - minus
    g1 = 5000
    M = build(n, [P7, B1], [(0, g1, 6.0 + EPS), (0, n - 2 * H - p0 - g1, 6.0 + 2 * EPS)], seed=9)
    return M, dict(pat=(4, 22, 0), dict=(4, 7), kind="stream", cover0=p0 / n)


def cover_quarter_case(minus):
    """exactly 3/4 of the rows tabulated (minus=1: one fewer): pattern 0, the boundary row and unique rows, of which the
    first 253 fill the pattern ids"""
    n = 20000
    p0 = 3 * n // 4 - 2 * H - 253 - minus
    u = n - 2 * H - p0
    M = build(n, [P7, B1], [(0, 1, 6.0 + k * EPS) for k in range(1, u + 1)], seed=10)
    return M, dict(pat=(255, 8 + 7 * 253, u - 253), dict=None, kind="stream")


def mask_repeat_case():
    """pattern 0 repeats an (offset, value) pair; rows that keep one of the pair are masked"""
    p0 = [(-4, -1.0), (-1, -1.0), (-1, -1.0), (0, 6.0), (1, -1.0), (1, -1.0), (4, -1.0)]
    q1 = [(-1, -1.0), (0, 6.0), (1, -1.0)]
    q2 = [(-4, -1.0), (-1, -1.0), (-1, -1.0), (0, 6.0)]
    M = build(20000, [p0, B1, q1, q2], [(2, 2000, None), (3, 1000, None)], seed=11)
    return M, dict(pat=(4, 7 + 1 + 3 + 4, 0), dict=(2, 5), kind="stream", masked=3)


def mask_order_case():
    """a row with pattern 0's entries in another order (not a subsequence: the table walk) and a masked one"""
    q = [P7[0], P7[1], P7[4], P7[3], P7[2], P7[5], P7[6]]
    M = build(20000, [P7, B1, q, [P7[2], P7[3], P7[4]]], [(2, 3000, None), (3, 1000, None)], seed=12)
    return M, dict(pat=(4, 7 + 1 + 7 + 3, 0), dict=(2, 7), kind="stream", masked=2)


def mask_zero_case():
    """pattern 0's diagonal is +0.0; a pattern whose diagonal is -0.0 is not masked (different bits), one that keeps
    +0.0 is"""
    p0 = [(o, 0.0 if o == 0 else x) for o, x in P7]
    M = build(20000, [p0, [(0, 0.0)], p0, [P7[2], (0, 0.0), P7[4]]], [(2, 3000, -0.0), (3, 1000, None)], seed=13)
    return M, dict(pat=(4, 7 + 1 + 7 + 3, 0), dict=(3, 7), kind="stream", masked=2)


EXTRA_OFFSETS = [o for o in range(-H, H + 1) if o not in {o for o, _ in P7}]
NAN_BITS = [0xFFFFFFFFFFFFFFFF, 0x0000000000000000, 0x8000000000000000, 0x7FF8000000000001, 0xFFF8000000000002,
            0x7FF0000000000003]


def dict_case(n_off=256, n_val=256, nan=False):
    """pattern 0 (7 offsets, values -1 and 6), pairs of rows [(o, -1), (0, 6)] with one more offset o each up to n_off
    offsets, and 255 single rows of pattern 0's structure whose diagonals bring the distinct values to n_val (the rest
    repeat the first).  nan: the rows of six offsets carry the all-ones NaN, +0.0, -0.0 and NaNs with other payloads
    instead of -1."""
    offs = EXTRA_OFFSETS[: n_off - 7]
    shapes = [P7, B1] + [sorted([(o, -1.0), (0, 6.0)]) for o in offs]
    specials = len(NAN_BITS) if nan else 0
    fresh = n_val - 2 - specials
    ks = [k if k <= fresh else 1 for k in range(1, 256)]
    groups = [(2 + i, 2, None) for i in range(len(offs))] + [(0, 1, 6.0 + k * EPS) for k in ks]
    M = build(20000, shapes, groups, seed=14)
    if nan:
        rows = np.repeat(np.arange(M.nrow), np.diff(M.rowptr))
        at = [np.flatnonzero(M.colindex - rows == o) for o in offs[:specials]]
        M = with_bits(M, np.concatenate(at), np.repeat(np.array(NAN_BITS, dtype=np.uint64), [a.size for a in at]))
    # table: pattern 0, the boundary row, the offset pairs and the rows repeating the first diagonal (two rows or
    # more each), then the first single rows
    dup = 255 - fresh
    slots = 255 - 2 - len(offs)
    tabulated = (1 + dup) + (slots - 1) if dup else slots
    ok = n_off <= 256 and n_val <= 256
    return M, dict(pat=(255, 8 + 2 * len(offs) + 7 * slots, 255 - tabulated), dict=(n_val, n_off) if ok else None,
                   kind="stream")


def rect_case():
    """a stencil block of nrow x (nrow + halo) with a diagonal: the shape of a multi-GPU local block.  The last rows
    reach into the halo columns."""
    M = build(20000, [P7, B1], [(0, 1000, 6.0 + EPS)], seed=15, halo=H)
    return M, dict(pat=(3, 15, 0), dict=(3, 7), kind="stream")


CASES = {
    **{f"patterns-{t}": (lambda t=t: patterns_case(t)) for t in (254, 255, 256, 300)},
    **{f"cand-{d}": (lambda d=d: candidates_case(d)) for d in (1 << 15, (1 << 15) + 1)},
    "cand-105000+35000": lambda: candidates_case(35002),
    "table-27": lambda: table_case(False),
    "table-full": lambda: table_case(True),
    "entries-2048": lambda: entries_exact_case(56),
    "entries-2049": lambda: entries_exact_case(57),
    "entries-skip": lambda: entries_skip_case(False),
    "entries-merged": lambda: entries_skip_case(True),
    "rowlen-64": lambda: row_length_case(64),
    "rowlen-65": lambda: row_length_case(65),
    **{f"len0-{m}": (lambda m=m: len0_case(m)) for m in (1, 2, 3, 4, 5, 6, 7, 8, 9, 27, 32, 33)},
    "cover-half": lambda: cover_half_case(0),
    "cover-half-1": lambda: cover_half_case(1),
    "cover-75": lambda: cover_quarter_case(0),
    "cover-75-1": lambda: cover_quarter_case(1),
    "mask-repeat": mask_repeat_case,
    "mask-order": mask_order_case,
    "mask-zero": mask_zero_case,
    "dict-256": lambda: dict_case(),
    "dict-257v": lambda: dict_case(n_val=257),
    "dict-257o": lambda: dict_case(n_off=257),
    "dict-nan-256": lambda: dict_case(nan=True),
    "dict-nan-257": lambda: dict_case(n_val=257, nan=True),
    "rect": rect_case,
}


@lru_cache(maxsize=None)
def case(name):
    return CASES[name]()


def base_kind(M):
    """choose_kernel (matrix.cu): the family from the row statistics, before any twin"""
    rp = M.rowptr.astype(np.int64)
    n = M.nrow
    i = np.arange(n)
    max_row = int(np.diff(rp).max())
    mean = M.nnz / n
    threads = 256 if mean <= 12.0 else 128
    win = int((rp[np.minimum(i + threads, n)] - rp[i]).max())
    smem = (((win + 8) + 3) & ~3) * 12
    if mean <= 2.5 and max_row <= 8:
        return "scalar"
    if smem <= 96 * 1024 and max_row <= 8 * mean + 16:
        return "stream"
    return "vector"


def caller_diag(M):
    """the extracted diagonal with a few rows moved by one ulp: those rows become escapes"""
    d = M.diagonal()
    rows = np.random.default_rng(M.nrow).choice(M.nrow, 7, replace=False)
    d[rows] = np.nextafter(d[rows], np.inf)
    return d


def table_masks(enc):
    """sparsh_pattern_masks of the host encoder's table"""
    from test_pattern_masks import masks

    _, ent_val, ent_off, start, n_pat, _ = enc
    return masks([list(zip(ent_off[start[p]:start[p + 1]], ent_val[start[p]:start[p + 1]])) for p in range(n_pat)])


def host_twins(M, diag=None):
    """what the host encoders make of M: pattern table (with the smoothing diagonal `diag`), its masks and dictionary
    sizes"""
    enc = _pattern_encode(M, None if diag is None else np.ascontiguousarray(diag))
    pat, _, _, start, n_pat, n_esc = enc
    _, dval, doff = _dict_encode(M)
    n = M.nrow
    m = table_masks(enc)
    p = pat[:n]
    rows_masked = np.count_nonzero((p == 0) | ((p != ESC) & (m[p] & VALID != 0))) if n_pat else 0
    return dict(enc=enc, n_pat=n_pat, n_ent=int(start[-1]) if n_pat else 0, n_esc=n_esc,
                cover0=np.count_nonzero(p == 0) / n if n_pat else 0.0, covered=n - n_esc,
                len0=int(start[1] - start[0]) if n_pat else 0, dict=(len(dval), len(doff)) if len(dval) else None,
                masked=int(np.count_nonzero(m[1:n_pat] & VALID)), cover_masked=rows_masked / n)


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", list(CASES))
def test_generator_reaches_its_limit(name):
    """the host encoders see exactly the intended pattern, entry, escape and dictionary counts"""
    M, want = case(name)
    h = host_twins(M)
    assert base_kind(M) == want["kind"], name
    assert (h["n_pat"], h["n_ent"], h["n_esc"]) == want["pat"], name
    assert h["dict"] == want["dict"], name
    if "cover0" in want:
        assert h["cover0"] == want["cover0"], name
    if "masked" in want:
        assert h["masked"] == want["masked"], name
    if h["n_pat"]:
        _check_pattern_decode(M, *h["enc"])


def test_limits_sit_on_both_sides():
    """the pairs the value-update tests cross: same sparsity, opposite sides of the limit"""
    n = 20000
    assert host_twins(case("cover-half")[0])["cover0"] == 0.5 and host_twins(case("cover-half-1")[0])["cover0"] < 0.5
    assert host_twins(case("cover-75")[0])["covered"] == 0.75 * n
    assert host_twins(case("cover-75-1")[0])["covered"] == 0.75 * n - 1
    for a, b in CROSSINGS:
        A, B = case(a)[0], case(b)[0]
        assert A.nrow == B.nrow and np.array_equal(A.rowptr, B.rowptr) and np.array_equal(A.colindex, B.colindex), (a, b)
        assert not np.array_equal(A.val.view(np.uint64), B.val.view(np.uint64)), (a, b)


def test_candidate_limit_is_the_device_encoders():
    """more than 2^15 distinct rows: the host encoder declines as the device encoder does, even where the rows it would
    tabulate cover 3/4 of the matrix (105 000 identical rows, 35 000 distinct ones)"""
    M, _ = case("cand-105000+35000")
    assert (105000 + 2 * H + 253) / M.nrow >= 0.75
    assert host_twins(M)["n_pat"] == 0
    assert host_twins(case("cand-32768")[0])["n_pat"] == 255
    assert host_twins(case("cand-32769")[0])["n_pat"] == 0


# ------------------------------------------------------------------------------------------------------------ GPU
CROSSINGS = [("patterns-255", "patterns-256"), ("patterns-254", "patterns-300"), ("cand-32768", "cand-32769"),
             ("cover-half", "cover-half-1"), ("cover-75", "cover-75-1"), ("entries-skip", "entries-merged"),
             ("table-27", "table-full"), ("table-full", "table-27"), ("dict-256", "dict-257v"),
             ("dict-nan-256", "dict-nan-257")]
ENVS = {"default": {}, "no-pattern": {"SPARSH_PATTERN": "0"}, "dict-always": {"SPARSH_DICT": "2"}}


@pytest.fixture(scope="module")
def sp():
    import sparsh_amg_b200 as s

    s.init(0)
    return s


def same_bits(got, want, msg):
    """NaN where the other has NaN, the same bits everywhere else (-0 and +0 differ).  A NaN's payload and sign are not
    compared: of two NaN operands an add keeps either one's."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (msg, got.shape, want.shape)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(np.ascontiguousarray(got[~nan]).view(np.uint64), np.ascontiguousarray(want[~nan]).view(np.uint64),
                                  err_msg=msg)


def set_env(monkeypatch, env):
    for k in ("SPARSH_PATTERN", "SPARSH_DICT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in ENVS[env].items():
        monkeypatch.setenv(k, v)


def has_twin(sp, dA, kind):
    """can the family run on this matrix (is its twin there)?  Leaves the matrix on that family when it can."""
    try:
        dA.force_kernel(kind, 128)
        return True
    except sp.SparshError:
        return False


def describe(dA):
    epis = ["spmv", "residual", "jacobi", "prolong", "sor", "spmv_dot", "resnorm"]
    return (dA.kernel(), [dA.kernel_name(e) for e in epis], dA.pattern_stats(), dA.pattern_mask_stats(), dA.transfer_info())


@pytest.mark.gpu
@pytest.mark.parametrize("env", list(ENVS))
@pytest.mark.parametrize("name", list(CASES))
def test_device_encoders_decide_as_the_host_encoders(sp, monkeypatch, name, env):
    """upload with the extracted and with a caller's diagonal: the twins, their statistics and the kernel family are
    the ones the host encoders' results call for"""
    set_env(monkeypatch, env)
    M, want = case(name)
    pmode = int(ENVS[env].get("SPARSH_PATTERN", "1"))
    dmode = int(ENVS[env].get("SPARSH_DICT", "1"))
    stream = base_kind(M) == "stream"
    for diag in (None, caller_diag(M)):
        msg = f"{name} {env} {'caller' if diag is not None else 'extracted'} diagonal"
        h = host_twins(M, diag)
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        pat = stream and pmode > 0 and h["n_pat"] > 0 and h["covered"] >= 0.75 * M.nrow
        dic = stream and h["dict"] is not None and (dmode == 2 or (dmode == 1 and not (pat and pmode == 1)))
        stats, mask_stats = dA.pattern_stats(), dA.pattern_mask_stats()
        if pat:
            assert stats == (h["n_pat"], h["n_ent"], h["n_esc"], h["cover0"]), msg
            assert mask_stats == (h["masked"], h["cover_masked"]), msg
        else:
            assert stats == (0, 0, M.nrow, 0.0) and mask_stats == (0, 0.0), msg
        kind, threads, _ = dA.kernel()
        lean = pat and h["len0"] in (5, 7) and h["cover0"] >= 0.5
        if pat and pmode == 1:
            assert (kind, threads) == (KIND["pattern"], 128), msg
            family = "csr_pat2_kernel" if lean else "csr_pattern_kernel"
            for e in ("spmv", "residual", "jacobi", "prolong", "spmv_dot", "resnorm"):
                assert dA.kernel_name(e).startswith(family), (msg, e, dA.kernel_name(e))
        elif dic:
            assert (kind, threads) == (KIND["dict"], 128), msg
        else:
            assert kind == KIND[base_kind(M)], msg
        assert has_twin(sp, dA, KIND["dict"]) == dic, msg
        assert has_twin(sp, dA, KIND["pattern"]) == pat, msg


# ---- kernels against the oracle
def two_product(a, b):
    """p = fl(a*b) and e with a*b = p + e exactly (Dekker), for finite a, b"""
    def split(x):
        c = 134217729.0 * x
        hi = c - (c - x)
        return hi, x - hi

    p = a * b
    ah, al = split(a)
    bh, bl = split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


@np.errstate(all="ignore")
def exact_dot(a, b):
    """(correctly rounded sum of a_i * b_i, sum of |a_i * b_i|); the non-finite cases by IEEE rules"""
    p = a * b
    if not np.all(np.isfinite(p)):
        return float(np.sum(p)), math.inf
    p, e = two_product(a, b)
    return math.fsum(np.concatenate([p, e])), math.fsum(np.abs(p))


def assert_reduction(got, exact, scale, n, msg):
    if not math.isfinite(exact):
        assert (math.isnan(got) and math.isnan(exact)) or got == exact, (msg, got, exact)
        return
    assert abs(got - exact) <= 2 * n * 2.0 ** -53 * scale, (msg, got, exact, scale)


def aggregation(oracle, M):
    """R = P^T of the oracle's HEM aggregation of M's square part (unit weights: the same R for every value set)"""
    rows = np.repeat(np.arange(M.nrow), np.diff(M.rowptr))
    keep = M.colindex < M.nrow
    rp = np.zeros(M.nrow + 1, dtype=np.int64)
    rp[1:] = np.cumsum(np.bincount(rows[keep], minlength=M.nrow))
    S = CSR(M.nrow, M.nrow, rp, M.colindex[keep], np.where(M.colindex[keep] == rows[keep], 6.0, -1.0))
    nc, agg = oracle.hem(S, 0)
    assert 0 < nc <= M.nrow and agg.min() >= 0 and agg.max() < nc
    return CSR(M.nrow, nc, np.arange(M.nrow + 1), agg, np.ones(M.nrow))


def special_x(M, enc, x):
    """x holding Inf, NaN and -0 next to escape rows and at the columns that masked rows skip"""
    pat, ent_val, ent_off, start, n_pat, _ = enc
    x = x.copy()
    cols = []
    esc = np.flatnonzero(pat[: M.nrow] == ESC) if n_pat else np.arange(M.nrow)  # no table: every row is CSR
    for r in esc[np.linspace(0, esc.size - 1, min(6, esc.size)).astype(int)]:
        cols += [c for c in (r - 1, r + 1) if 0 <= c < M.ncol]
    if n_pat:
        m = table_masks(enc)
        off0 = ent_off[start[0]:start[1]]
        for p in range(1, n_pat):
            if m[p] & VALID and len(cols) < 24:
                r = np.flatnonzero(pat[: M.nrow] == p)[0]
                cols += [r + o for k, o in enumerate(off0) if not m[p] & (1 << k) and 0 <= r + o < M.ncol][:2]
    cols += [M.ncol - 1, M.ncol - 2] if M.ncol > M.nrow else []
    if not cols:  # nothing escapes and nothing is masked: spread them
        cols = list(np.linspace(0, M.ncol - 1, 6).astype(int))
    for i, c in enumerate(cols):
        x[c] = (np.inf, np.nan, -0.0)[i % 3]
    return x


@np.errstate(all="ignore")  # Inf and NaN in x or in the matrix are part of the cases
def reference(oracle, M, diag, P, x, b, xc, xf):
    square = M.nrow == M.ncol
    r = oracle.store_residual(M, b, x)
    y = oracle.spmv(M, x)
    out = dict(spmv=y, residual=r, prolong=oracle.transfer_solution(M, xc, xf), rr=oracle.transfer_residual(P, r))
    if diag is not None:
        out["jacobi_zero"] = (OMEGA * b) / diag
    if square:
        out["jacobi2"] = oracle.jacobi(M, diag, b, x, OMEGA, 1)
        out["jacobi7"] = oracle.jacobi(M, diag, b, x, OMEGA, 6)
        out["spmv_dot"] = y
        out["dot"] = exact_dot(x, y)
    out["resnorm"] = exact_dot(r, r)
    return out


def device_ops(sp, dA, dR, keys, x, b, xc, xf):
    V = sp.DeviceVector
    out = dict(spmv=dA.spmv(V(data=x)).download(), residual=dA.residual(V(data=b), V(data=x)).download(),
               prolong=dA.prolong_add(V(data=xc), V(data=xf)).download(), rr=dA.residual_restrict(dR, V(data=b), V(data=x)).download(),
               resnorm=dA.residual_norm(V(data=b), V(data=x)))
    if "jacobi_zero" in keys:
        out["jacobi_zero"] = dA.jacobi_zero(V(data=b), OMEGA).download()
    if "jacobi2" in keys:
        out["jacobi2"] = dA.jacobi(V(data=b), V(data=x), OMEGA, 2).download()
        out["jacobi7"] = dA.jacobi(V(data=b), V(data=x), OMEGA, 7).download()
        y, out["dot"] = dA.spmv_dot(V(data=x))
        out["spmv_dot"] = y.download()
    return out


def families(sp, dA):
    K = sp.capi
    fams = [(K.KIND_SCALAR, 256), (K.KIND_STREAM, 128), (K.KIND_STREAM, 256)]
    for kind in (K.KIND_PATTERN, K.KIND_DICT):
        if has_twin(sp, dA, kind):
            fams += [(kind, 128), (kind, 256)]
    return fams


def check_against_oracle(sp, oracle, dA, dR, M, diag, P, x, b, xc, xf, msg):
    want = reference(oracle, M, diag, P, x, b, xc, xf)
    ran = []
    for kind, tl in families(sp, dA):
        dA.force_kernel(kind, tl)
        got = device_ops(sp, dA, dR, want, x, b, xc, xf)
        m = f"{msg} kind {kind}/{tl} {dA.kernel_name('spmv')}"
        for key, w in want.items():
            if key == "dot":
                assert_reduction(got["dot"], w[0], w[1], M.nrow, m + " spmv_dot")
            elif key == "resnorm":
                assert_reduction(got["resnorm"] ** 2, w[0], w[1], M.nrow + 2, m + " resnorm")
            else:
                same_bits(got[key], w, f"{m} {key}")
        ran.append(dA.kernel_name("jacobi" if "jacobi2" in want else "spmv").split("<")[0])
    return ran


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_every_family_matches_the_oracle(sp, oracle, monkeypatch, name):
    """every kernel family the matrix supports (both twins built) against the oracle, bit for bit; the fused dot and
    residual norm within the bound of an n-term sum of the exact products"""
    set_env(monkeypatch, "dict-always")
    M, _ = case(name)
    P = aggregation(oracle, M)
    dR = sp.DeviceMatrix.from_csr(P, transpose=True)
    rng = np.random.default_rng(41)
    x, b = rng.standard_normal(M.ncol), rng.standard_normal(M.nrow)
    xc, xf = rng.standard_normal(M.ncol), rng.standard_normal(M.nrow)
    square = M.nrow == M.ncol
    for diag in (None, caller_diag(M)):  # a rectangular block without a given diagonal has none: no smoothing
        dg = diag if diag is not None else M.diagonal() if square else None
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        enc = host_twins(M, diag)["enc"]
        ran = []
        for xs in (x, special_x(M, enc, x)):
            ran += check_against_oracle(sp, oracle, dA, dR, M, dg, P, xs, b, xc, xf, name)
        if dA.pattern_stats()[0]:
            assert any(r.startswith("csr_pat") for r in ran), (name, ran)


# ---- value updates across each limit
def assert_same_matrix(sp, oracle, got, want, M, P, msg):
    """got (updated) and want (fresh upload of the same values): every choice, the arrays, and every op of every family
    bit for bit (the reductions too: same kernel, same summation tree)"""
    assert describe(got) == describe(want), msg
    for a, b_, what in zip(got.fetch(), want.fetch(), ("rowptr", "colindex", "val", "diag")):
        same_bits(np.asarray(a, dtype=np.float64), np.asarray(b_, dtype=np.float64), f"{msg} {what}")
    fams = families(sp, want)
    assert families(sp, got) == fams, msg
    rng = np.random.default_rng(43)
    x, b, xc, xf = (rng.standard_normal(M.nrow) for _ in range(4))
    dR = sp.DeviceMatrix.from_csr(P, transpose=True)
    keys = ("jacobi_zero", "jacobi2")
    for kind, tl in fams:
        got.force_kernel(kind, tl)
        want.force_kernel(kind, tl)
        g, w = device_ops(sp, got, dR, keys, x, b, xc, xf), device_ops(sp, want, dR, keys, x, b, xc, xf)
        for key in w:
            same_bits(g[key], w[key], f"{msg} kind {kind}/{tl} {key}")


@pytest.mark.gpu
@pytest.mark.parametrize("env", list(ENVS))
@pytest.mark.parametrize("pair", CROSSINGS, ids=[f"{a}>{b}" for a, b in CROSSINGS])
def test_value_update_across_a_limit_equals_a_fresh_upload(sp, oracle, monkeypatch, pair, env):
    """upload one side, update the values to the other side and back: each time the matrix equals a fresh upload of the
    values it now holds (the device encoders' gather path and the reuse of the earlier table arrays)"""
    set_env(monkeypatch, env)
    A, B = case(pair[0])[0], case(pair[1])[0]
    P = aggregation(oracle, A)
    dA = sp.DeviceMatrix.from_csr(A)
    for step, M in enumerate((B, A)):
        dA.update_values(M.val)
        assert_same_matrix(sp, oracle, dA, sp.DeviceMatrix.from_csr(M), M, P, f"{pair} {env} step {step}")


@pytest.mark.gpu
def test_refresh_across_the_cover_limit(sp):
    """a hierarchy refresh whose level-0 values leave fewer than 3/4 of the rows tabulated (the twin goes, coarse levels
    change with the Galerkin products), then the original values (the twin returns)"""
    from test_refresh import assert_levels_equal, assert_same_hierarchy, extracted_diag, galerkin_levels, hierarchy_state, host_levels

    levels, amg, _ = host_levels("hem", 24)
    A0 = levels[0]["A"]
    n = A0.nrow
    lens = np.diff(A0.rowptr)
    rows = np.random.default_rng(47).choice(np.flatnonzero(lens == 7), int(0.3 * n), replace=False)
    rs = np.repeat(np.arange(n), np.diff(A0.rowptr))
    dpos = np.flatnonzero(A0.colindex == rs)
    v = A0.val.copy()
    v[dpos[rows]] += np.arange(1, rows.size + 1) * EPS
    A1 = CSR(n, n, A0.rowptr, A0.colindex, v)
    assert host_twins(A0)["covered"] >= 0.75 * n > host_twins(A1)["covered"]
    dH = sp.DeviceHierarchy(levels, use_graph=False)
    before = hierarchy_state(dH)
    assert dH.level(0)[0].pattern_stats()[0] > 0
    dH.refresh(A1.val)
    assert dH.level(0)[0].pattern_stats()[0] == 0
    fresh = sp.DeviceHierarchy(galerkin_levels(sp, A1, extracted_diag(A1), levels), use_graph=False)
    assert_same_hierarchy(sp, dH, fresh, len(levels), "below the cover limit")
    fresh.free()
    dH.refresh(A0.val, diag=levels[0]["diag"])
    assert hierarchy_state(dH) == before
    assert_levels_equal(sp, dH, levels, "back")
    dH.free()
    amg.free()
