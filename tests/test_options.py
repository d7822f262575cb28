"""The test options on every kernel route, and the p-value at the edges of its formula.

Three options turn U into a p-value -- ``alternative`` (two-sided / less / greater), ``use_continuity`` and
``tie_correct`` -- and the score plane adds a fourth.  Each kernel route wires them on its own: ``ovo_kernel`` from a
per-group table, ``ovr_kernel`` and ``ovr_table_kernel`` through ``compute_pval``, the fused epilogue (narrow, wide and
SCORE instantiations, shared by the dense and CSR passes) from ``fused_group_kernel``'s constants and, for
one-versus-rest, the gene's tie correction stored by ``fused_gene_kernel``.  Every route below runs all 12 option
combinations with ``score=True`` against ``oracle.run`` with the same flags, and each route's matrix plants the
statistics where the formula changes regime: U exactly at its mean, |U - mu| = 1/2, pairs in which every cell is tied,
p-values from 1e-260 through the subnormals to exactly 0, a single group and two groups of one-versus-rest.  The
profile shows that each route's kernel ran.  Last, ``illico_bh_adjust`` is compared bit for bit with statsmodels'
Benjamini-Hochberg restated in numpy, at the sizes and values where its sort and reverse running minimum go wrong."""
import functools
import zlib
from collections import namedtuple

import numpy as np
import pytest

import oracle
from tests.golden import cases as C
from tests.parity import assert_parity
from tests.test_dtypes import _debug
from tests.test_limits import _assert_exact, _plant, _pool, cap
from tests.test_rank_genes import bh_reference, score_reference
from tests.util import FakeAnnData

OPTIONS = [(alt, cc, tc) for alt in C.ALTERNATIVES for cc in (True, False) for tc in (True, False)]
DBL_MIN = float(np.finfo(np.float64).tiny)     # smallest normal double

# ---------------------------------------------------------------------------------------------------------------
# the planted matrices
#
# Group sizes.  The tail groups are completely separated from their partner (the control, or the rest of the cells) in
# the tail genes; their sizes put the z of full separation, sqrt(3 n_r n_t / (n_r + n_t + 1)), at about 34.6 (p near
# 1e-262), 37.3 / 37.7 / 38.1 / 38.5 (p subnormal: the window is z = 37.55 .. 38.5) and 38.9 and above (p = 0).
# "A" is the pair of the mean regimes: the control (one-versus-reference) or the rest (one-versus-rest) holds an integer
# multiple of A's cells.
OVO_SIZES = {"ctrl": 2000, "A": 500, "t604": 604, "t621": 621, "t639": 639, "t657": 657, "t675": 675, "P": 1100, "s40": 40}
OVR_SIZES = {"A": 600, "t430": 430, "t510": 510, "t520": 520, "t530": 530, "t540": 540, "t560": 560, "t650": 650,
             "s40": 40, "big": 1620}
OVO_TAIL = ("A", "t604", "t621", "t639", "t657", "t675", "P")
OVR_TAIL = ("t430", "t510", "t520", "t530", "t540", "t560", "t650")

# Alphabets: integer codes 0 .. K and the monotone map from a code to a cell value (code 0 -> 0).  The planted genes
# draw even codes, so that an odd code is a value strictly between two of them.
#   narrow:  <= 12 distinct non-zero values per gene (fused narrow table, CSR pass, ovr_table_kernel's <= T_CAP)
#   wide:    13 .. 64 distinct integers (fused wide table)
#   hist:    21 .. 2048 distinct multiples of 1/16 (ovr_kernel path H)
#   cont:    more than 2048 distinct multiples of 1/1024 (ovr_kernel path S; ovo_kernel's sorted and hashed tiers)
#   recoded: <= 12 distinct non-zero multiples of 1/10 in float64, which float32 cannot hold (recoded per batch)
ALPHABETS = {
    "narrow": (12, lambda c: c.astype(np.float32)),
    "wide": (60, lambda c: c.astype(np.float32)),
    "hist": (400, lambda c: (c / 16.0).astype(np.float32)),
    "cont": (30000, lambda c: (c / 1024.0).astype(np.float32)),
    "recoded": (12, lambda c: c / 10.0),
}
N_GENES = 32


def _labels(sizes, rng):
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    return labels


def _ovo_tier_genes(labels, rng):
    """One gene on each side of every tier cap of ovo_kernel (as test_limits plants them): control non-zeros at REF_CAP,
    distinct control values at DT_CAP and ST_CAP (hashed and sorted), values of group A the control lacks at NE_CAP,
    non-zeros of group P at STREAM_MAX, WARP_CAP / 2 and WARP_CAP."""
    n = labels.size
    ctrl, A, P = (np.flatnonzero(labels == x) for x in ("ctrl", "A", "P"))
    genes = []

    def gene(ctrl_nnz, ctrl_distinct):
        col = np.zeros(n, np.float32)
        pool = _pool(ctrl_distinct, len(genes))
        _plant(col, ctrl, ctrl_nnz, pool, rng)
        extra = pool[-1] + 0.25 + np.arange(1, 9, dtype=np.float32) / 4
        for g in np.unique(labels[labels != "ctrl"]):
            _plant(col, np.flatnonzero(labels == g), 6, np.concatenate([pool[:3], extra[:1]]), rng)
        genes.append(col)
        return col

    REF_CAP, DT_CAP, NE_CAP, ST_CAP, W = cap("REF_CAP"), cap("DT_CAP"), cap("NE_CAP"), cap("ST_CAP"), cap("WARP_CAP")
    for k in (REF_CAP, REF_CAP + 1):
        gene(k, k)
    for d in (DT_CAP, DT_CAP + 1):
        gene(1500, d)
    for e in (NE_CAP, NE_CAP + 1):
        col = gene(1500, 10)
        col[A] = 0
        absent = (_pool(10, 99)[:e] + 100.0).astype(np.float32)
        _plant(col, A, 60, np.concatenate([absent, col[ctrl][col[ctrl] > 0][:5]]), rng)
    for d in (ST_CAP, ST_CAP + 1):
        gene(REF_CAP + 300, d)               # hashed: more than REF_CAP control non-zeros
    for d in (ST_CAP, ST_CAP + 1):
        gene(REF_CAP - 100, d)               # sorted
    for m in (cap("STREAM_MAX"), cap("STREAM_MAX") + 1, W // 2, W // 2 + 1, W, W + 1):
        col = gene(1500, 200)
        col[P] = 0
        _plant(col, P, m, np.concatenate([col[ctrl][col[ctrl] > 0][:150], _pool(400, 7) + 50]), rng)
    return genes


def _holds(alphabet, test):
    """Regimes the route can hold: on ovr_kernel's routes a gene with few distinct values goes to ovr_table_kernel, and
    on path S (> 2048 distinct values) the rest cannot hold A's multiset an integer number of times."""
    out = {"tail"}
    if not (test == "ovr" and alphabet in ("hist", "cont")):
        out |= {"tie_zero", "tie_const"}
    if not (test == "ovr" and alphabet == "cont"):
        out |= {"mu", "half"}
    return out


@functools.lru_cache(maxsize=None)
def _case(alphabet, test, tiers=False):
    """(X, labels, meta): about 6 000 - 7 000 cells x 32 (48 with the tiers) genes of `alphabet`.  meta: gene index of
    each planted regime; "tail": (gene, group, direction) with direction +1 when the group holds the high values."""
    K, f = ALPHABETS[alphabet]
    rng = np.random.RandomState(zlib.crc32(f"{alphabet}:{test}:{tiers}".encode()))
    sizes = OVO_SIZES if test == "ovo" else OVR_SIZES
    labels = _labels(sizes, rng)
    n = labels.size
    inA = labels == "A"
    partner = labels == "ctrl" if test == "ovo" else ~inA
    r = int(partner.sum()) // int(inA.sum())
    assert r * inA.sum() == partner.sum()
    holds = _holds(alphabet, test)
    cols, meta = [], {"tail": []}

    def add(name, codes):
        meta[name] = len(cols)
        cols.append(codes)

    def even(size):
        return 2 * rng.randint(0, K // 2 + 1, size)

    if "mu" in holds:
        # the partner holds A's multiset r times: U = mu exactly
        a = even(inA.sum())
        c = np.zeros(n, np.int64)
        c[inA] = a
        c[partner] = rng.permutation(np.repeat(a, r))
        c[~(inA | partner)] = even((~(inA | partner)).sum())
        add("mu", c)
        # the same, with one code held once by A and r times by the partner; one of those r moves one code up
        # (a value between it and the next, which A does not hold): |U - mu| = 1/2
        h = c.copy()
        v = 2 * (K // 4)
        a2 = np.where(a == v, v + 2 if v + 2 <= K else v - 2, a)
        a2[0] = v
        h[inA] = a2
        h[partner] = rng.permutation(np.repeat(a2, r))
        h[np.flatnonzero(partner & (h == v))[0]] += 1
        add("half", h)
    if "tie_zero" in holds:
        c = np.zeros(n, np.int64)
        if test == "ovo":
            others = ~(inA | partner)
            c[others] = even(others.sum())
        add("tie_zero", c)
        c = c.copy()
        c[inA | partner] = 2
        add("tie_const", c)
    for g in (OVO_TAIL if test == "ovo" else OVR_TAIL):
        inG = labels == g
        for d in (1, -1):
            lo, hi = rng.randint(0, K // 2, n), rng.randint(K // 2 + 1, K + 1, n)
            meta["tail"].append((len(cols), g, d))
            cols.append(np.where(inG == (d > 0), hi, lo))
    genes = [f(c) for c in cols]
    if tiers:
        genes += _ovo_tier_genes(labels, rng)
    width = N_GENES if not tiers else 48
    while len(genes) < width:
        c = rng.randint(1, K + 1, n) * (rng.rand(n) < 0.6)
        genes.append(f(c))
    X = np.stack(genes, axis=1)
    return X, labels, meta


# ---------------------------------------------------------------------------------------------------------------
# the route table

Route = namedtuple("Route", "fmt test alphabet env kernels absent fused_var")
_SHARE = {"ILLICO_FUSED_LIST_SHARE": "1.0"}     # genes a fused pass cannot hold go back one by one
ROUTES = {
    "dense_ovo_fused_narrow": Route("dense", "ovo", "narrow", {"ILLICO_FUSED_WIDE": "0", **_SHARE},
                                    ("fused_pass_kernel", "fused_epilogue_kernel"), ("fused_wide_pass_kernel",),
                                    "ILLICO_OVO_FUSED"),
    "dense_ovo_fused_wide": Route("dense", "ovo", "wide", _SHARE, ("fused_wide_pass_kernel", "fused_wide_epilogue_kernel"),
                                  (), "ILLICO_OVO_FUSED"),
    "dense_ovo_general": Route("dense", "ovo", "tiers", {"ILLICO_OVO_FUSED": "0"}, ("ovo_kernel",),
                               ("fused_pass_kernel",), None),
    "dense_ovr_fused": Route("dense", "ovr", "narrow", _SHARE, ("fused_pass_kernel", "fused_epilogue_kernel"), (),
                             "ILLICO_OVR_FUSED"),
    "dense_ovr_table": Route("dense", "ovr", "narrow", {"ILLICO_OVR_FUSED": "0"}, ("ovr_table_kernel",),
                             ("fused_pass_kernel",), None),
    "dense_ovr_path_h": Route("dense", "ovr", "hist", {"ILLICO_OVR_FUSED": "0"}, ("ovr_kernel",), ("fused_pass_kernel",),
                              None),
    "dense_ovr_path_s": Route("dense", "ovr", "cont", {"ILLICO_OVR_FUSED": "0"}, ("ovr_kernel",), ("fused_pass_kernel",),
                              None),
    "csr_ovo_fused": Route("csr", "ovo", "narrow", _SHARE, ("fused_csr_pass_kernel", "fused_epilogue_kernel"), (),
                           "ILLICO_CSR_FUSED"),
    "csr_ovr_fused": Route("csr", "ovr", "narrow", _SHARE, ("fused_csr_pass_kernel", "fused_epilogue_kernel"), (),
                           "ILLICO_CSR_FUSED"),
    "csr_ovo_general": Route("csr", "ovo", "cont", {"ILLICO_CSR_FUSED": "0"}, ("ovo_kernel",),
                             ("fused_csr_pass_kernel",), None),
    "csr_ovr_general": Route("csr", "ovr", "hist", {"ILLICO_CSR_FUSED": "0"}, ("ovr_kernel",),
                             ("fused_csr_pass_kernel",), None),
    "csc_ovo": Route("csc", "ovo", "narrow", {}, ("ovo_kernel",), ("fused_pass_kernel", "fused_csr_pass_kernel"), None),
    "csc_ovr": Route("csc", "ovr", "narrow", {}, ("ovr_table_kernel",), ("fused_pass_kernel", "fused_csr_pass_kernel"),
                     None),
    "recoded_dense_ovo": Route("dense", "ovo", "recoded", _SHARE, ("wide_collect_dense_kernel", "fused_pass_kernel"), (),
                               "ILLICO_OVO_FUSED"),
    "recoded_dense_ovr": Route("dense", "ovr", "recoded", {}, ("wide_collect_dense_kernel", "ovr_kernel"), (), None),
    "recoded_csr_ovo": Route("csr", "ovo", "recoded", _SHARE, ("wide_collect_csr_kernel", "fused_csr_pass_kernel"), (),
                             "ILLICO_CSR_FUSED"),
    "recoded_csr_ovr": Route("csr", "ovr", "recoded", {}, ("wide_collect_csr_kernel", "ovr_kernel"), (), None),
    "recoded_csc_ovo": Route("csc", "ovo", "recoded", {}, ("wide_collect_csc_kernel", "ovo_kernel"), (), None),
    "recoded_csc_ovr": Route("csc", "ovr", "recoded", {}, ("wide_collect_csc_kernel", "ovr_kernel"), (), None),
}
OVR_ROUTES = [k for k, r in ROUTES.items() if r.test == "ovr"]


def _route_case(name):
    r = ROUTES[name]
    if r.alphabet == "tiers":
        X, labels, meta = _case("cont", r.test, tiers=True)
    else:
        X, labels, meta = _case(r.alphabet, r.test)
    return C.to_format(X, r.fmt), labels, meta


@functools.lru_cache(maxsize=None)
def _want(name, alt, cc, tc, labels_key=None):
    """oracle.run on the route's matrix (float64 values): (groups, p, U, fc, ties)."""
    Xf, labels, _ = _route_case(name)
    if labels_key is not None:
        labels = _two_group_labels(labels)
    r = ROUTES[name]
    ref = "ctrl" if r.test == "ovo" else None
    return oracle.run(Xf, labels, ref, want_ties=True, alternative=alt, use_continuity=cc, tie_correct=tc,
                      n_threads=oracle.max_threads())


# ============================================ CPU ==============================================================

@pytest.mark.parametrize("name", list(ROUTES))
def test_route_cases_plant_what_they_claim(name):
    """Distinct values per gene fit the route; U sits exactly at mu and mu -/+ 1/2 in the mean regimes, every cell of the
    pair is tied in the tie regimes, and the tail genes reach normal p-values below 1e-200, subnormal ones and 0."""
    r = ROUTES[name]
    Xf, labels, meta = _route_case(name)
    X = Xf.toarray() if hasattr(Xf, "toarray") else Xf
    assert 3000 <= X.shape[0] <= 7000 and X.shape[1] % 4 == 0
    assert (X >= 0).all()
    for j in range(X.shape[1] if r.alphabet != "tiers" else N_GENES):
        d = np.unique(X[:, j][X[:, j] != 0]).size
        if r.alphabet in ("narrow", "recoded"):
            assert d <= cap("DCAP") and d <= cap("T_CAP"), (j, d)
        elif r.alphabet == "wide":
            assert np.array_equal(X[:, j], np.round(X[:, j])) and X[:, j].max() <= 64 and (j in meta.values() or d > 12)
        elif r.alphabet == "hist":
            assert cap("T_CAP") < d <= cap("MAX_DISTINCT"), (j, d)
        elif r.test == "ovr":
            assert d > cap("MAX_DISTINCT"), (j, d)
    if r.alphabet == "recoded":
        assert X.dtype == np.float64 and np.any(X.astype(np.float32).astype(np.float64) != X)
    groups, p, U, fc, ties = _want(name, "two-sided", True, True)
    rows = {g: i for i, g in enumerate(groups)}
    a = rows["A"]
    n_a = np.count_nonzero(labels == "A")
    n_p = np.count_nonzero(labels == "ctrl") if r.test == "ovo" else labels.size - n_a
    mu = n_a * n_p / 2.0
    holds = _holds("cont" if r.alphabet == "tiers" else r.alphabet, r.test)
    if "mu" in holds:
        assert U[a, meta["mu"]] == mu and abs(U[a, meta["half"]] - mu) == 0.5
    if "tie_zero" in holds:
        for k in ("tie_zero", "tie_const"):
            pair = (labels == "A") | ((labels == "ctrl") if r.test == "ovo" else (labels != "A"))
            assert np.unique(X[pair, meta[k]]).size == 1, k
    for alt in C.ALTERNATIVES:
        for cc in (True, False):
            for tc in (True, False):
                _, p, U, _, _ = _want(name, alt, cc, tc)
                tail = np.array([p[rows[g], j] for j, g, d in meta["tail"] if alt == "two-sided" or (d > 0) == (alt == "less")])
                what = f"{name}:{alt}:cc={cc}:tc={tc}: tail p {np.sort(tail)}"
                assert (tail == 0).any() and ((tail > 0) & (tail < DBL_MIN)).any() and ((tail > DBL_MIN) & (tail < 1e-200)).any(), what


# ============================================ GPU ==============================================================

@pytest.fixture
def cuda_lib():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from illico_b200 import _lib

    lib = _lib.load()
    before = _lib.launch_count()
    yield lib
    assert _lib.launch_count() > before, "no kernel of libillico_b200.so was launched"


@pytest.fixture
def profile(monkeypatch, cuda_lib):
    """``report()`` -> {kernel name: (ms, launches)} of the launches since the previous ``report()``."""
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_PROFILE", "1")
    _lib.profile_report()
    return _lib.profile_report


def _run(Xf, labels, ref, score=True, **kw):
    """(p, U, fc) planes and the score plane (None without score) of asymptotic_wilcoxon(return_array=True)."""
    from illico_b200 import asymptotic_wilcoxon

    ret = asymptotic_wilcoxon(FakeAnnData(Xf, labels), group_keys="pert", reference=ref, is_log1p=False, score=score,
                              return_array=True, **kw)
    out = ret[2]
    return (out[:, :, 0], out[:, :, 1], out[:, :, 2]), (ret[3]["score"] if score else None)


def _check_route_ran(rep, r, what):
    for k in r.kernels:
        assert k in rep, f"{what}: {k} did not run: {sorted(rep)}"
    for k in r.absent:
        assert k not in rep, f"{what}: {k} ran: {sorted(rep)}"


def _same_bits(a, b, rows, what):
    np.testing.assert_array_equal(a[1][rows], b[1][rows], err_msg=f"{what}: U")
    np.testing.assert_array_equal(a[0][rows], b[0][rows], err_msg=f"{what}: p")


def _score_want(labels, ref, U, ties, n, tc):
    from illico_b200.groups import encode_and_count_groups

    _, grpc = encode_and_count_groups(labels, ref)
    ref_row = grpc.encoded_ref_group if ref is not None else None
    return score_reference(U, ties, grpc.counts, ref_row, n, tc)


@pytest.mark.gpu
@pytest.mark.parametrize("alt,cc,tc", OPTIONS)
@pytest.mark.parametrize("name", list(ROUTES))
def test_options_on_every_route(monkeypatch, profile, name, alt, cc, tc):
    """One route, one (alternative, continuity, tie correction): p, U and fold change against the oracle, the score
    plane bit for bit, score=False bit-identical to score=True, the fused route bit for bit against the general path,
    and the planted regimes."""
    from illico_b200 import dispatch

    r = ROUTES[name]
    Xf, labels, meta = _route_case(name)
    ref = "ctrl" if r.test == "ovo" else None
    kw = dict(alternative=alt, use_continuity=cc, tie_correct=tc)
    groups, p, U, fc, ties = _want(name, alt, cc, tc)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    rows = np.arange(groups.size) != (ref_row if ref_row is not None else -1)
    what = f"{name}:{alt}:cc={cc}:tc={tc}"
    for k, v in r.env.items():
        monkeypatch.setenv(k, v)
    dispatch.clear_caches()
    got, score = _run(Xf, labels, ref, **kw)
    rep = profile()
    _check_route_ran(rep, r, what)
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=what)
    np.testing.assert_array_equal(score, _score_want(labels, ref, U, ties, labels.size, tc), err_msg=f"{what}: score")

    plain, none = _run(Xf, labels, ref, score=False, **kw)
    assert none is None
    _check_route_ran(profile(), r, f"{what} score=False")
    _same_bits(plain, got, rows, f"{what}: score=False")
    if r.alphabet == "recoded":      # (float64 group sums of non-integer values may be added in another order)
        np.testing.assert_allclose(plain[2][rows], got[2][rows], rtol=1e-14, atol=0, err_msg=f"{what}: fold change")
    else:
        np.testing.assert_array_equal(plain[2][rows], got[2][rows], err_msg=f"{what}: fold change")

    if r.fused_var is not None:
        monkeypatch.setenv(r.fused_var, "0")
        general, gscore = _run(Xf, labels, ref, **kw)
        monkeypatch.delenv(r.fused_var)
        grep = profile()
        assert not any(k.startswith("fused_") for k in grep), f"{what}: the fused path was not turned off: {sorted(grep)}"
        _same_bits(got, general, rows, f"{what}: fused vs general path")
        np.testing.assert_array_equal(score, gscore, err_msg=f"{what}: score, fused vs general path")

    # the planted regimes
    gp, gU, _ = got
    a = int(np.searchsorted(groups, "A"))
    holds = _holds("cont" if r.alphabet == "tiers" else r.alphabet, r.test)
    if "mu" in holds:
        j, h = meta["mu"], meta["half"]
        if alt == "two-sided":
            assert gp[a, j] == 1.0, f"{what}: U = mu, p {gp[a, j]!r}"
            assert (gp[a, h] == 1.0) == cc and gp[a, h] <= 1.0, f"{what}: |U - mu| = 1/2, p {gp[a, h]!r}"
    if "tie_zero" in holds:
        for k in ("tie_zero", "tie_const"):
            j = meta[k]
            if tc:
                assert gp[a, j] == 1.0 and score[a, j] == 0.0, f"{what}: {k}: p {gp[a, j]!r}, score {score[a, j]!r}"
    for j, g, d in meta["tail"]:
        i = int(np.searchsorted(groups, g))
        if alt != "two-sided" and (d > 0) != (alt == "less"):
            assert gp[i, j] > 0.999, f"{what}: tail gene {j} ({g}), the other side: p {gp[i, j]!r}"

    if (alt, cc, tc) == OPTIONS[0]:
        # the exact 2U and tie sums of the general path (a dispatcher called with debug= never takes a fused pass)
        dgot, dbg = _debug(r.fmt, r.test, Xf, labels, ref, dict(kw, is_log1p=False))
        assert_parity(dgot, (p, U, fc), ref_row=ref_row, what=f"{what} debug call")
        _assert_exact(dbg, U, ties, ref_row, what)
    dispatch.clear_caches()


def _two_group_labels(labels):
    """The route's groups cut into two: "L" = the first half of the group names, "R" = the others."""
    names = np.unique(labels)
    return np.where(np.isin(labels, names[: names.size // 2]), "L", "R")


@pytest.mark.gpu
@pytest.mark.parametrize("name", OVR_ROUTES)
def test_two_group_one_versus_rest(monkeypatch, profile, name):
    """Two groups: each is the other's rest, so U_L + U_R = n_L n_R and the two-sided p-values are bit-identical."""
    from illico_b200 import dispatch

    r = ROUTES[name]
    Xf, labels, _ = _route_case(name)
    labels2 = _two_group_labels(labels)
    n_l = int(np.count_nonzero(labels2 == "L"))
    for k, v in r.env.items():
        monkeypatch.setenv(k, v)
    dispatch.clear_caches()
    for cc in (True, False):
        for tc in (True, False):
            what = f"{name}: two groups: cc={cc}:tc={tc}"
            groups, p, U, fc, ties = _want(name, "two-sided", cc, tc, labels_key="two")
            got, score = _run(Xf, labels2, None, alternative="two-sided", use_continuity=cc, tie_correct=tc)
            _check_route_ran(profile(), r, what)
            assert_parity(got, (p, U, fc), what=what)
            gp, gU, _ = got
            np.testing.assert_array_equal(gU[0] + gU[1], float(n_l * (labels.size - n_l)), err_msg=f"{what}: U_L + U_R")
            np.testing.assert_array_equal(gp[0], gp[1], err_msg=f"{what}: p")
            np.testing.assert_array_equal(score, _score_want(labels2, None, U, ties, labels.size, tc), err_msg=f"{what}: score")
    dispatch.clear_caches()


def _single_group_case(fmt):
    """3 000 cells of one group: narrow, wide and continuous genes, an all-zero and a constant gene."""
    rng = np.random.RandomState(17)
    n = 3000
    X = np.zeros((n, 16), np.float32)
    X[:, 0:4] = rng.randint(0, 9, (n, 4)) * (rng.rand(n, 4) < 0.5)
    X[:, 4:8] = rng.poisson(20.0, (n, 4))
    X[:, 8:12] = rng.lognormal(0, 1, (n, 4)) * (rng.rand(n, 4) < 0.6)
    X[:, 13] = 2.0
    X[:, 14] = rng.randint(0, 3, n)
    X[:, 15] = rng.randint(0, 1000, n)
    assert not X[:, 12].any()
    return C.to_format(X, fmt), np.array(["only"] * n)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_single_group_one_versus_rest(cuda_lib, fmt):
    """One label in the whole matrix: sigma = 0, so p is NaN where the oracle's is (1 where every cell is tied), the
    score NaN or 0 as epilogue.cuh states it, and every p_adj NaN (statsmodels' Benjamini-Hochberg)."""
    from illico_b200 import asymptotic_wilcoxon

    Xf, labels = _single_group_case(fmt)
    for alt, cc, tc in OPTIONS:
        what = f"{fmt}: one group: {alt}:cc={cc}:tc={tc}"
        kw = dict(alternative=alt, use_continuity=cc, tie_correct=tc)
        groups, p, U, fc, ties = oracle.run(Xf, labels, None, want_ties=True, **kw)
        _, _, out, extra = asymptotic_wilcoxon(FakeAnnData(Xf, labels), group_keys="pert", is_log1p=False, score=True,
                                               p_adjust=True, return_array=True, **kw)
        gp = out[:, :, 0]
        # (one-sided with continuity: z = +-0.5 / 0 = +-inf, a finite p)
        assert np.isnan(p).any() == (alt == "two-sided" or not cc), f"{what}: NaN p-values {np.isnan(p).sum()}"
        np.testing.assert_array_equal(np.isnan(gp), np.isnan(p), err_msg=f"{what}: NaN pattern of p")
        assert_parity((gp, out[:, :, 1], out[:, :, 2]), (p, U, fc), what=what)
        np.testing.assert_array_equal(extra["score"], _score_want(labels, None, U, ties, labels.size, tc), err_msg=f"{what}: score")
        if tc:
            assert np.array_equal(gp[0, [12, 13]], [1.0, 1.0]) and not extra["score"][0, [12, 13]].any(), what
        assert np.isnan(extra["p_adj"]).all() == np.isnan(p).any(), f"{what}: p_adj"
        np.testing.assert_array_equal(extra["p_adj"], bh_reference(gp), err_msg=f"{what}: p_adj")


# ---------------------------------------------------------------------------------------------------------------
# Benjamini-Hochberg at the edges of its sort and reverse running minimum (512 threads; thread t owns the ranks
# [N - (t + 1) per, N - t per) of the ascending order, per = ceil(N / 512))

def _bh_planes(N, G, seed):
    """[G, N] p-values: uniform; two-decimal ties with runs of exact 1.0 and 0.0 across thread chunks and the first warp
    boundary; subnormal and tiny values among 1.0s; all 1.0."""
    rng = np.random.RandomState(seed)
    per = -(-N // 512)
    p = np.empty((G, N))
    for g in range(G):
        kind = g % 4
        if kind == 0:
            row = rng.rand(N)
        elif kind == 1:
            row = np.round(rng.rand(N), 2)
            ones, zeros = min(N // 3, 32 * per + per // 2 + 1), min(N // 4, 3 * per + 1)
            pick = rng.permutation(N)
            row[pick[:ones]] = 1.0
            row[pick[ones:ones + zeros]] = 0.0
        elif kind == 2:
            row = 10.0 ** -rng.uniform(290, 324.5, N)
            row[rng.rand(N) < 0.3] = 1.0
        else:
            row = np.ones(N)
        p[g] = row
    return p


def _bh_device(p, gene_stride):
    """illico_bh_adjust on p placed every `gene_stride` doubles (the other slots hold -7, which would rank as 0)."""
    import torch

    from illico_b200 import _lib

    G, N = p.shape
    buf = np.full((G, N, gene_stride), -7.0)
    buf[:, :, 0] = p
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    src = torch.from_numpy(buf).to(dev)
    padj = torch.full((G, N), -1.0, dtype=torch.float64, device=dev)
    ws = torch.empty(int(lib.illico_bh_workspace_bytes(G, N)), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.illico_bh_adjust(src.data_ptr(), N * gene_stride, gene_stride, G, N, padj.data_ptr(), ws.data_ptr(),
                                    ws.numel(), st), "illico_bh_adjust")
    return padj.cpu().numpy()


BH_CASES = {f"N{N}": (N, 4) for N in (1, 2, 511, 512, 513, 36601)}
BH_CASES.update({"G1": (1000, 1), "G300": (200, 300)})


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(BH_CASES))
def test_bh_adjust_bit_for_bit(cuda_lib, case):
    N, G = BH_CASES[case]
    p = _bh_planes(N, G, seed=N + G)
    if case == "N36601":
        assert (p[2][p[2] > 0] < DBL_MIN).any() and (p[2] == 0).any()
    want = bh_reference(p)
    for stride in (1, 3):
        np.testing.assert_array_equal(_bh_device(p, stride), want, err_msg=f"{case}: gene_stride {stride}")


@pytest.mark.gpu
@pytest.mark.parametrize("N", [513, 36601])
def test_bh_adjust_group_with_nan(cuda_lib, N):
    """A NaN p-value (one-versus-rest with a single group) makes every p_adj of its group NaN, as in statsmodels; the
    other groups are untouched."""
    p = _bh_planes(N, 8, seed=5)
    p[1, N // 2] = np.nan
    p[4, -1] = np.nan
    p[6, :] = np.nan
    with np.errstate(invalid="ignore"):
        want = bh_reference(p)
    assert np.isnan(want[[1, 4, 6]]).all() and not np.isnan(want[[0, 2, 3, 5, 7]]).any()
    for stride in (1, 3):
        np.testing.assert_array_equal(_bh_device(p, stride), want, err_msg=f"gene_stride {stride}")
