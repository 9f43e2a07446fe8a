"""Segment-length kernel (k4_seglen) at its edges, against oracle/seglen_oracle.py: every sort width (4, 8 and 16 elements
per thread), exact ties of the sort keys (and ties with the padding of the network), max_nb_states edges, the
shared-memory boundary, persistent CTAs that process many chunks (state reset, lattice reuse, the > 600 rescale) and the
bit reproducibility of the histogram.

CPU tests check the fixtures themselves (their ties change the result) and that the GPU cases cover every path of the
kernel's sizing.  GPU tests go through Engine.seglen_hist (per-chunk histograms; LP and histories of one chunk) and the
public histograms.P_segment_len / len_hist.

Comparison (one helper, `check_chunk`): rows are matched by state history per track (a multiset: the leave children of
isBL repeat a history); histories must agree per track except on a track where the oracle finds a non-zero near-tie
(relative gap < 1e-12 between adjacent sort keys, where a last-bit difference of the library log may reorder two keys),
and such tracks must stay rare; exact ties never excuse a difference.  LP 1e-9 relative per matched row; histogram 1e-9
absolute, 1e-6 for a chunk with a flagged track."""
import warnings

import numpy as np
import pytest

from helpers import random_walk_tracks
from oracle import extrack_oracle as orc
from oracle import seglen_oracle as so

SEG_THREADS = 256        # XT_SEG_THREADS
SMEM_MARGIN = 256        # the engine's margin for static shared memory (subtracted from the opt-in limit)
B200_OPTIN = 232448      # opt-in shared memory per block of a B200 (227 KB)
B200_SM = 148
NEAR_TIE = 1e-12


# ------------------------------------------------------------------------------------------------------------------
# sizing: a mirror of xt_seglen_host.inl / xt_seg_smem / xt_k4.cu
def live_counts(nS, L, mx):
    """[(children nC, pruned)] of steps 2 .. L-1 of a track of L localisations."""
    out, nB = [], nS * nS
    for step in range(2, L):
        nC = nB * nS
        prune = step < L - 1 and nC > mx
        out.append((nC, prune))
        nB = mx if prune else nC
    return out


def sizing(nS, d, KS, mx, Ls, n_chunks=1, n_sm=B200_SM, optin=B200_OPTIN - SMEM_MARGIN):
    Ls = list(Ls)
    steps = [s for L in Ls for s in live_counts(nS, L, mx)]
    cap = max([nS * nS] + [nC for nC, _ in steps])
    n2 = 4
    while n2 < cap:
        n2 <<= 1
    Lmax = max(Ls)
    smem = 2 * cap * (d + KS + 2) * 8 + n2 * 12 + 2 * cap + 16 + 2 * Lmax * nS * 8 + 64
    ept = 4 if n2 <= 4 * SEG_THREADS else 8 if n2 <= 8 * SEG_THREADS else 16 if n2 <= 16 * SEG_THREADS else None
    fits = ept is not None and cap <= 65535 and smem <= optin
    per_sm = max(1, (228 * 1024) // (smem + 2048))
    pruned = [nC for nC, p in steps if p]
    return dict(cap=cap, n2=n2, ept=ept, smem=smem, fits=fits, grid=min(n_chunks, n_sm * per_sm), per_sm=per_sm,
                pruned=pruned, smem_stage=bool(pruned) and ept is not None and n2 >= 64 * ept,
                padding=any(nC < n2 for nC in pruned))


def largest_fitting(nS, d, KS, L, optin):
    mx = 1
    while sizing(nS, d, KS, mx + 1, [L], optin=optin)["fits"]:
        mx += 1
    return mx


# ------------------------------------------------------------------------------------------------------------------
# models and tracks
def model(Ds, Fs, Tr, le=(0.02,), pBL=0.07):
    Ds = np.asarray(Ds, float)
    return orc.Model(np.asarray(le, float), np.sqrt(2 * Ds * 0.02), np.asarray(Fs, float), np.asarray(Tr, float), pBL, [1.0], 1,
                     6, 3, 0.2, 120)


def std_model(nS, le=(0.02,)):
    """Tie-free by construction (distinct D, F and rates)."""
    Ds = np.array([1e-5, 0.04, 0.25, 0.6])[:nS]
    Fs = np.array([0.45, 0.3, 0.15, 0.1])[:nS]
    Tr = np.array([[0, 0.06, 0.03, 0.01], [0.05, 0, 0.04, 0.02], [0.01, 0.07, 0, 0.03], [0.02, 0.03, 0.08, 0]])[:nS, :nS]
    return model(Ds, Fs / Fs.sum(), Tr + np.diag(1 - Tr.sum(1)), le)


# Exact ties.  States 1 and 2 of MIRROR3 (2 and 3 of MIRROR4) have equal D and F and mirrored rates, so a sequence and its
# mirror image get bitwise-equal keys (the same operations on the same values, on the GPU as in numpy).  The rate between
# the mirrored states is zero: otherwise sequences that switch between them at different steps add the same terms in
# another order and differ in the last bit (near-ties) instead of tying.  P01ZERO: log 0 = -inf keys, and -inf sequences
# meet the -inf padding of the network when nC is not a power of two.
MIRROR3 = dict(Ds=[1e-5, 0.1, 0.1], Fs=[0.4, 0.3, 0.3], Tr=[[0.9, 0.05, 0.05], [0.08, 0.92, 0.0], [0.08, 0.0, 0.92]])
MIRROR4 = dict(Ds=[1e-5, 0.04, 0.25, 0.25], Fs=[0.4, 0.3, 0.15, 0.15],
               Tr=[[0.86, 0.06, 0.04, 0.04], [0.03, 0.91, 0.03, 0.03], [0.02, 0.05, 0.93, 0.0], [0.02, 0.05, 0.0, 0.93]])
P01ZERO = dict(Ds=[1e-5, 0.25], Fs=[0.6, 0.4], Tr=[[1.0, 0.0], [0.1, 0.9]])
TIE_MODELS = dict(mirror3=MIRROR3, mirror4=MIRROR4, p01zero=P01ZERO)

# name, model, max_nb_states, L, d, isBL, nT, ties at the cut (the surviving-history set depends on the tie rule)
TIE_CASES = [
    ("mirror3_ept4", "mirror3", 30, 10, 2, 1, 16, True),
    ("mirror3_ept8", "mirror3", 400, 12, 2, 1, 16, True),
    ("mirror3_ept16", "mirror3", 700, 12, 1, 0, 12, True),
    ("mirror4_ept4", "mirror4", 100, 8, 2, 1, 24, True),
    ("mirror4_ept8", "mirror4", 300, 8, 2, 0, 12, True),
    ("mirror4_ept16", "mirror4", 520, 8, 1, 1, 12, True),
    ("p01zero_ept4", "p01zero", 5, 12, 2, 1, 30, False),    # ties only in the ranks the LL slice reads
    ("p01zero_ept8", "p01zero", 600, 14, 2, 1, 16, True),
    ("p01zero_ept16", "p01zero", 1100, 14, 1, 0, 12, True),
]


def tie_input(case):
    name, mname, mx, L, d, isBL, nT, _ = case
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)   # log 0 of P01ZERO
        m = model(**TIE_MODELS[mname])
    C = random_walk_tracks(nT, L, d, np.random.default_rng(7), Ds=m.ds**2 / 0.04)
    return m, C, isBL, mx


# name, nS, d, LocErr, max_nb_states, L, isBL, nT: sort widths n2 = 8 ... 4096
WIDTH_CASES = [
    ("n2_8", 2, 1, (0.03,), 4, 10, 1, 20),
    ("n2_32", 3, 3, (0.02, 0.03, 0.04), 10, 9, 0, 20),
    ("n2_128", 4, 2, (0.02,), 30, 7, 1, 20),
    ("n2_256", 2, 3, (0.02,), 100, 12, 0, 20),
    ("n2_1024", 3, 2, (0.02, 0.03), 300, 10, 1, 16),
    ("n2_2048", 2, 1, (0.02,), 1000, 13, 0, 12),
    ("n2_4096_s2", 2, 2, (0.02,), 1100, 14, 1, 10),
    ("n2_4096_s3", 3, 1, (0.02,), 700, 10, 0, 10),
    ("n2_4096_s4", 4, 1, (0.02,), 520, 8, 1, 8),
]

# name, nS, d, max_nb_states, L, isBL
MX_CASES = [
    ("mx1_s2", 2, 2, 1, 10, 1),
    ("mx1_s3", 3, 2, 1, 8, 0),
    ("mx2_s2", 2, 1, 2, 9, 0),
    ("mx_nS-1_s3", 3, 2, 2, 8, 1),
    ("mx_nS-1_s4", 4, 1, 3, 7, 0),
    ("mx_odd7_s2", 2, 2, 7, 12, 1),
    ("mx_odd33_s3", 3, 3, 33, 9, 1),
    ("mx_eq_8_s2", 2, 2, 8, 11, 0),       # nS^3: step 2 has exactly max_nb_states children, not cut
    ("mx_eq_27_s3", 3, 1, 27, 8, 1),
    ("mx_eq_16_s4", 4, 2, 16, 6, 0),
    ("L3_s2", 2, 2, 1, 3, 1),             # only step 2, which is the last: never cut
    ("L3_s4", 4, 2, 5, 3, 0),
    ("last_step_s2", 2, 2, 2, 4, 1),      # step 2 cut, step 3 = L-1 keeps all nS * 2 children
]


# ------------------------------------------------------------------------------------------------------------------
# comparison
def check_chunk(got_LP, got_Bs, got_hist, want, label=""):
    """GPU (LP [nT, nBf], histories [nT, nBf, L], hist [L-1, nS]) against the oracle's (LP, hist, H, gaps).
    Returns the number of flagged tracks (near-ties) of the chunk."""
    LP0, h0, H0, gaps = want
    nT = LP0.shape[0]
    assert got_LP.shape == LP0.shape and got_Bs.shape == H0.shape, label
    flagged = gaps < NEAR_TIE
    for t in range(nT):
        Hg, Ho = got_Bs[t].astype(np.int64), H0[t].astype(np.int64)
        og, oo = np.lexsort(Hg.T[::-1]), np.lexsort(Ho.T[::-1])
        same = np.array_equal(Hg[og], Ho[oo])
        if flagged[t] and not same:
            continue
        assert same, f"{label}: histories of track {t} differ"
        np.testing.assert_allclose(got_LP[t][og], LP0[t][oo], rtol=1e-9, err_msg=f"{label}: LP of track {t}")
    np.testing.assert_allclose(got_hist, h0, rtol=0, atol=1e-6 if flagged.any() else 1e-9, err_msg=f"{label}: histogram")
    return int(flagged.sum())


def oracle_chunk(C, m, isBL, mx, min_l):
    with np.errstate(divide="ignore"):
        return so.segment_len_chunk(C, m, isBL, mx, min_l, want_histories=True, want_gaps=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU plumbing
def tables(m, min_l, mx, d):
    from extrack_b200 import histograms as xh

    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)   # log 0 of a zero rate
        p, leave, nS = xh._tables(m.loc_err, m.ds, m.Fs, m.TrMat, m.pBL, [1.0], 1, min_l, mx, d)
    return p, leave


class Upload:
    """One engine with the buckets `segs` (isBL per bucket) in chunks of `chunk_size` tracks."""

    def __init__(self, segs, bl, chunk_size, m, mx, min_l):
        from extrack_b200 import _native

        self.segs, self.bl, self.cs = segs, bl, chunk_size
        self.p, self.leave = tables(m, min_l, mx, segs[0].shape[2])
        self.nS = m.nS
        self.Lmax = max(s.shape[1] for s in segs)
        self.eng = _native.Engine(0)
        self.eng.upload(segs, bl, chunk_size)
        self.chunks = []   # (bucket, first track, nT) in chunk-id order (bucket by bucket)
        for b, s in enumerate(segs):
            for a in range(0, len(s), chunk_size):
                self.chunks.append((b, a, min(chunk_size, len(s) - a)))
        # the kernel's order: longest tracks first, stable
        self.corder = sorted(range(len(self.chunks)), key=lambda c: -segs[self.chunks[c][0]].shape[1])

    def tracks(self, c):
        b, a, n = self.chunks[c]
        return self.segs[b][a:a + n], self.bl[b]

    def hist(self):
        return self.eng.seglen_hist(self.p, self.leave, self.Lmax, self.nS, len(self.chunks))

    def dbg(self, c):
        C, _ = self.tracks(c)
        return self.eng.seglen_hist(self.p, self.leave, self.Lmax, self.nS, len(self.chunks), dbg_chunk=c, dbg_shape=C.shape[:2])

    def close(self):
        self.eng.close()


def run_one_chunk(C, m, isBL, mx, min_l=3):
    """A single chunk on the GPU -> (LP, Bs, hist [L-1, nS])."""
    up = Upload([C], [isBL], len(C), m, mx, min_l)
    try:
        hist, LP, Bs = up.dbg(0)
    finally:
        up.close()
    L = C.shape[1]
    assert not hist[0, L - 1:].any()
    return LP, Bs, hist[0, :L - 1]


def device_limits():
    import torch

    pr = torch.cuda.get_device_properties(0)
    return pr.shared_memory_per_block_optin - SMEM_MARGIN, pr.multi_processor_count


# ==================================================================================================================
# CPU: the fixtures and the coverage of the GPU cases
@pytest.mark.parametrize("case", TIE_CASES, ids=[c[0] for c in TIE_CASES])
def test_tie_fixture_changes_with_the_tie_rule(case):
    """Reversing only the tie order (equal keys by ascending index) moves the oracle's histogram by > 1e-3; where the
    ties sit at the cut it also changes the surviving histories of at least one track in four.  Exact ties, not
    near-ties: no track has a non-zero gap below 1e-12."""
    m, C, isBL, mx = tie_input(case)
    with np.errstate(divide="ignore"):
        LP, h, H, gaps = so.segment_len_chunk(C, m, isBL, mx, 3, want_histories=True, want_gaps=True)
        LPr, hr, Hr = so.segment_len_chunk(C, m, isBL, mx, 3, want_histories=True, ties_ascending=True)
    assert np.abs(h - hr).max() > 1e-3
    assert not (gaps < NEAR_TIE).any()
    changed = sum(set(map(bytes, H[t].astype(np.int8))) != set(map(bytes, Hr[t].astype(np.int8))) for t in range(len(C)))
    if case[7]:
        assert 4 * changed >= len(C), changed
    else:
        assert changed == 0
    # what the GPU case exercises: the sort width it names, and real -inf keys next to the padding for P01ZERO
    sz = sizing(m.nS, C.shape[2], 1, mx, [C.shape[1]])
    assert sz["fits"] and "ept%d" % sz["ept"] in case[0]
    if case[1] == "p01zero":
        assert sz["padding"] and np.isneginf(LP).any()


def test_oracle_defaults_unchanged_by_the_test_options():
    """The test-only options do not change the default results (the golden tests pin the defaults themselves)."""
    m, C, isBL, mx = tie_input(TIE_CASES[0])
    with np.errstate(divide="ignore"):
        a = so.segment_len_chunk(C, m, isBL, mx, 3, want_histories=True)
        b = so.segment_len_chunk(C, m, isBL, mx, 3, want_histories=True, want_gaps=True)
        _, _, g = so.segment_len_chunk(C[:, :4], m, isBL, 10**6, 3, want_gaps=True)   # no pruning, no gaps
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert len(b) == 4 and b[3].shape == (len(C),)
    assert np.isinf(g).all()


def test_gpu_cases_cover_every_sort_path():
    """The GPU parametrization reaches 4, 8 and 16 elements per thread, sort widths 8 ... 4096, sorts with and without
    shared-memory stages, and pruning steps with padding (nC < n2)."""
    szs = [sizing(nS, d, len(le), mx, [L]) for _, nS, d, le, mx, L, _, _ in WIDTH_CASES]
    szs += [sizing(nS, d, 1, mx, [L]) for _, nS, d, mx, L, _ in MX_CASES]
    szs += [sizing(len(TIE_MODELS[c[1]]["Ds"]), c[4], 1, c[2], [c[3]]) for c in TIE_CASES]
    assert all(s["fits"] for s in szs)
    assert {s["ept"] for s in szs if s["pruned"]} == {4, 8, 16}
    assert {8, 32, 128, 256, 1024, 2048, 4096} <= {s["n2"] for s in szs if s["pruned"]}
    assert any(s["smem_stage"] for s in szs) and any(s["pruned"] and not s["smem_stage"] for s in szs)
    assert any(s["padding"] for s in szs) and any(s["pruned"] and not s["padding"] for s in szs)
    # the named widths are the ones reached
    for (name, nS, d, le, mx, L, _, _), s in zip(WIDTH_CASES, szs):
        assert name.split("_")[1] == str(s["n2"]) and s["pruned"], name


def test_sizing_edges():
    """max_nb_states edges as the host sizes them: nS^k is not cut (nC > max_nb_states strictly), the last step never."""
    assert live_counts(2, 11, 8)[:2] == [(8, False), (16, True)]
    assert live_counts(3, 3, 1) == [(27, False)]
    assert live_counts(2, 4, 2) == [(8, True), (4, False)]
    s = sizing(2, 2, 1, 1100, [14])
    assert (s["cap"], s["n2"], s["ept"]) == (2200, 4096, 16) and s["fits"] and s["per_sm"] == 1
    # the boundaries on a B200 with the fixed-point bins (12 localisations): first max_nb_states that does not fit
    assert largest_fitting(2, 2, 1, 12, B200_OPTIN - SMEM_MARGIN) == 1113
    assert largest_fitting(3, 1, 1, 12, B200_OPTIN - SMEM_MARGIN) == 921


# ==================================================================================================================
# GPU
@pytest.fixture(scope="module")
def gpu():
    """(opt-in shared memory per block less the engine's margin, SM count) of device 0."""
    return device_limits()


@pytest.mark.gpu
@pytest.mark.parametrize("case", WIDTH_CASES, ids=[c[0] for c in WIDTH_CASES])
def test_gpu_sort_widths(gpu, case):
    name, nS, d, le, mx, L, isBL, nT = case
    m = std_model(nS, le)
    C = random_walk_tracks(nT, L, d, np.random.default_rng(11), Ds=m.ds**2 / 0.04, loc_err=le[0])
    LP, Bs, hist = run_one_chunk(C, m, isBL, mx)
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, isBL, mx, 3), name) <= 0.05 * nT


@pytest.mark.gpu
@pytest.mark.parametrize("case", TIE_CASES, ids=[c[0] for c in TIE_CASES])
def test_gpu_exact_ties(gpu, case):
    m, C, isBL, mx = tie_input(case)
    LP, Bs, hist = run_one_chunk(C, m, isBL, mx)
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, isBL, mx, 3), case[0]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", MX_CASES, ids=[c[0] for c in MX_CASES])
def test_gpu_max_nb_states_edges(gpu, case):
    name, nS, d, mx, L, isBL = case
    m = std_model(nS)
    C = random_walk_tracks(12, L, d, np.random.default_rng(13), Ds=m.ds**2 / 0.04)
    LP, Bs, hist = run_one_chunk(C, m, isBL, mx)
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, isBL, mx, 3), name) <= 0.05 * len(C)


@pytest.mark.gpu
@pytest.mark.parametrize("nS,d", [(2, 2), (3, 1)])
def test_gpu_shared_memory_boundary(gpu, nS, d):
    """The largest max_nb_states that fits the device runs and matches the oracle; one more raises ValueError, never a
    CUDA error."""
    from extrack_b200 import histograms as xh

    optin, _ = gpu
    L = 14
    mx = largest_fitting(nS, d, 1, L, optin)
    s = sizing(nS, d, 1, mx, [L], optin=optin)
    assert s["fits"] and s["cap"] == nS * mx and not sizing(nS, d, 1, mx + 1, [L], optin=optin)["fits"]
    m = std_model(nS)
    C = random_walk_tracks(4, L, d, np.random.default_rng(17), Ds=m.ds**2 / 0.04)
    LP, Bs, hist = xh.P_segment_len(C, m.loc_err[None, None], m.ds, m.Fs, m.TrMat, min_l=3, pBL=m.pBL, isBL=1, cell_dims=[1.0],
                                    nb_substeps=1, max_nb_states=mx)
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, 1, mx, 3), "boundary") == 0
    with pytest.raises(ValueError, match="do not fit in shared memory"):
        xh.P_segment_len(C, m.loc_err[None, None], m.ds, m.Fs, m.TrMat, min_l=3, pBL=m.pBL, isBL=1, cell_dims=[1.0], nb_substeps=1,
                         max_nb_states=mx + 1)


# ---- reused CTAs: many small chunks, a rescaled bucket with more chunks than CTAs --------------------------------
REUSE_MX = 600            # 2 states, 3-D: 1200 live sequences, n2 = 2048 (EPT 8), one CTA per SM
REUSE_LOC = 0.002         # immobile tracks with a small LocErr: the final LP passes 600 within 50 localisations
REUSE_BUCKETS = [(8, 300, 1), (12, 300, 1), (50, 340, 0)]   # L, tracks, isBL (the longest bucket has no leave term)
REUSE_CHUNK = 2


def reuse_model():
    return std_model(2, (REUSE_LOC,))


def reuse_tracks(m):
    rng = np.random.default_rng(23)
    segs = []
    for L, n, _ in REUSE_BUCKETS:
        Ds = [1e-5] if L == 50 else m.ds**2 / 0.04
        segs.append(random_walk_tracks(n, L, 3, rng, Ds=Ds, loc_err=REUSE_LOC))
    return segs


@pytest.fixture(scope="module")
def reuse(gpu):
    _, n_sm = gpu
    m = reuse_model()
    segs = reuse_tracks(m)
    min_l = min(L for L, _, _ in REUSE_BUCKETS)
    up = Upload(segs, [b for _, _, b in REUSE_BUCKETS], REUSE_CHUNK, m, REUSE_MX, min_l)
    s = sizing(2, 3, 1, REUSE_MX, [L for L, _, _ in REUSE_BUCKETS], len(up.chunks), n_sm=n_sm)
    want = {}
    for c in range(len(up.chunks)):
        C, isBL = up.tracks(c)
        want[c] = oracle_chunk(C, m, isBL, REUSE_MX, min_l)
    yield up, s, want, m, min_l
    up.close()


@pytest.mark.gpu
def test_gpu_reused_ctas_every_chunk(reuse):
    up, s, want, m, min_l = reuse
    assert s["ept"] == 8 and s["per_sm"] == 1
    n = len(up.chunks)
    assert n >= 3 * s["grid"], (n, s["grid"])
    rescaled = [c for c in up.corder if np.isclose(want[c][0].max(), 600.0)]
    assert len(rescaled) > s["grid"] and len(rescaled) < n   # rescaled chunks on reused CTAs, and chunks that are not
    hist = up.hist()
    flagged = 0
    for c in range(n):
        C, _ = up.tracks(c)
        L = C.shape[1]
        assert not hist[c, L - 1:].any(), c
        h0 = want[c][1]
        flagged += int((want[c][3] < NEAR_TIE).any())
        np.testing.assert_allclose(hist[c, :L - 1], h0, rtol=0, atol=1e-6 if (want[c][3] < NEAR_TIE).any() else 1e-9,
                                   err_msg=f"chunk {c}")
    assert flagged <= 0.05 * n


@pytest.mark.gpu
def test_gpu_reused_ctas_dbg_rows(reuse):
    """LP and histories of the last chunk in longest-first order, and of a rescaled chunk past the first grid positions."""
    up, s, want, m, min_l = reuse
    rescaled_late = [c for i, c in enumerate(up.corder) if i >= s["grid"] and np.isclose(want[c][0].max(), 600.0)]
    assert rescaled_late
    for c in (up.corder[-1], rescaled_late[len(rescaled_late) // 2]):
        hist, LP, Bs = up.dbg(c)
        L = up.tracks(c)[0].shape[1]
        assert check_chunk(LP, Bs, hist[c, :L - 1], want[c], f"chunk {c}") == 0


@pytest.mark.gpu
def test_gpu_reused_ctas_len_hist(gpu):
    """len_hist over a multi-bucket dict of the same kind (chunks of 50 tracks) against the oracle's len_hist."""
    from extrack_b200 import histograms as xh
    from extrack_b200 import tracking as xt

    params = xt.generate_params(nb_states=2, LocErr_type=1, nb_dims=3, LocErr_bounds=[0.0005, 0.1], D_max=10,
                                Fractions_bounds=[0.001, 0.99], estimated_LocErr=[REUSE_LOC], estimated_Ds=[1e-5, 0.25],
                                estimated_Fs=[0.6, 0.4], estimated_transition_rates=0.1)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, 0.02, 2, 1)
    m = orc.Model(np.asarray(LocErr).reshape(-1), ds, Fs, TrMat, pBL, [1.0], 1, 6, 3, 0.2, REUSE_MX)
    segs = [a[:n] for a, n in zip(reuse_tracks(m), (120, 60, 110))]
    tracks = {str(a.shape[1]): a for a in segs}
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        got = xh.len_hist(tracks, params, 0.02, cell_dims=[1.0], nb_states=2, max_nb_states=REUSE_MX)
    want = so.len_hist(segs, m, REUSE_MX)
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)


# ---- invariants and determinism -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_identical_tracks_identical_rows(gpu):
    m = std_model(3, (0.02, 0.03))
    rng = np.random.default_rng(29)
    base = random_walk_tracks(3, 11, 2, rng, Ds=m.ds**2 / 0.04)
    C = np.concatenate([base, base[[1, 1, 0]], random_walk_tracks(2, 11, 2, rng, Ds=m.ds**2 / 0.04)])
    LP, Bs, hist = run_one_chunk(C, m, 1, 400)   # 1200 live sequences: EPT 8
    for a, b in ((1, 3), (1, 4), (0, 5)):
        assert LP[a].tobytes() == LP[b].tobytes() and np.array_equal(Bs[a], Bs[b]), (a, b)
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, 1, 400, 3), "identical") == 0


@pytest.mark.gpu
def test_gpu_bitwise_reproducible(reuse):
    """Two identical calls give the same bits (histogram, LP, histories), and a chunk uploaded alone has the bits it has
    inside the many-chunk upload."""
    up, s, want, m, min_l = reuse
    c = [c for c in up.corder if np.isclose(want[c][0].max(), 600.0)][-1]
    h1, LP1, B1 = up.dbg(c)
    h2, LP2, B2 = up.dbg(c)
    h3 = up.hist()
    assert h1.tobytes() == h2.tobytes() == h3.tobytes()
    assert LP1.tobytes() == LP2.tobytes() and B1.tobytes() == B2.tobytes()
    for cc in (c, up.corder[-1]):
        C, isBL = up.tracks(cc)
        alone = Upload([C], [isBL], REUSE_CHUNK, m, REUSE_MX, min_l)
        try:
            ha, LPa, Ba = alone.dbg(0)
        finally:
            alone.close()
        L = C.shape[1]
        assert ha[0, :L - 1].tobytes() == h3[cc, :L - 1].tobytes(), cc
        if cc == c:
            assert LPa.tobytes() == LP1.tobytes() and Ba.tobytes() == B1.tobytes()
