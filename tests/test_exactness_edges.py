"""Exact search where the scan's error bound is easiest to break (DESIGN.md §6).

Every answer rests on one premise: the scan's approximate cosine of every row is within the per-query bound eps_q of
the reference's fp64 cosine.  When it fails the proof can still pass and the answer is silently wrong, so these tests
feed the inputs where it can fail:
  * queries and rows far outside unit scale - the reference's fp64 result does not change under power-of-two
    scaling (checked on the CPU first), so the answer must not change either;
  * corpora whose scores rise inside every scan unit's tile range, so thresholds keep lagging, the candidate lists
    flood and the finalize kernel has to stream a query's keys from L2 instead of staging them in shared memory;
  * the small-batch CUDA graph replayed after in-place mutations that leave its key unchanged.
Nothing here reads the reference project.
"""
import numpy as np
import pytest

from oracle import pyref

WINDOW = (2.0 ** -60, 2.0 ** 100)    # row norms inside which the scan stays on its fast path (DESIGN.md §6)


@pytest.fixture(scope="module")
def rb(native):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import runbookai_b200
    return runbookai_b200


def _bits(x):
    from runbookai_b200 import synth
    return synth.f32_to_bf16_bits(np.asarray(x, dtype=np.float32))


def _vals(bits):
    from runbookai_b200 import synth
    return synth.bf16_bits_to_f32(bits).astype(np.float64)


def _scaled_bits(bits, s):
    """bf16 rows times 2^s, still bf16 (s keeps every element a normal bf16)."""
    v = np.ldexp(_vals(bits), s)
    out = _bits(v)
    assert (_vals(out) == v).all()
    return out


def _in_window(norms):
    return (norms >= WINDOW[0]) & (norms <= WINDOW[1])


def _same(a, b):
    """bit-identical float arrays"""
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


def _stats_delta(ix, before):
    st = ix.stats()
    return st, {k: st[k] - before[k] for k in ("fallback_queries", "retry_batches", "graph_replays")}


def _check(got, want, nq):
    slots, scores, counts = got
    es, ev, ec = want
    for b in range(nq):
        assert counts[b] == ec[b], (b, counts[b], ec[b])
        assert (slots[b, :ec[b]] == es[b, :ec[b]]).all(), (b, slots[b, :ec[b]], es[b, :ec[b]])
        assert _same(scores[b, :ec[b]], ev[b, :ec[b]]), (b, scores[b, :ec[b]], ev[b, :ec[b]])
        assert (slots[b, ec[b]:] == -1).all() and np.isnan(scores[b, ec[b]:]).all()


def _oracle_f64(oracle_mod, rows, queries, k_fetch, min_score, live=None):
    nq = queries.shape[0]
    es = np.full((nq, k_fetch), -1, dtype=np.int64)
    ev = np.full((nq, k_fetch), np.nan)
    ec = np.zeros(nq, dtype=np.int32)
    for b in range(nq):
        s, v = oracle_mod.search(rows, queries[b], k_fetch, min_score, live=live)
        es[b, :len(s)], ev[b, :len(s)], ec[b] = s, v, len(s)
    return es, ev, ec


# --------------------------------------------------------------------------- A: the premise of the tests (CPU)
def test_power_of_two_scaling_leaves_the_oracle_bit_identical(oracle_mod):
    """The reference's fp64 cosine is invariant, bit for bit, under power-of-two scaling of the query or the rows as
    long as fp64 itself neither overflows nor underflows: every product, partial sum, norm and square root is scaled
    exactly.  So 'equal to the oracle on the unscaled inputs' is what the GPU tests below may demand."""
    rng = np.random.default_rng(5)
    n, d = 400, 48
    rows = rng.standard_normal((n, d))
    q = rng.standard_normal((3, d))
    for i in range(3):                                       # hits above 0.5 for the thresholded search
        rows[rng.choice(n, 6, replace=False)] = q[i] + rng.uniform(0.2, 1.0, (6, 1)) * rng.standard_normal((6, d))
    scales = (-300, -100, -60, 0, 60, 100, 300)
    base = {(b, ms): oracle_mod.search(rows, q[b], 25, ms) for b in range(3) for ms in (None, 0.5)}
    base_scores = [oracle_mod.scores(rows, q[b]) for b in range(3)]
    assert all(len(base[(b, 0.5)][0]) >= 6 for b in range(3))
    for s_c in scales:
        rs = np.ldexp(rows, s_c)
        for s_q in scales:
            for b in range(3):
                qs = np.ldexp(q[b], s_q)
                assert _same(oracle_mod.scores(rs, qs), base_scores[b]), (s_c, s_q, b)
                for ms in (None, 0.5):
                    s, v = oracle_mod.search(rs, qs, 25, ms)
                    assert (s == base[(b, ms)][0]).all() and _same(v, base[(b, ms)][1]), (s_c, s_q, b, ms)
    # the same statement from the independent pure-Python restatement
    a, c = q[0][:16], rows[:5, :16]
    for s_c in scales:
        for s_q in scales:
            for r in c:
                want = pyref.cosine_similarity(a.tolist(), r.tolist())
                got = pyref.cosine_similarity(np.ldexp(a, s_q).tolist(), np.ldexp(r, s_c).tolist())
                assert _same(got, want) and _same(want, oracle_mod.cosine(a, r)), (s_c, s_q)


# --------------------------------------------------------------------------- B: scale sweep against the oracle
@pytest.mark.gpu
def test_default_index_scale_sweep_matches_the_oracle(rb, oracle_mod):
    """bf16-exact rows at 2^s_c, float64 queries at 2^s_q: ids and fp64 scores bit-identical to the oracle on the
    same scaled values.  B = 5 runs the 1-CTA kernel through the captured graph, B = 200 the CTA-pair kernel.  Rows
    inside the norm window never need the wide rescan or the exhaustive kernel, whatever the query's scale."""
    from runbookai_b200 import synth
    n, d, B = 4000, 128, 200
    base = synth.random_corpus(n, d, 61)
    q32 = synth.random_queries(B, d, 62)
    synth.plant_neighbours(base, q32, 8, 63)
    for s_c in (-100, -60, 0, 60, 100):
        bits = _scaled_bits(base, s_c)
        fast = bool(_in_window(np.linalg.norm(_vals(bits), axis=1)).all())
        assert fast == (abs(s_c) <= 60)
        with rb.Index(d) as ix:
            ix.append_bf16(bits)
            for s_q in (-300, -160, -80, 0, 70, 300):
                qs = np.ldexp(q32.astype(np.float64), s_q)
                for ms in (None, 0.5):
                    for k in (10, 112):
                        want = oracle_mod.search_batch_mt(bits, qs, k, ms)
                        if ms is not None:
                            assert want[2].min() >= 1, "planted rows must pass the threshold"
                        for nb in (5, B):
                            before = ix.stats()
                            s, v, c, _ = ix.search(qs[:nb], k, ms)
                            _check((s, v, c), want, nb)
                            _, dl = _stats_delta(ix, before)
                            if fast:
                                assert dl["fallback_queries"] == 0 and dl["retry_batches"] == 0, (s_c, s_q, ms, k, nb, dl)


@pytest.mark.gpu
def test_keep_f64_index_scale_sweep_matches_the_oracle(rb, oracle_mod):
    """RBK_INDEX_KEEP_F64 with arbitrary float64 rows at 2^-300 .. 2^300 (and one corpus whose rows span that range
    individually): bit-identical to the oracle on the float64 rows, for queries far from unit scale too."""
    rng = np.random.default_rng(71)
    n, d, B = 3000, 96, 200
    base = rng.standard_normal((n, d))
    q = rng.standard_normal((B, d))
    for i in range(B):                                       # 4 near-duplicates per query, cosines 0.55 .. 0.95
        slots = rng.choice(n, 4, replace=False)
        base[slots] = q[i] + rng.uniform(0.3, 1.5, (4, 1)) * rng.standard_normal((4, d))
    mixed = rng.choice([-300, -80, 0, 80, 300], n)
    corpora = [(s, np.ldexp(base, s)) for s in (-300, -80, 0, 80, 300)] + [("mixed", np.ldexp(base, mixed[:, None]))]
    for name, rows in corpora:
        with np.errstate(over="ignore"):
            norms = np.linalg.norm(_vals(_bits(rows)), axis=1)
        fast = bool(_in_window(norms).all())
        assert fast == (name in (0, 80))
        with rb.Index(d, keep_f64=True) as ix:
            ix.append_f64(rows)
            for s_q in (-300, -80, 0, 70, 300):
                qs = np.ldexp(q, s_q)
                for ms in (None, 0.5):
                    for k in (10, 24):
                        want = _oracle_f64(oracle_mod, rows, qs, k, ms)
                        for nb in (5, B):
                            before = ix.stats()
                            s, v, c, _ = ix.search(qs[:nb], k, ms)
                            _check((s, v, c), want, nb)
                            _, dl = _stats_delta(ix, before)
                            if fast:
                                assert dl["fallback_queries"] == 0 and dl["retry_batches"] == 0, (name, s_q, ms, k, nb, dl)


# --------------------------------------------------------------------------- C: the premise itself
@pytest.mark.gpu
@pytest.mark.parametrize("d,B", [(100, 3), (100, 130), (768, 3), (768, 130)])
def test_scan_scores_within_error_bound_at_extreme_scales(rb, d, B):
    """The scan's approximate cosine stays within (d+8)*2^-22 of the fp64 cosine for every row whose norm is inside
    the window, at query and row scales far from 1 (f32 queries: scales stay inside f32)."""
    from runbookai_b200 import synth
    n = 1200
    rng = np.random.default_rng(81 + d + B)
    base = synth.random_corpus(n, d, 82)
    q = synth.random_queries(B, d, 83)
    spread = rng.integers(-45, 46, n)                        # per-row exponents around the corpus scale
    eps = (d + 8) * 2.0 ** -22
    for s_q, s_c in ((-70, -70), (-100, -40), (60, 60), (100, 20), (0, 100), (0, -100)):
        t = np.clip(s_c + spread, -110, 110)
        bits = _bits(np.ldexp(_vals(base), t[:, None]))
        bits[17] = 0                                         # zero row -> NaN
        qs = np.ldexp(q.astype(np.float64), s_q).astype(np.float32)
        with rb.Index(d) as ix:
            ix.append_bf16(bits)
            got = ix.debug_scores(qs)
        cf = _vals(bits)
        qf = qs.astype(np.float64)
        norms = np.linalg.norm(cf, axis=1)
        with np.errstate(invalid="ignore", divide="ignore"):
            ref = (qf @ cf.T) / (np.linalg.norm(qf, axis=1)[:, None] * norms[None, :])
        assert np.isnan(got[:, 17]).all()
        checked = _in_window(norms)
        assert checked.sum() >= 50, (s_q, s_c, checked.sum())
        err = np.abs(got[:, checked] - ref[:, checked])
        assert not np.isnan(err).any() and err.max() <= eps, (s_q, s_c, np.nanmax(err), eps)


# --------------------------------------------------------------------------- D: flooded candidate lists
_FLOOD_CACHE = {}


def _flood_corpus(n_tiles, R, d=64, seed=91):
    """Rows whose cosine with u rises from 0.1 to 0.8 inside every scan unit's tile range (unit r reads tiles
    [n_tiles*r//R, n_tiles*(r+1)//R)), so every tile beats the thresholds of the tiles before it and the candidate
    lists keep filling.  144 rows well above that band (cosines 0.86 + 0.0008 j, all along one direction w0, so their
    order cannot be shuffled by the queries' noise) sit in unit 0's last tile: the proofs pass and the finalize
    kernel's own answer is what gets checked."""
    key = (n_tiles, R, d, seed)
    if key in _FLOOD_CACHE:
        return _FLOOD_CACHE[key]
    rng = np.random.default_rng(seed)
    u = rng.standard_normal(d)
    u /= np.linalg.norm(u)
    n = n_tiles * 256
    c = np.empty(n)
    for r in range(R):
        a, b = n_tiles * r // R * 256, n_tiles * (r + 1) // R * 256
        c[a:b] = np.linspace(0.1, 0.8, b - a)
    w = rng.standard_normal((n, d)).astype(np.float32)
    w -= (w @ u.astype(np.float32))[:, None] * u.astype(np.float32)[None, :]
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    top0 = (n_tiles // R - 1) * 256                          # first row of unit 0's last tile
    w[top0:top0 + 144] = w[top0]
    c[top0:top0 + 144] = 0.86 + 0.0008 * np.arange(144)
    rows = c[:, None].astype(np.float32) * u.astype(np.float32) + np.sqrt(1 - c * c)[:, None].astype(np.float32) * w
    out = (_bits(rows), u)
    _FLOOD_CACHE[key] = out
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 128, 300, 1024])
def test_flooded_candidate_lists_stream_keys_through_finalize(rb, oracle_mod, B):
    """Rising scores flood every unit's lists, so a query's candidates outnumber the keys the finalize kernel can
    stage in shared memory (16384 keys up to 160 queries, 8192 up to 320, 2048 beyond) and it reads them from the
    lists in L2 on every radix pass and in the selection.  Results stay bit-identical to the oracle, on the fast
    path.  B = 1 and 128: 1-CTA kernel (graph path); 300 and 1024: CTA-pair kernel."""
    d = 64
    with rb.Index(d) as probe:
        sm_count = probe.stats()["sm_count"]
    pairs = B > 128
    units = sm_count // 2 if pairs else sm_count
    QB = -(-B // (256 if pairs else 128))
    R = max(1, units // QB)
    n_tiles = 8 * R                                          # a multiple of R, 8 tiles per unit
    bits, u = _flood_corpus(n_tiles, R, d)
    assert max(1, min(units // QB, n_tiles)) == R
    rng = np.random.default_rng(92 + B)
    queries = _vals(_bits(u[None, :] + 0.01 * rng.standard_normal((B, d)))).astype(np.float32)
    nq = min(B, 64)
    with rb.Index(d) as ix:
        ix.append_bf16(bits)
        for k in (16, 112):
            for ms in (None, 0.5):
                before = ix.stats()
                s, v, c, _ = ix.search(queries, k, ms)
                want = oracle_mod.search_batch_verify(bits, queries[:nq].astype(np.float64), k, ms)
                _check((s, v, c), want, nq)
                assert (c == k).all()
                _, dl = _stats_delta(ix, before)
                assert dl["fallback_queries"] == 0 and dl["retry_batches"] == 0, (k, ms, dl)


# --------------------------------------------------------------------------- E: graph replay after mutations
def _bf16_angle_ratio(rows):
    return np.linalg.norm(rows - _vals(_bits(rows)), axis=1) / np.linalg.norm(rows, axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("keep_f64", [False, True])
def test_graph_replay_after_in_place_mutations(rb, oracle_mod, keep_f64):
    """Host searches with B <= 128 replay a captured graph that bakes in every pointer and scalar.  Mutations that
    keep its key (tombstone, bulk overwrite, clear + append of as many rows, a keep-f64 overwrite that grows the
    corpus-side error bound held on the device) must be seen by the replay."""
    from runbookai_b200 import synth
    rng = np.random.default_rng(101)
    n, d, B, k, ms = 3000, 96, 8, 20, 0.25
    q = synth.random_queries(B, d, 102)
    if keep_f64:
        rows = rng.standard_normal((n, d))
        for i in range(B):
            rows[rng.choice(n, 10, replace=False)] = q[i] + rng.uniform(0.3, 1.5, (10, 1)) * rng.standard_normal((10, d))
    else:
        bits = synth.random_corpus(n, d, 103)
        synth.plant_neighbours(bits, q, 10, 104)
        rows = _vals(bits)
    live = np.ones(n, dtype=np.uint8)
    with rb.Index(d, keep_f64=keep_f64) as ix:
        ix.append_f64(rows)
        replays = [ix.stats()["graph_replays"]]

        def search_and_check():
            s, v, c, _ = ix.search(q, k, ms)
            corpus = rows if keep_f64 else _bits(rows)
            _check((s, v, c), _oracle_f64(oracle_mod, corpus, q.astype(np.float64), k, ms, live=live), B)
            replays.append(ix.stats()["graph_replays"])
            return s, c

        s, c = search_and_check()                            # captures the graph
        # 1. tombstone the current top hit of query 0
        top = int(s[0, 0])
        ix.tombstone([top])
        live[top] = 0
        s, c = search_and_check()
        assert s[0, 0] != top
        # 2. a live slot becomes 3 * q[1]: the new top hit of query 1
        slot = int(np.flatnonzero(live)[7])
        rows[slot] = 3.0 * q[1]
        ix.overwrite_f64_batch([slot], rows[slot][None, :])
        s, c = search_and_check()
        assert s[1, 0] == slot
        if keep_f64:
            # 3. the k-th hit of query 2 moved to 0.49 bf16 ulps off its rounding in every element: a larger
            # rounding angle than any earlier row, so eps_c_max grows in place, right where the proof is decided
            kth = int(s[2, min(k, c[2]) - 1])
            x = rows[kth]
            xb = _vals(_bits(x))
            ulp = np.ldexp(1.0, np.frexp(xb)[1] - 8)
            y = xb + 0.49 * ulp * rng.choice([-1.0, 1.0], d)
            assert (_bits(y) == _bits(xb)).all()
            assert _bf16_angle_ratio(y[None, :])[0] > _bf16_angle_ratio(rows[live.astype(bool)]).max()
            rows[kth] = y
            ix.overwrite_f64_batch([kth], y[None, :])
            search_and_check()
        # 4. clear, then as many different rows: same pointers, same row count
        ix.clear()
        rows[:] = rng.standard_normal((n, d)) if keep_f64 else _vals(synth.random_corpus(n, d, 105))
        live[:] = 1
        ix.append_f64(rows)
        search_and_check()
    assert replays[1] >= 1 and all(b == a + 1 for a, b in zip(replays[1:], replays[2:])), replays
