"""Stage 3 on every model the extraction accepts: the gapped alphabet, several strand flags, k = 14, more than 8192
model classes, windows wider than the shared-memory tile.  Scores are compared with the CPU oracle (which recounts
every window with the extraction's counter), with extraction + LogPdf, and with themselves.  Needs a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GAP = dict(alphabet="gapped-nucleotide")


def make_model(K, O, seqs, M, N, n_feat, members=1, pairs=0, summary="", seed=0, max_ambiguous=None, **flags):
    """a model over classes observed in seqs: n_feat singles (+ pairs), random theta"""
    rng = np.random.default_rng(seed)
    binarize = flags.pop("binarize", False)
    ocfg = O.make_config(M, N, binarize=binarize, max_ambiguous=-1 if max_ambiguous is None else max_ambiguous, **flags)
    ref = O.extract(ocfg, seqs)
    k, code = ref.classes()
    pick = np.sort(rng.choice(ref.m, size=min(n_feat, ref.m), replace=False))
    ck, cc = k[pick], code[pick]
    feats = [(i, i) for i in range(len(pick))]
    for _ in range(pairs):
        a, b = sorted(rng.choice(len(pick), 2, replace=False))
        feats.append((int(a), int(b)))
    theta = rng.normal(scale=0.3, size=(members, len(feats) + 1))
    kmd = dict(counter=K.NewKmerCounter(M, N, binarize=binarize, max_ambiguous=max_ambiguous, **flags), class_k=ck,
               class_code=cc, features=feats, theta=theta, summary=summary)
    omd = dict(cfg=ocfg, class_k=ck, class_code=cc, features=feats, theta=theta, summary=summary)
    return kmd, omd


def regions(seed=3):
    from kmerlr_b200 import synth
    rng = np.random.default_rng(seed)
    lens = [1000, 200, 201, 150, 777, 4096, 0, 210, 5000]
    seqs = []
    for i, L in enumerate(lens):
        s = bytes(synth.random_bases(L, 3, offset=100000 * i)).decode()
        seqs.append(s)
    s = list(seqs[4])
    for p in rng.choice(777, 12, replace=False):
        s[p] = "N"
    seqs[4] = "".join(s).lower()
    return seqs


def check(K, O, kms, oms, seqs, W, step, tol=1e-12):
    out = K.genomicKmerLr(kms).predict_window_genomic(seqs, W, step)
    ref = O.score_windows(oms, seqs, W, step)
    flat = np.concatenate(out) if len(out) else np.zeros(0)
    assert len(flat) == len(ref)
    assert np.allclose(flat, ref, rtol=tol, atol=tol)
    # slots the strict loop bound never writes stay exactly 0.0 (kmerLr_predict_genomic.go:153-159)
    assert np.array_equal(flat == 0.0, ref == 0.0)
    return flat


def fixture_regions(fixtures, W, step):
    """the kmerLr_test sequences, plus lowercase, N runs, empty, shorter than W, and W, W + 1, W + step long"""
    buf, off = fixtures["kmerLr_test_seq"], fixtures["kmerLr_test_off"]
    seqs = [bytes(buf[off[i]:off[i + 1]]).decode() for i in range(len(off) - 1)]
    a = seqs[0]
    n_runs = a[:300] + "N" * 7 + a[300:520] + "NN" + a[520:700]
    return seqs + [seqs[1][:600].lower(), n_runs, "", a[:W - 1], a[:W], a[100:W + 101], a[200:W + step + 200]]


def test_gapped_models(K, oracle, fixtures):
    """gapped alphabet, k = 4..8 revcomp (TestKmers1): linear, binarized, pairs, 3-member ensembles"""
    W, step = 200, 10
    seqs = fixture_regions(fixtures, W, step)
    train = seqs[:2]
    km, om = make_model(K, oracle, train, 4, 8, 100, seed=1, revcomp=True, **GAP)
    check(K, oracle, [km], [om], seqs, W, step)
    km, om = make_model(K, oracle, train, 4, 8, 80, seed=2, revcomp=True, binarize=True, **GAP)
    check(K, oracle, [km], [om], seqs, W, step)
    km, om = make_model(K, oracle, train, 4, 8, 80, pairs=30, seed=3, revcomp=True, **GAP)
    check(K, oracle, [km], [om], seqs, W, step)
    for i, summary in enumerate(("mean", "product", "min", "max")):
        km, om = make_model(K, oracle, train, 4, 8, 40, members=3, pairs=5, summary=summary, seed=4 + i, revcomp=True,
                            **GAP)
        check(K, oracle, [km], [om], seqs, W, step)


@pytest.mark.parametrize("max_ambiguous", [None, 0, 1, 3])
@pytest.mark.parametrize("flags", [{}, dict(complement=True), dict(reverse=True), dict(complement=True, reverse=True)])
def test_gapped_rules(K, oracle, fixtures, max_ambiguous, flags):
    W, step = 120, 7
    seqs = fixture_regions(fixtures, W, step)
    km, om = make_model(K, oracle, seqs[:1], 3, 7, 60, seed=5, max_ambiguous=max_ambiguous, **flags, **GAP)
    check(K, oracle, [km], [om], seqs, W, step)
    km2, om2 = make_model(K, oracle, seqs[:1], 3, 7, 40, pairs=10, seed=6, max_ambiguous=max_ambiguous, **flags,
                          binarize=True, **GAP)
    check(K, oracle, [km2], [om2], seqs, W, step)
    check(K, oracle, [km, km2], [om, om2], seqs, W, step)            # a linear and a generic model summed


@pytest.mark.parametrize("flags", [dict(complement=True, reverse=True), dict(complement=True, revcomp=True),
                                   dict(reverse=True, revcomp=True), dict(complement=True, reverse=True, revcomp=True)])
def test_several_strand_flags(K, oracle, flags):
    seqs = regions()
    km, om = make_model(K, oracle, seqs[:1], 1, 8, 100, seed=1, **flags)
    check(K, oracle, [km], [om], seqs, 200, 10)
    km2, om2 = make_model(K, oracle, seqs[:1], 2, 6, 60, pairs=20, seed=2, binarize=True, **flags)
    check(K, oracle, [km2], [om2], seqs, 150, 25)
    km3, om3 = make_model(K, oracle, seqs[:1], 2, 5, 30, members=3, summary="mean", seed=3, **flags)
    check(K, oracle, [km3], [om3], seqs, 150, 25)


def test_long_kmers(K, oracle):
    """k = 12..14, with classes of 14 bases (28-bit codes)"""
    seqs = regions()
    for flags in ({}, dict(revcomp=True), dict(complement=True, reverse=True)):
        km, om = make_model(K, oracle, seqs[:2], 12, 14, 300, seed=7, **flags)
        assert 14 in set(np.asarray(km["class_k"]).tolist())
        check(K, oracle, [km], [om], seqs, 200, 10)
        km2, om2 = make_model(K, oracle, seqs[:2], 12, 14, 200, pairs=20, seed=8, **flags)
        check(K, oracle, [km2], [om2], seqs, 200, 10)


def test_large_class_lists(K, oracle):
    from kmerlr_b200 import synth
    big = [bytes(synth.random_bases(60_000, 11)).decode()]
    seqs = regions()[:6]
    km, om = make_model(K, oracle, big, 1, 9, 50_000, seed=9, revcomp=True)
    assert len(km["class_k"]) == 50_000
    check(K, oracle, [km], [om], seqs, 200, 10)
    km, om = make_model(K, oracle, big, 1, 8, 20_000, pairs=200, seed=10, revcomp=True, binarize=True)
    check(K, oracle, [km], [om], seqs, 200, 10)
    # the same model cut to 8192 and 8193 classes: shared-memory counts on one side, the hit table on the other
    K.api.profile(True)
    try:
        for n in (8192, 8193):
            feats = [f for f in km["features"] if f[0] < n and f[1] < n]
            th = np.concatenate([km["theta"][:, :1], km["theta"][:, 1:][:, [i for i, f in enumerate(km["features"])
                                                                            if f[0] < n and f[1] < n]]], axis=1)
            kc = dict(km, class_k=km["class_k"][:n], class_code=km["class_code"][:n], features=feats, theta=th)
            oc = dict(om, class_k=om["class_k"][:n], class_code=om["class_code"][:n], features=feats, theta=th)
            before = K.api.profile_dump()
            check(K, oracle, [kc], [oc], seqs, 200, 10)
            after = K.api.profile_dump()
            ran = {name for name in after if "score_" in name and after[name][1] > before.get(name, (0, 0))[1]}
            assert ran == ({"score_generic"} if n == 8192 else {"score_hits"}), ran
    finally:
        K.api.profile(False)


def test_wide_windows(K, oracle):
    """k = 1..13 linear model, W = 20 000 on a 200 kbp region: the prefix rows leave shared memory"""
    from kmerlr_b200 import synth
    region = bytes(synth.random_bases(200_000, 13)).decode()
    km, om = make_model(K, oracle, [region[:30_000]], 1, 13, 400, seed=11, revcomp=True)
    g = K.genomicKmerLr([km])
    for W, step in ((20_000, 1_000), (20_000, 27_000)):
        out = g.predict_window_genomic([region], W, step)[0]
        starts = np.arange(0, len(region) - W, step)
        assert len(out) == oracle.window_slots(len(region), W, step)
        # every window sums more than 10^4 terms: bound 64 eps sum |terms|, sum |terms| from the window's counts
        cw = np.zeros(len(km["class_k"]))
        for j, (a, b) in enumerate(km["features"]):
            cw[a] += km["theta"][0, j + 1]
        frozen = (km["class_k"], km["class_code"])
        for w in range(0, len(starts), 4):
            sub = region[starts[w]:starts[w] + W]
            ref = oracle.score_windows([om], [sub + "A"], W, W)[0]
            cnt = oracle.extract(om["cfg"], [sub], frozen=frozen).dense()[0]
            bound = 64 * np.finfo(float).eps * (np.abs(cnt * cw).sum() + abs(km["theta"][0, 0]))
            assert abs(out[w] - ref) <= bound + 1e-12 * abs(ref), (w, out[w], ref, bound)
        assert np.all(out[len(starts):] == 0.0)


def _logpdf_of_windows(K, km, seqs, W, step, sample):
    cfg = km["counter"]
    lr = K.logisticRegression(km["theta"][0])
    subs, pos = [], []
    for r, s in enumerate(seqs):
        for j in range(0, max(len(s) - W, 0), step):
            pos.append((r, j // step))
            subs.append(s[j:j + W])
    pick = sample.choice(len(subs), size=min(60, len(subs)), replace=False)
    d = K.compile_test_data(None, cfg, (km["class_k"], km["class_code"]), km["features"], False, cfg.binarize,
                            [subs[i] for i in pick])
    lp = lr.LogPdf(d)
    d.free()
    return [pos[i] for i in pick], lp


def test_scoring_is_extraction_plus_logpdf(K, oracle, fixtures):
    """single-member models of each new kind: a window's score = LogPdf of its extracted, frozen row"""
    W, step = 200, 10
    gseqs = fixture_regions(fixtures, W, step)[:2]
    nseqs = regions()[:6]
    rng = np.random.default_rng(12)
    cases = [
        (gseqs, make_model(K, oracle, gseqs[:1], 4, 8, 100, seed=1, revcomp=True, **GAP)[0]),
        (gseqs, make_model(K, oracle, gseqs[:1], 4, 8, 60, pairs=20, seed=2, revcomp=True, binarize=True, **GAP)[0]),
        (nseqs, make_model(K, oracle, nseqs[:1], 1, 8, 100, seed=3, complement=True, reverse=True)[0]),
        (nseqs, make_model(K, oracle, nseqs[:1], 2, 7, 60, pairs=20, seed=4, reverse=True, revcomp=True)[0]),
        (nseqs, make_model(K, oracle, nseqs[:2], 12, 14, 200, seed=5, revcomp=True)[0]),
    ]
    for seqs, km in cases:
        out = K.genomicKmerLr([km]).predict_window_genomic(seqs, W, step)
        pos, lp = _logpdf_of_windows(K, km, seqs, W, step, rng)
        got = np.array([out[r][j] for r, j in pos])
        assert np.allclose(got, lp, rtol=1e-12, atol=1e-12)


def test_trained_gapped_model_end_to_end(K, oracle, fixtures):
    """train gapped k = 4..8 revcomp on kmerLr_test_fg/bg, estimate to N = 5, score kmerLr_test_seq"""
    fg = (fixtures["kmerLr_test_fg_seq"], fixtures["kmerLr_test_fg_off"])
    bg = (fixtures["kmerLr_test_bg_seq"], fixtures["kmerLr_test_bg_off"])
    counter = K.NewKmerCounter(4, 8, revcomp=True, alphabet="gapped-nucleotide")
    data = K.compile_training_data(None, counter, None, None, True, False, fg, bg)
    est = K.KmerLrEstimator(tie=K.TIE_GO118)
    est.estimate_loop(data, 5)
    k, code = data.Kmers()
    idx = np.asarray(est.active_idx, dtype=np.int64) - 1          # theta index -> column
    assert len(idx) > 0
    ck, cc = np.asarray(k)[idx], np.asarray(code)[idx]
    feats = [(i, i) for i in range(len(idx))]
    theta = np.asarray(est.Theta, dtype=np.float64)[None, :]
    km = dict(counter=counter, class_k=ck, class_code=cc, features=feats, theta=theta, summary="")
    om = dict(cfg=oracle.make_config(4, 8, revcomp=True, alphabet="gapped-nucleotide"), class_k=ck, class_code=cc,
              features=feats, theta=theta, summary="")
    buf, off = fixtures["kmerLr_test_seq"], fixtures["kmerLr_test_off"]
    seqs = [bytes(buf[off[i]:off[i + 1]]).decode() for i in range(len(off) - 1)]
    f = check(K, oracle, [km], [om], seqs, 200, 10)
    assert np.any(f != 0.0)
    data.free()


def test_layouts_feeds_and_repeatability(K, oracle, fixtures):
    seqs = fixture_regions(fixtures, 200, 7)
    km, _ = make_model(K, oracle, seqs[:1], 4, 8, 60, seed=13, revcomp=True, **GAP)
    g = K.genomicKmerLr([km])
    W, step = 200, 7
    pw = g.predict_window(seqs, W, step)
    gen = g.predict_window_genomic(seqs, W, step)
    for s, a, b in zip(seqs, pw, gen):
        n = len(s) - W
        assert len(a) == max(n, 0)
        if n <= 0:
            continue
        starts = np.arange(0, n, step)
        assert np.array_equal(a[starts], b[:len(starts)])
        rest = np.ones(n, dtype=bool)
        rest[starts] = False
        assert np.all(a[rest] == 0.0)
    # generic models: two identical calls give identical bits
    kb, _ = make_model(K, oracle, seqs[:1], 4, 8, 60, pairs=20, seed=14, revcomp=True, binarize=True, **GAP)
    gb = K.genomicKmerLr([kb])
    x, y = gb.predict_window_genomic(seqs, W, 1), gb.predict_window_genomic(seqs, W, 1)
    assert all(np.array_equal(a, b) for a, b in zip(x, y))


def test_host_buffers_arrive_in_chunks(K, oracle, fixtures):
    """host buffers above 16 MB (chunked feed) = resident scoring, bit for bit, for a multi-flag linear model and a
    gapped linear model"""
    from kmerlr_b200 import synth
    lens = [300_000, 0, 150, 5_000_000, 17, 11_000_000, 201, 2_500_000, 64, 9_000_000, 123_457, 1_000]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    buf = synth.random_bases(int(off[-1]), 7)
    buf[1000:1040] = ord("N")
    small = [bytes(buf[off[0]:off[1]]).decode()]
    km, om = make_model(K, oracle, small, 1, 8, 100, seed=1, complement=True, reverse=True, revcomp=True)
    kg, og = make_model(K, oracle, [small[0][:3000]], 4, 8, 100, seed=2, revcomp=True, **GAP)
    W, step = 200, 10
    slots = [oracle.window_slots(int(L), W, step) for L in lens]
    for models, omodels in (([km], [om]), ([kg], [og]), ([km, kg], [om, og])):
        g = K.genomicKmerLr(models)
        out = g.predict_window_genomic((buf, off), W, step)
        assert [len(o) for o in out] == slots
        seqs = K.Sequences((buf, off))
        res = g.predict_resident(seqs, W, step, fetch=True, total_slots=sum(slots))
        seqs.free()
        assert np.array_equal(np.concatenate(out), res[:sum(slots)])
        for i in (2, 4, 6, 8):
            s = bytes(buf[off[i]:off[i + 1]]).decode()
            assert np.allclose(out[i], oracle.score_windows(omodels, [s], W, step), rtol=1e-12, atol=1e-12), i
        s = bytes(buf[off[0]:off[0] + 20_000]).decode()
        assert np.allclose(out[0][:1980], oracle.score_windows(omodels, [s], W, step)[:1980], rtol=1e-12, atol=1e-12)


def _kernels_of(K, fn):
    before = K.api.profile_dump()
    fn()
    after = K.api.profile_dump()
    # the scoring kernels only (packing the host buffers launches others)
    return {name for name in after if "score_" in name and after[name][1] > before.get(name, (0, 0))[1]}


def test_routing(K, oracle):
    """the models of test_score_gpu.py launch the kernels they launched before; the new kinds the generalised paths"""
    seqs = regions()[:5]
    K.api.profile(True)
    try:
        def run(*models, W=200, step=10, on=seqs):
            g = K.genomicKmerLr(list(models))
            return _kernels_of(K, lambda: g.predict_window_genomic(on, W, step))
        old_linear = "(score_linear<false, false>)"
        for kw in (dict(M=1, N=8, revcomp=True), dict(M=3, N=6), dict(M=2, N=5, complement=True)):
            M, N = kw.pop("M"), kw.pop("N")
            km, _ = make_model(K, oracle, seqs[:1], M, N, 40, seed=1, **kw)
            assert run(km) == {old_linear}
        km, _ = make_model(K, oracle, seqs[:1], 2, 6, 60, pairs=20, seed=5, revcomp=True, binarize=True)
        assert run(km) == {"score_generic"}
        km, _ = make_model(K, oracle, seqs[:1], 2, 5, 30, members=3, summary="mean", seed=7, revcomp=True)
        assert run(km) == {"score_generic"}
        kg, _ = make_model(K, oracle, seqs[:1], 4, 8, 40, seed=2, revcomp=True, **GAP)
        assert run(kg) == {"(score_linear<true, false>)"}
        kf, _ = make_model(K, oracle, seqs[:1], 1, 8, 40, seed=3, complement=True, reverse=True)
        assert run(kf) == {"(score_linear<true, false>)"}
        kw_, _ = make_model(K, oracle, seqs[:1], 1, 13, 40, seed=4, revcomp=True)
        from kmerlr_b200 import synth
        long_region = [bytes(synth.random_bases(20_000, 5)).decode()]
        assert run(kw_, W=17_000, step=100, on=long_region) == {"(score_linear<false, true>)"}
        kb, _ = make_model(K, oracle, seqs[:1], 4, 8, 40, seed=5, revcomp=True, binarize=True, **GAP)
        assert run(kb) == {"score_hits"}
    finally:
        K.api.profile(False)


def test_remaining_refusals(K, oracle):
    seqs = regions()[:1]
    km, _ = make_model(K, oracle, seqs, 2, 4, 10)

    def fails(**change):
        with pytest.raises(K.KmerLrError):
            K.genomicKmerLr([dict(km, **change)]).predict_window_genomic(seqs, 100, 10)

    iupac = K.NewKmerCounter(2, 4)
    iupac.alphabet = 2
    fails(counter=iupac)
    fails(theta=np.zeros((17, len(km["features"]) + 1)), summary="mean")
    fails(theta=np.zeros((2, len(km["features"]) + 1)), summary="")
    fails(class_k=np.where(np.arange(len(km["class_k"])) == 0, 5, km["class_k"]))
    fails(class_k=np.concatenate([km["class_k"][:1], km["class_k"][:-1]]),
          class_code=np.concatenate([km["class_code"][:1], km["class_code"][:-1]]))
    fails(features=km["features"][:-1] + [(0, len(km["class_k"]))])
