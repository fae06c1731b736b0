"""The oracle (oracle/pire_oracle.c) pinned against the reference:
 * the committed golden fixtures (generated from the real reference by
   tests/golden/make_golden.py) -- always;
 * the real reference's answers to the same questions, recorded (tests/refgolden.py).
"""
import numpy as np
import pytest

from conftest import GOLDEN
from pire_ut_vectors import VECTORS
from refpire import Oracle, csr


@pytest.mark.parametrize("case", GOLDEN, ids=lambda c: c.name)
def test_oracle_matches_golden(case):
    orc = Oracle(case.image)
    assert (orc.states, orc.letters) == (case.states, case.letters) or orc.empty
    corpus, offs = csr(case.strings)
    for shortcuts in (False, True):
        final, mask, state = orc.run(corpus, offs, begin=case.begin, end=case.end, shortcuts=shortcuts)
        assert final.tolist() == case.final
        assert mask.tolist() == case.mask()
        assert state.tolist() == case.state


def test_oracle_alignment_independent():
    # pire_ut.cpp Aligned@729: results must not depend on where a string starts
    case = next(c for c in GOLDEN if c.name == "Aligned@729b")
    orc = Oracle(case.image)
    for shift in range(0, 17):
        strings = [b"J" * shift] + case.strings
        corpus, offs = csr(strings)
        final, _, _ = orc.run(corpus, offs, shortcuts=True)
        assert final.tolist()[1:] == case.final


def test_oracle_rejects_bad_images():
    case = GOLDEN[0]
    with pytest.raises(ValueError):
        Oracle(b"\0" * 128)
    with pytest.raises(ValueError):
        Oracle(case.image[: len(case.image) // 2])


def test_oracle_vs_reference_live(ref):
    """Every vector group, compiled by the real reference, incl. random text."""
    rng = np.random.default_rng(7)
    for name, pat, opts, acc, den in VECTORS:
        sc = ref.compile(pat, opts)
        orc = Oracle(sc.save())
        noise = [bytes(rng.integers(0x20, 0x7F, size=int(n), dtype=np.uint8)) for n in rng.integers(0, 200, size=64)]
        # splice the known strings into noise so that longer walks hit the accept paths too
        mixed = [noise[i] + s + noise[-i - 1] for i, s in enumerate(acc + den)]
        corpus, offs = csr(acc + den + noise + mixed)
        for begin, end in ((True, True), (False, False), (True, False), (False, True)):
            f_ref, m_ref, s_ref = sc.run(corpus, offs, begin=begin, end=end, variant=0)
            for shortcuts in (False, True):
                f, m, s = orc.run(corpus, offs, begin=begin, end=end, shortcuts=shortcuts)
                assert (f == f_ref).all() and (m == m_ref).all() and (s == s_ref).all(), name


def test_reference_variants_agree(ref):
    # NonrelocScanner (ExitMasks) and NonrelocScannerNoMask are the CPU baselines bench.py times
    from pire_b200 import workloads as W
    sc = ref.compile(*W.HEADLINE)
    spec = W.SynthSpec(512, 1024, plants=W.HEADLINE_PLANTS)
    corpus = spec.host_sample(0, 512)
    f0, _, s0 = sc.run(corpus, fixed_len=1024, variant=0)
    f1, _, _ = sc.run(corpus, fixed_len=1024, variant=1)
    f2, _, _ = sc.run(corpus, fixed_len=1024, variant=2, threads=4)
    assert (f0 == f1).all() and (f0 == f2).all()
    assert int(f0.sum()) == 512 // 8          # exactly the planted strings match
    orc = Oracle(sc.save())
    f, _, s = orc.run(corpus, fixed_len=1024, shortcuts=True)
    assert (f == f0).all() and (s == s0).all()


def test_oracle_prefix_scans_match_golden():
    """ScanBoundaries@343 / ScanTermination@475 (pire_ut.cpp): LongestPrefix / ShortestPrefix lengths."""
    from conftest import GOLDEN_PREFIX
    from refpire import oracle_prefix
    for pat, image, text, shortest, longest in GOLDEN_PREFIX:
        orc = Oracle(image)
        corpus, offs = csr([b"junk", text, b""])
        assert oracle_prefix(orc, corpus, offs, shortest=True)[1] == shortest, pat
        assert oracle_prefix(orc, corpus, offs, shortest=False)[1] == longest, pat


def test_oracle_prefix_scans_vs_reference_live(ref):
    from refpire import oracle_prefix
    rng = np.random.default_rng(21)
    for pat, opts in [(b"a+b", ""), (b"foo.*bar", "n"), (rb"[0-9]+\.[0-9]+", ""), (b"x*", "n"), (b"(ab)*c", "n"), (b".*z", "n"),
                      (b"^ab", "")]:
        sc = ref.compile(pat, opts)
        orc = Oracle(sc.save())
        strs = [bytes(rng.choice(np.frombuffer(b"abfoxz019. r", np.uint8), size=int(n))) for n in rng.integers(0, 90, size=300)]
        corpus, offs = csr(strs)
        for tb in (False, True):
            for te in (False, True):
                for shortest in (False, True):
                    want = sc.prefix(corpus, offs, shortest=shortest, through_begin=tb, through_end=te, variant=2)
                    got = oracle_prefix(orc, corpus, offs, shortest=shortest, through_begin=tb, through_end=te)
                    assert (got == want).all(), (pat, tb, te, shortest)


def test_oracle_half_final_counts_match_golden():
    """count_ut.cpp HalfFinal@553 / HalfFinalSerialization@578: Result(0..4) of the glued counters."""
    from conftest import GOLDEN_COUNTS
    from refpire import oracle_count
    for case in GOLDEN_COUNTS:
        orc = Oracle(case.image)
        assert (orc.states, orc.regexps) == (case.states, case.regexps)
        corpus, offs = csr(case.strings)
        counts, final = oracle_count(orc, corpus, offs)
        assert counts[0].tolist() == case.expect                 # the number written in the reference's test
        assert counts.tolist() == case.counts and final.tolist() == case.final
        if case.single:
            image, want, fin = case.single
            counts, final = oracle_count(Oracle(image), corpus, offs)
            assert counts[:, 0].tolist() == want and final.tolist() == fin


def test_oracle_half_final_vs_reference_live(ref):
    """All five counters, their glue and the plain HalfFinalScanner(fsm), every mark combination."""
    from pire_ut_vectors import COUNT_CASES
    from refpire import oracle_count
    rng = np.random.default_rng(5)
    for pat in sorted({p for p, _, _ in COUNT_CASES}):
        scs = [ref.compile_half_final(pat, "un", mode) for mode in (1, 2, 3, 4, 5)]
        glued = scs[0]
        for sc in scs[1:]:
            glued = ref.glue_half_final(glued, sc)
        strs = [bytes(rng.choice(np.frombuffer(b"abcde z", np.uint8), size=int(k))) for k in rng.integers(0, 120, size=150)]
        corpus, offs = csr(strs)
        for sc in scs + [glued, ref.compile_half_final(pat, "u", 0)]:
            orc = Oracle(sc.save())
            for begin, end in ((True, True), (False, False), (True, False), (False, True)):
                want, wfin = sc.count(corpus, offs, begin=begin, end=end)
                got, gfin = oracle_count(orc, corpus, offs, begin=begin, end=end)
                assert (want == got).all() and (wfin == gfin).all(), (pat, begin, end)


def test_oracle_suffix_scans_match_golden():
    """PrefixSuffix@278 (scanner of the reversed pattern) and ScanBoundaries@469-471 (the prefix table through the
    suffix scans on the reversed text)."""
    from conftest import GOLDEN_PREFIX, GOLDEN_SUFFIX
    from refpire import oracle_suffix
    for pat, image, texts, shortest, longest in GOLDEN_SUFFIX:
        orc = Oracle(image)
        corpus, offs = csr(texts)
        assert oracle_suffix(orc, corpus, offs, shortest=True).tolist() == shortest
        assert oracle_suffix(orc, corpus, offs, shortest=False).tolist() == longest
    for pat, image, text, shortest, longest in GOLDEN_PREFIX:
        orc = Oracle(image)
        corpus, offs = csr([b"junk", text[::-1], b""])
        assert oracle_suffix(orc, corpus, offs, shortest=True)[1] == shortest, pat
        assert oracle_suffix(orc, corpus, offs, shortest=False)[1] == longest, pat


def test_oracle_suffix_scans_vs_reference_live(ref):
    from refpire import oracle_suffix
    rng = np.random.default_rng(22)
    for pat, opts in [(b"a+b", "n"), (b"a+b", "nr"), (b"foo.*bar", "n"), (b"x*", "n"), (b"(ab)*c", "nr"), (b".*z", "n"), (b"^ab", ""),
                      (b"ab$", "r"), (b"[^x]*", "n")]:
        sc = ref.compile(pat, opts)
        orc = Oracle(sc.save())
        strs = [bytes(rng.choice(np.frombuffer(b"abfoxz019. r", np.uint8), size=int(n))) for n in rng.integers(0, 90, size=300)]
        corpus, offs = csr(strs)
        for te in (False, True):
            for tb in (False, True):
                for shortest in (False, True):
                    want = sc.suffix(corpus, offs, shortest=shortest, through_end=te, through_begin=tb, variant=2)
                    assert (want == sc.suffix(corpus, offs, shortest=shortest, through_end=te, through_begin=tb, variant=0)).all()
                    got = oracle_suffix(orc, corpus, offs, shortest=shortest, through_end=te, through_begin=tb)
                    assert (got == want).all(), (pat, opts, te, tb, shortest)


def test_oracle_fuzz_vs_reference_live(ref):
    """Differential fuzz on the CPU: random patterns (alternation, classes, repetition, anchors, UTF-8,
    case-insensitive, reversed), singly and glued in threes -- run, prefix / suffix scans and (as
    HalfFinalScanner) counting of the oracle port against the real reference."""
    from refpire import oracle_count, oracle_prefix, oracle_suffix
    from test_gpu_parity import _random_pattern
    rng = np.random.default_rng(777)
    alphabet = np.frombuffer(b"abcxABX 019\t." + "аб".encode(), np.uint8)
    strings = [bytes(rng.choice(alphabet, size=int(n))) for n in rng.integers(0, 100, size=400)]
    corpus, offs = csr(strings)
    compiled = []
    while len(compiled) < 40:
        pat = _random_pattern(rng)
        if rng.random() < 0.2:
            pat = b"^" + pat
        if rng.random() < 0.2:
            pat = pat + b"$"
        opts = "".join(o for o in "iunr" if rng.random() < 0.25)
        try:
            compiled.append((pat, opts, ref.compile(pat, opts)))
        except ValueError:
            continue
    for k in range(0, 12, 3):
        try:
            g = ref.glue(ref.glue(compiled[k][2], compiled[k + 1][2]), compiled[k + 2][2])
        except ValueError:
            continue
        if not g.empty:
            compiled.append((b"glue", "", g))
    for pat, opts, sc in compiled:
        orc = Oracle(sc.save())
        for begin, end in ((True, True), (False, False)):
            f_ref, m_ref, s_ref = sc.run(corpus, offs, begin=begin, end=end, variant=0)
            for shortcuts in (False, True):
                f, m, s = orc.run(corpus, offs, begin=begin, end=end, shortcuts=shortcuts)
                assert (f == f_ref).all() and (m == m_ref).all() and (s == s_ref).all(), (pat, opts, begin, end, shortcuts)
        for shortest in (False, True):
            for m1, m2 in ((False, False), (True, True)):
                want = sc.prefix(corpus, offs, shortest=shortest, through_begin=m1, through_end=m2, variant=2)
                assert (oracle_prefix(orc, corpus, offs, shortest=shortest, through_begin=m1, through_end=m2) == want).all(), (pat, opts)
                want = sc.suffix(corpus, offs, shortest=shortest, through_end=m1, through_begin=m2, variant=2)
                assert (oracle_suffix(orc, corpus, offs, shortest=shortest, through_end=m1, through_begin=m2) == want).all(), (pat, opts)
    # the same patterns as HalfFinalScanners (mode 0) and as greedy / non-greedy counters
    checked = 0
    for pat, opts, _ in compiled[:24]:
        if pat == b"glue":
            continue
        for mode in (0, 1, 4):
            try:
                hf = ref.compile_half_final(pat, opts.replace("r", ""), mode)
            except ValueError:
                continue
            if hf.empty or hf.size > 4000:
                continue
            orc = Oracle(hf.save())
            want, wfin = hf.count(corpus, offs)
            got, gfin = oracle_count(orc, corpus, offs)
            assert (got == want).all() and (gfin == wfin).all(), (pat, opts, mode)
            checked += 1
    assert checked >= 30
