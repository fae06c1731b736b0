"""The scan kernels on generated automata (tests/synthdfa.py), checked bit-exact against a numpy walk of the same
table, the plain-C oracle and, for the shift register, a closed form.

Regexp front ends only make automata with a resting state and at most a few tens of thousands of states.  These
families reach what they do not: complete tables of more than 65 536 states (u32 entries: SlowStep, ReplayChunk's
packed flag, FullNext, VisitCountKernel), walks that stay outside the hot rows, one hot row, one letter or every
byte and both marks as letters, long and repeated accept lists, absorbing states.

The CPU part checks the images and the walker against the host handle and the oracle; the GPU part (each test
marked `gpu`) runs every entry point on every family."""
import functools

import numpy as np
import pytest

import synthdfa as SD
from conftest import GOLDEN
from pire_b200 import BeginMark, EndMark, Scanner
from pire_b200 import _native as N
from refpire import Oracle, oracle_count, oracle_prefix, oracle_suffix

FAMILIES = {
    # wide (u32 complete table) first
    "ring140000": lambda: SD.ring(140000),
    "ring65537": lambda: SD.ring(65537, seed=1),
    "ring65836": lambda: SD.ring(65536 + 300, seed=2),
    "shift15": lambda: SD.shift_register(15),
    "shift16": lambda: SD.shift_register(16),
    "search70000": lambda: SD.search(70000, seed=3),
    "dense70000x40": lambda: SD.dense_random(70000, 40, seed=4, absorbing=8),
    # narrow
    "ring65536": lambda: SD.ring(65536, seed=5),
    "ring65535": lambda: SD.ring(65535, seed=6),
    "search300": lambda: SD.search(300, seed=7),
    "dense1x1": lambda: SD.dense_random(1, 1, seed=8, final_share=1.0),
    "dense2x1": lambda: SD.dense_random(2, 1, seed=9, final_share=0.5),
    "dense2x2": lambda: SD.dense_random(2, 2, seed=10, final_share=0.5),
    "dense300x258": lambda: SD.dense_random(300, 258, seed=11, absorbing=6),
    "dense3000x40": lambda: SD.dense_random(3000, 40, seed=12, absorbing=6),
    "dense500x8many64": lambda: SD.dense_random(500, 8, seed=13, regexps=64, accept="many"),
    "dense500x8repeat": lambda: SD.dense_random(500, 8, seed=14, regexps=8, accept="repeat"),
    "dense40x6repeat20": lambda: SD.dense_random(40, 6, seed=15, regexps=20, accept="repeat", absorbing=4),
}
WIDE = ["ring140000", "ring65537", "ring65836", "shift15", "shift16", "search70000", "dense70000x40"]
ALL = list(FAMILIES)
MAX_HOT = (255, 6, 2, 1)
MARKS = [(True, True), (False, False), (True, False), (False, True)]


@functools.lru_cache(maxsize=None)
def family(name):
    dfa = FAMILIES[name]()
    return dfa, dfa.image()


def corpus_for(dfa, rng, nbytes, other_rate=1 / 400):
    """Bytes for a family: uniform over 0..255, except a/b for the shift register with a rare other byte."""
    if dfa.name.startswith("shift_register"):
        out = np.where(rng.random(nbytes) < 0.5, ord("a"), ord("b")).astype(np.uint8)
        hit = rng.random(nbytes) < other_rate
        out[hit] = rng.integers(0, 256, int(hit.sum()))
        return out
    return rng.integers(0, 256, nbytes, dtype=np.uint8)


def ragged(dfa, rng, n, max_len=300):
    lens = rng.integers(0, max_len + 1, n)
    lens[rng.random(n) < 0.05] = 0
    offs = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    corpus = np.concatenate([corpus_for(dfa, rng, int(offs[-1]), other_rate=1 / (4 * max_len)), np.zeros(32, np.uint8)])
    return corpus, offs


def strings_of(corpus, offs):
    return [bytes(corpus[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]


# ============================================================================ CPU

@pytest.mark.parametrize("name", ALL)
def test_host_handle_equals_generator_table(name):
    """Initialize / Next on every byte and both marks / Final / AcceptedRegexps / StateIndex of the host handle equal
    the generator's table on a sample of states, and the complete table has the width the state count calls for."""
    dfa, image = family(name)
    sc = Scanner(image, device=-1)
    info = sc.info()
    assert (info.states, info.letters, info.regexps, info.empty) == (dfa.states, dfa.letters, dfa.regexps, 0)
    assert info.table_bytes == dfa.states * dfa.letters * (4 if dfa.states > 65536 else 2)
    assert sc.Initialize() == dfa.initial
    rng = np.random.default_rng(len(name))
    sample = {0, dfa.initial, dfa.states - 1} | {s for s in (65535, 65536, 65537) if s < dfa.states}
    sample |= set(rng.integers(0, dfa.states, min(dfa.states, 160)).tolist())
    chars = list(range(256)) + [BeginMark, EndMark]
    for s in sorted(sample):
        assert [sc.Next(s, c) for c in chars] == [int(dfa.next[s, dfa.class_of[c]]) for c in chars], s
        assert sc.Final(s) == bool(dfa.final[s])
        assert sc.Dead(s) == bool(dfa.dead[s])
        assert sc.AcceptedRegexps(s) == list(dfa.accept.get(s, []))
        assert sc.StateIndex(s) == s


def test_table_width_switches_above_65536_states():
    """65 536 states keep u16 entries, 65 537 take u32 -- the count (a|b)*a(a|b){15} determinises to."""
    sr = SD.shift_register(15)
    assert sr.states == 65537
    for dfa, width in ((SD.ring(65536), 2), (SD.ring(65537), 4), (sr, 4)):
        info = Scanner(dfa.image(), device=-1).info()
        assert info.table_bytes == dfa.states * dfa.letters * width, dfa


@pytest.mark.parametrize("name", ALL)
def test_oracle_equals_walker(name):
    """The oracle over the written image and the numpy walk agree on ragged strings, every mark combination; the
    oracle's prefix, suffix and count scans run on the image (their final bits equal the walk's)."""
    dfa, image = family(name)
    orc = Oracle(image)
    rng = np.random.default_rng(100 + len(name))
    corpus, offs = ragged(dfa, rng, 3000)
    for begin, end in MARKS:
        want = dfa.walk(corpus, offs, begin=begin, end=end)
        got = orc.run(corpus, offs, begin=begin, end=end)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all(), (begin, end)
        if dfa.name.startswith("shift_register"):
            assert (want[0] == SD.shift_register_answer(dfa.states.bit_length() - 2, strings_of(corpus, offs))).all()
        counts, final = oracle_count(orc, corpus, offs, begin=begin, end=end)
        assert (final.astype(bool) == want[0]).all() and counts.shape == (3000, max(1, dfa.regexps))
        for shortest in (False, True):
            assert len(oracle_prefix(orc, corpus, offs, shortest=shortest, through_begin=begin, through_end=end)) == 3000
            assert len(oracle_suffix(orc, corpus, offs, shortest=shortest, through_end=end, through_begin=begin)) == 3000


def test_walker_long_string_path_equals_host_walk():
    """The walker's one-by-one path for long strings agrees with a walk through the host handle."""
    dfa, _ = family("dense3000x40")
    rng = np.random.default_rng(5)
    corpus = rng.integers(0, 256, 3 * 5000, dtype=np.uint8)
    offs = np.array([0, 5000, 10000, 15000])
    whole = dfa.walk(corpus, offs, begin=True, end=True)
    sc = Scanner(family("dense3000x40")[1], device=-1)
    for i in range(3):
        st = sc.Next(sc.Initialize(), BeginMark)
        for b in corpus[offs[i]:offs[i + 1]].tolist():
            st = sc.Next(st, b)
        st = sc.Next(st, EndMark)
        assert whole[2][i] == st


@pytest.mark.parametrize("case", GOLDEN, ids=lambda c: c.name)
def test_writer_round_trip_on_golden_images(case):
    """Rebuild each reference-written golden scanner from host-handle queries, write it back out: the oracle on the new
    image and the host handle on it give the golden answers."""
    src = Scanner(case.image, device=-1)
    dfa = SD.from_host_scanner(src, case.name)
    image = dfa.image()
    sc = Scanner(image, device=-1)
    corpus = np.frombuffer(b"".join(case.strings) + b"\0" * 8, np.uint8)
    offs = np.zeros(len(case.strings) + 1, np.int64)
    np.cumsum([len(s) for s in case.strings], out=offs[1:])
    final, mask, state = Oracle(image).run(corpus, offs, begin=case.begin, end=case.end)
    wf, wm, ws = dfa.walk(corpus, offs, begin=case.begin, end=case.end)
    assert final.tolist() == case.final and wf.astype(np.uint8).tolist() == case.final
    assert mask.tolist() == case.mask() and wm.tolist() == case.mask()
    if not src.Empty():
        assert state.tolist() == case.state and ws.tolist() == case.state
    assert [sc.AcceptedRegexps(int(s)) for s in state] == case.ids


# ============================================================================ GPU

def _dev(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr)).to("cuda:0")


def _unbits(bits, n):
    return np.unpackbits(bits.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)


def _run(sc, batch, begin, end):
    import torch
    n = batch.n
    bits = torch.zeros((n + 31) // 32, dtype=torch.int32, device="cuda:0")
    masks = torch.empty(n, dtype=torch.int32, device="cuda:0")
    states = torch.empty(n, dtype=torch.int32, device="cuda:0")
    flags = (N.RUN_BEGIN if begin else 0) | (N.RUN_END if end else 0)
    sc.run_batch(batch, flags, bits, masks, states)
    return _unbits(bits, n), masks.cpu().numpy().view(np.uint32), states.cpu().numpy().view(np.uint32)


def _same(got, want, what):
    for k, part in enumerate(("match bits", "accept masks", "StateIndex")):
        bad = np.nonzero(got[k] != want[k])[0]
        assert len(bad) == 0, "%s: %s differ on %d strings, first %d: got %r want %r" % (
            what, part, len(bad), bad[0], got[k][bad[0]], want[k][bad[0]])


def _reach(dfa, want, n):
    """A wide case must walk through the upper half of the table, and end there when enough states lie above it."""
    if not dfa.wide:
        return
    final, mask, state, top = want
    assert (top >= 65536).sum() >= 3, "hardly a walk enters a state >= 65536"
    if (dfa.states - 65536) / dfa.states * n >= 50 or dfa.name.startswith("shift"):
        assert (state >= 65536).sum() >= 3, "hardly a walk ends in a state >= 65536"


def _uniform(dfa, rng, n, length):
    import torch
    host = corpus_for(dfa, rng, n * length, other_rate=1 / (8 * length))
    dev = torch.empty(n * length, dtype=torch.uint8, device="cuda:0")
    dev.copy_(torch.from_numpy(host))
    import pire_b200 as P
    return host, P.Batch(dev, fixed_len=length, n=n)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_uniform_run_batch(name, cuda_device):
    """Fixed-length 32-byte aligned batches (the uniform kernels): variants 1..6 and AUTO, max_hot 255/6/2/1, lengths
    32, 64, 1024, n = 32k + 7."""
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(7)
    orc = Oracle(image)
    for length, n, (begin, end) in ((32, 32 * 130 + 7, (True, True)), (64, 32 * 128 + 7, (False, False)),
                                    (1024, 32 * 64 + 7, (True, False))):
        host, batch = _uniform(dfa, rng, n, length)
        want = dfa.walk(host, fixed_len=length, n=n, begin=begin, end=end, track_max=True)
        _reach(dfa, want, n)
        _same(orc.run(host, fixed_len=length, n=n, begin=begin, end=end), want, "oracle")
        if dfa.name.startswith("shift_register") and begin and end:
            strings = [bytes(host[i * length:(i + 1) * length]) for i in range(n)]
            assert (want[0] == SD.shift_register_answer(dfa.states.bit_length() - 2, strings)).all()
        for max_hot in MAX_HOT:
            sc.set_max_hot(max_hot)
            for variant in (1, 2, 3, 4, 5, 6, 0):
                sc.set_variant(variant)
                _same(_run(sc, batch, begin, end), want, "L=%d max_hot=%d variant=%d" % (length, max_hot, variant))
    # LOOK resolves as asked where every exit of hot id 0 is hot (the search family with 255 hot rows), and falls back to
    # PRED where one is cold: with a single hot row every byte that leaves it does
    sc.set_variant(N.VARIANT_LOOK)
    if name.startswith("search"):
        sc.set_max_hot(255)
        assert sc.info().variant == N.VARIANT_LOOK
    start = int(dfa.step(dfa.initial, SD.BEGIN_MARK))        # the first hot state (StaticHotOrder)
    if (dfa.next[start, dfa.class_of[:256]] != start).any():
        sc.set_max_hot(1)
        assert sc.info().variant == N.VARIANT_PRED


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_csr_generic(name, cuda_device):
    """Ragged CSR batches (empty strings, every start alignment 0..31) through the generic kernel: variants 0/1/2/4,
    max_hot 255/6/2/1, with and without marks."""
    import pire_b200 as P
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(11)
    corpus, offs = ragged(dfa, rng, 2500, max_len=200)
    assert set((offs[:-1] % 32).tolist()) == set(range(32)) and (np.diff(offs) == 0).any()
    batch = P.Batch(_dev(corpus), _dev(offs), n=len(offs) - 1)
    for begin, end in ((True, True), (False, False)):
        want = dfa.walk(corpus, offs, begin=begin, end=end)
        for max_hot in MAX_HOT:
            sc.set_max_hot(max_hot)
            for variant in (0, 1, 2, 4):
                sc.set_variant(variant)
                _same(_run(sc, batch, begin, end), want, "marks=%s max_hot=%d variant=%d" % ((begin, end), max_hot, variant))


SPLIT_LENGTHS = [8191, 8192, 8193, 16411, 40000, 65536, 70001, 131089]


@pytest.mark.gpu
@pytest.mark.parametrize("name", WIDE + ["ring65536", "search300", "dense300x258", "dense2x2"])
def test_length_ordered_split(name, cuda_device):
    """bin_by_length(): strings of 8 191 .. 131 089 bytes go one per warp through the split kernel (stitched across
    cold marks), the rest through the generic kernel; variants 1/2/4, max_hot 255/6/2/1, marks on and off."""
    import pire_b200 as P
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(13)
    lens = np.array(SPLIT_LENGTHS + rng.integers(0, 300, 1500).tolist() + rng.integers(4000, 8192, 20).tolist())
    lens = lens[rng.permutation(len(lens))]
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    corpus = np.concatenate([corpus_for(dfa, rng, int(offs[-1]), other_rate=1 / 30000), np.zeros(32, np.uint8)])
    batch = P.Batch(_dev(corpus), _dev(offs), n=len(lens)).bin_by_length()
    for begin, end in ((True, True), (False, False)):
        want = dfa.walk(corpus, offs, begin=begin, end=end, track_max=True)
        _reach(dfa, want, len(lens))
        for max_hot in MAX_HOT:
            sc.set_max_hot(max_hot)
            for variant in (1, 2, 4):
                sc.set_variant(variant)
                _same(_run(sc, batch, begin, end), want, "marks=%s max_hot=%d variant=%d" % ((begin, end), max_hot, variant))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_lines(name, cuda_device):
    """Batch.from_text (the lines kernel): newline-free lines, variants 1/2, max_hot 255/6/2/1."""
    import pire_b200 as P
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(17)
    corpus, offs = ragged(dfa, rng, 2000, max_len=160)
    corpus[corpus == 10] = 11
    lines = strings_of(corpus, offs)
    text = b"\n".join(lines) + b"\n"
    batch = P.Batch.from_text(_dev(np.frombuffer(text, np.uint8)))
    assert batch.n == len(lines)
    want = dfa.walk(corpus, offs, begin=True, end=True)
    for max_hot in MAX_HOT:
        sc.set_max_hot(max_hot)
        for variant in (1, 2):
            sc.set_variant(variant)
            r = P.Runner(sc).Begin().Run(batch).End()
            _same((r.Matches(), r.AcceptMasks(), r.States()), want, "max_hot=%d variant=%d" % (max_hot, variant))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_prefix_and_suffix(name, cuda_device, monkeypatch):
    """Longest/ShortestPrefix and Longest/ShortestSuffix against the oracle: all four mark combinations, the uniform
    body and the ring path of fixed-length batches, a ragged CSR batch, max_hot 255/6/2/1."""
    import pire_b200 as P
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    orc = Oracle(image)
    rng = np.random.default_rng(19)
    n, length = 32 * 40 + 7, 64
    host, batch = _uniform(dfa, rng, n, length)
    corpus, offs = ragged(dfa, rng, 1000, max_len=150)
    csr = P.Batch(_dev(corpus), _dev(offs), n=len(offs) - 1)
    fns = ((P.LongestPrefix, oracle_prefix, False), (P.ShortestPrefix, oracle_prefix, True),
           (P.LongestSuffix, oracle_suffix, False), (P.ShortestSuffix, oracle_suffix, True))
    wants = {}
    for tb, te in MARKS:
        for fn, ofn, shortest in fns:
            kw = dict(shortest=shortest, through_begin=tb, through_end=te)
            wants[tb, te, fn] = (ofn(orc, host, fixed_len=length, n=n, **kw), ofn(orc, corpus, offs, **kw))
    for max_hot in MAX_HOT:
        sc.set_max_hot(max_hot)
        for (tb, te, fn), (want, want_csr) in wants.items():
            what = (fn.__name__, tb, te, max_hot)
            kw = dict(throughBeginMark=tb, throughEndMark=te)
            monkeypatch.delenv("PIRE_B200_NO_UNIFORM_BODY", raising=False)
            got = fn(sc, batch, **kw)
            monkeypatch.setenv("PIRE_B200_NO_UNIFORM_BODY", "1")
            ring = fn(sc, batch, **kw)
            monkeypatch.delenv("PIRE_B200_NO_UNIFORM_BODY", raising=False)
            assert (got == want).all() and (ring == want).all(), what
            assert (fn(sc, csr, **kw) == want_csr).all(), what


COUNT_CASES = ["ring140000", "search70000", "dense70000x40", "shift16", "ring65535", "dense500x8many64",
               "dense500x8repeat", "dense40x6repeat20", "dense300x258", "dense1x1", "search300"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", COUNT_CASES)
def test_half_final_count(name, cuda_device, monkeypatch):
    """HalfFinalCount against the oracle: count modes 0..3, <= 16 and > 16 regexps, an id listed 16+ times in one
    state (packed counting off), uniform body and ring path, CSR, max_hot 255/2."""
    import pire_b200 as P
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    orc = Oracle(image)
    rng = np.random.default_rng(23)
    n, length = 32 * 40 + 7, 96
    host, batch = _uniform(dfa, rng, n, length)
    corpus, offs = ragged(dfa, rng, 700, max_len=150)
    csr = P.Batch(_dev(corpus), _dev(offs), n=len(offs) - 1)
    for begin, end in ((True, True), (False, False)):
        want = oracle_count(orc, host, fixed_len=length, n=n, begin=begin, end=end)
        want_csr = oracle_count(orc, corpus, offs, begin=begin, end=end)
        assert (want[1].astype(bool) == dfa.walk(host, fixed_len=length, n=n, begin=begin, end=end)[0]).all()
        for max_hot in (255, 2):
            sc.set_max_hot(max_hot)
            for mode in (0, 1, 2, 3):
                sc.set_count_mode(mode)
                for body in ("uniform", "ring"):
                    if body == "ring":
                        monkeypatch.setenv("PIRE_B200_NO_UNIFORM_BODY", "1")
                    res = P.HalfFinalCount(sc, batch, begin=begin, end=end)
                    monkeypatch.delenv("PIRE_B200_NO_UNIFORM_BODY", raising=False)
                    what = (begin, end, max_hot, mode, body)
                    assert (res.counts == want[0]).all() and (res.final == want[1].astype(bool)).all(), what
                res = P.HalfFinalCount(sc, csr, begin=begin, end=end)
                assert (res.counts == want_csr[0]).all() and (res.final == want_csr[1].astype(bool)).all(), (begin, end, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ring140000", "dense70000x40", "search70000", "shift16"])
def test_tune_on_wide_table(name, cuda_device):
    """Tune() counts visits with VisitCountKernel over the u32 table and rebuilds the hot rows: results unchanged."""
    dfa, image = family(name)
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(29)
    n, length = 32 * 64 + 7, 256
    host, batch = _uniform(dfa, rng, n, length)
    want = dfa.walk(host, fixed_len=length, n=n)
    assert sc.info().tuned == 0
    sc.Tune(batch)
    assert sc.info().tuned == 1
    for variant in (0, 1, 2, 3, 4):
        sc.set_variant(variant)
        _same(_run(sc, batch, True, True), want, "tuned, variant %d" % variant)
    import pire_b200 as P
    corpus, offs = ragged(dfa, rng, 1500)
    csr = P.Batch(_dev(corpus), _dev(offs), n=len(offs) - 1)
    sc.Tune(csr, begin=False, end=False)
    sc.set_variant(0)
    _same(_run(sc, csr, False, False), dfa.walk(corpus, offs, begin=False, end=False), "tuned on CSR")


@pytest.mark.gpu
def test_accept_sets_on_wide_table(cuda_device):
    """pire_gpu_accept_sets with 64 regexps on a 140 000-state scanner: every id, also 32..63, comes back."""
    import torch
    dfa, image = family("ring140000")
    sc = Scanner(image, cuda_device)
    assert dfa.regexps == 64 and N.lib.pire_gpu_accept_words(sc._h) == 2
    rng = np.random.default_rng(31)
    n, length = 32 * 100 + 7, 64
    host, batch = _uniform(dfa, rng, n, length)
    final, mask, state = dfa.walk(host, fixed_len=length, n=n)
    got = _run(sc, batch, True, True)
    _same(got, (final, mask, state), "run")
    states = _dev(got[2].view(np.int32))
    sets = torch.empty((n, 2), dtype=torch.int32, device="cuda:0")
    N.check(N.lib.pire_gpu_accept_sets(sc._h, states.data_ptr(), n, sets.data_ptr(), None), "pire_gpu_accept_sets")
    sets = sets.cpu().numpy().view(np.uint32)
    seen = set()
    for i in range(n):
        ids = [k for k in range(64) if (int(sets[i, k // 32]) >> (k % 32)) & 1]
        assert ids == sorted(set(dfa.accept.get(int(state[i]), []))), i
        seen.update(ids)
    assert any(k >= 32 for k in seen) and (state >= 65536).sum() > n // 10


@pytest.mark.gpu
def test_run_batch_host_chunks_on_wide_table(cuda_device, monkeypatch):
    """pire_gpu_run_batch_host in 1 MiB chunks on a 140 000-state scanner, fixed-length and CSR."""
    monkeypatch.setenv("PIRE_B200_HOST_CHUNK_MB", "1")
    dfa, image = family("ring140000")
    sc = Scanner(image, cuda_device)
    rng = np.random.default_rng(37)
    n, length = 5 * 1024 + 9, 1024
    host = corpus_for(dfa, rng, n * length)
    bits, masks, states = sc.run_batch_host(host, fixed_len=length, n=n, want_masks=True, want_states=True)
    got = (np.unpackbits(bits.view(np.uint8), bitorder="little")[:n].astype(bool), masks, states)
    _same(got, dfa.walk(host, fixed_len=length, n=n), "fixed length")
    corpus, offs = ragged(dfa, rng, 12000, max_len=700)
    bits, masks, states = sc.run_batch_host(corpus, offsets=offs, want_masks=True, want_states=True)
    n = len(offs) - 1
    got = (np.unpackbits(bits.view(np.uint8), bitorder="little")[:n].astype(bool), masks, states)
    _same(got, dfa.walk(corpus, offs), "CSR")
