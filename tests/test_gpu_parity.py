"""Parity of the CUDA path (through the C ABI) with the reference.

Checkers, in order of authority:
  1. committed golden fixtures generated from the real reference;
  2. the real reference's answers, recorded (tests/refgolden.py);
  3. the C restatement oracle/pire_oracle.c.
Bar: bit-exact match bits, accept masks and StateIndex for every string.
"""
import numpy as np
import pytest

from conftest import GOLDEN
from refpire import Oracle, csr

pytestmark = pytest.mark.gpu


def gpu_run(sc, strings, begin=True, end=True):
    import pire_b200 as P
    batch = P.Batch.from_strings(strings)
    r = P.Runner(sc)
    if begin:
        r.Begin()
    r.Run(batch)
    if end:
        r.End()
    return r.Matches().astype(np.uint8), r.AcceptMasks(), r.States()


def checker_run(image, strings, begin, end, ref_sc=None):
    corpus, offs = csr(strings)
    if ref_sc is not None:
        return ref_sc.run(corpus, offs, begin=begin, end=end, variant=0)
    return Oracle(image).run(corpus, offs, begin=begin, end=end)


@pytest.mark.parametrize("variant", [1, 2, 4, 6], ids=["plain", "pred", "look", "look1"])
@pytest.mark.parametrize("case", GOLDEN, ids=lambda c: c.name)
def test_golden_vectors(case, variant, cuda_device):
    import pire_b200 as P
    sc = P.Scanner(case.image, cuda_device)
    sc.set_variant(variant)
    final, mask, state = gpu_run(sc, case.strings, case.begin, case.end)
    assert final.tolist() == case.final
    assert mask.tolist() == case.mask()
    if not sc.Empty():
        assert state.tolist() == case.state
    for i, ids in enumerate(case.ids):
        assert sc.AcceptedRegexps(int(state[i])) == ids


def test_alignment_and_ragged_lengths(cuda_device):
    """pire_ut.cpp Aligned@729 and the head/body/tail split of run.h:186-226: every
    golden string at every start alignment 0..31, surrounded by junk strings of
    ragged lengths (0..70), empty strings included."""
    import pire_b200 as P
    rng = np.random.default_rng(3)
    for case in [c for c in GOLDEN if c.begin and c.name.split("@")[0] in ("Aligned", "TestShortcuts", "String", "UTF8")]:
        sc = P.Scanner(case.image, cuda_device)
        strings, expect = [], []
        for shift in range(32):
            for s, f in zip(case.strings, case.final):
                strings.append(bytes(rng.integers(0x20, 0x7F, size=shift, dtype=np.uint8)))
                expect.append(None)
                strings.append(s)
                expect.append(f)
                strings.append(b"")
                expect.append(None)
        junk = [bytes(rng.integers(0, 256, size=int(n), dtype=np.uint8)) for n in rng.integers(0, 70, size=50)]
        strings += junk
        expect += [None] * len(junk)
        f2, m2, s2 = checker_run(case.image, strings, True, True)
        for variant in (0, 2, 4):                    # AUTO (plain for CSR), exit filter, look-ahead filter
            sc.set_variant(variant)
            final, mask, state = gpu_run(sc, strings)
            assert (final == f2).all() and (mask == m2).all() and (state == s2).all(), (case.name, variant)
            for got, want in zip(final.tolist(), expect):
                assert want is None or got == want


def test_mark_flag_combinations(cuda_device, ref):
    import pire_b200 as P
    sc_ref = ref.compile(rb"^abc$|x+y", "")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    strings = [b"abc", b"zabc", b"abcz", b"xxy", b"", b"x", b"y" * 40 + b"xy", b"abc" * 20]
    for begin in (False, True):
        for end in (False, True):
            got = gpu_run(sc, strings, begin, end)
            want = checker_run(None, strings, begin, end, sc_ref)
            for g, w in zip(got, want):
                assert (g == w).all(), (begin, end)


def test_empty_batch_and_empty_scanner(cuda_device):
    import torch
    import pire_b200 as P
    case = next(c for c in GOLDEN if c.name == "EmptyScanner@784")
    sc = P.Scanner(case.image, cuda_device)
    assert sc.Empty() and sc.RegexpsCount() == 0
    final, mask, _ = gpu_run(sc, [b"a string", b"", b"regex" * 100])
    assert final.tolist() == [0, 0, 0] and mask.tolist() == [0, 0, 0]
    # n == 0 is a no-op (pire_ut.cpp NullPointer@832: Run(nullptr, nullptr) is legal)
    batch = P.Batch(torch.zeros(32, dtype=torch.uint8, device="cuda:0"), fixed_len=0, n=0)
    assert P.Runner(sc).Begin().Run(batch).End().Matches().size == 0
    # n > 0 strings of length zero
    batch = P.Batch(torch.zeros(32, dtype=torch.uint8, device="cuda:0"), fixed_len=0, n=5)
    sc2 = P.Scanner(next(c for c in GOLDEN if c.name == "Misc@238a").image, cuda_device)
    assert P.Runner(sc2).Begin().Run(batch).End().Matches().tolist() == [True] * 5   # ^[^\s=/>]*$ accepts ""


def random_text(rng, n, length, alphabet=None):
    if alphabet is None:
        return rng.integers(0x20, 0x7F, size=(n, length), dtype=np.uint8)
    return rng.choice(np.frombuffer(alphabet, np.uint8), size=(n, length))


@pytest.mark.parametrize("variant", [1, 2, 3, 4, 5, 6], ids=["plain", "pred", "priv", "look", "look64", "look1"])
def test_uniform_kernel_headline(variant, cuda_device, ref):
    """Fixed 1 KiB strings (the BASELINE configs' shape) through the uniform kernel,
    full comparison with the reference on 64 Ki strings, incl. StateIndex."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.compile(*W.HEADLINE)
    sc = P.Scanner(sc_ref.save(), cuda_device)
    sc.set_variant(variant)
    n = 65536 + 7                      # ragged last warp
    spec = W.SynthSpec(n, 1024, plants=W.HEADLINE_PLANTS)
    dev = torch.empty(spec.total_bytes(), dtype=torch.uint8, device="cuda:0")
    spec.fill_device(dev)
    host = spec.host_sample(0, n)
    assert (dev.cpu().numpy() == host).all()          # host and device generators agree
    r = P.Runner(sc).Begin().Run(P.Batch(dev, fixed_len=1024, n=n)).End()
    f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=1024, n=n, variant=1, threads=8)
    assert (r.Matches().astype(np.uint8) == f_ref).all()
    assert (r.AcceptMasks() == m_ref).all()
    assert (r.States() == s_ref).all()
    assert int(f_ref.sum()) == (n + 7) // 8
    # bits past n in the last bitmap word are zero
    words = r.MatchBits().cpu().numpy().view(np.uint32)
    assert int(words[-1]) >> (n % 32) == 0


@pytest.mark.parametrize("max_hot,tune", [(255, False), (255, True), (6, False), (2, True)],
                         ids=["static", "tuned", "hot6", "hot2-tuned"])
def test_glued_ten_patterns(max_hot, tune, cuda_device, ref):
    """The 10-regexp glued scanner (29 664 states): hot rows in shared memory, the
    rest replayed through the L2-resident table.  Tiny hot sets force the replay
    and cold-state paths on almost every chunk."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.glue_all(W.GLUE10)
    sc = P.Scanner(sc_ref.save(), cuda_device)
    assert (sc.Size(), sc.RegexpsCount()) == (sc_ref.size, 10)
    n = 16384
    spec = W.SynthSpec(n, 1024, plants=W.GLUE10_PLANTS)
    dev = torch.empty(spec.total_bytes(), dtype=torch.uint8, device="cuda:0")
    spec.fill_device(dev)
    batch = P.Batch(dev, fixed_len=1024, n=n)
    sc.set_max_hot(max_hot)
    if tune:
        sc.Tune(batch, 4096)
        assert sc.info().tuned == 1
    host = spec.host_sample(0, n)
    f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=1024, n=n, variant=1, threads=8)
    assert int((m_ref != 0).sum()) >= n // 8
    for variant in (1, 2, 3, 4, 5):
        sc.set_variant(variant)
        r = P.Runner(sc).Begin().Run(batch).End()
        assert (r.Matches().astype(np.uint8) == f_ref).all(), variant
        assert (r.AcceptMasks() == m_ref).all(), variant
        assert (r.States() == s_ref).all(), variant
    # every planted literal is reported under its own regexp id
    for i in range(0, 80, 8):
        assert m_ref[i] & (1 << ((i // 8) % 10))


def test_generic_kernel_mixed_lengths_utf8(cuda_device, ref):
    """BASELINE config 4's shape: UTF-8 + CaseInsensitive pattern, lengths 16 B..64 KiB
    (CSR offsets), bytes from the whole 0..255 range."""
    import pire_b200 as P
    sc_ref = ref.compile(rb"hello\s+w.+d$", "iu")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    rng = np.random.default_rng(11)
    lens = np.exp(rng.uniform(np.log(16), np.log(65536), size=600)).astype(int)
    alphabet = b"abcdehlorw HELOWRD\t" + "привет мир".encode() + bytes(range(0x20, 0x7F))
    strings = []
    for i, n in enumerate(lens):
        body = bytearray(random_text(rng, 1, int(n), alphabet)[0].tobytes())
        if i % 5 == 0:
            hit = b"HeLLo \t WoRLD"
            body[-len(hit):] = hit
        strings.append(bytes(body))
    got = gpu_run(sc, strings)
    want = checker_run(None, strings, True, True, sc_ref)
    for g, w in zip(got, want):
        assert (g == w).all()
    assert int(want[0].sum()) >= len(strings) // 5


@pytest.mark.parametrize("variant", [1, 2, 3, 4, 5, 6], ids=["plain", "pred", "priv", "look", "look64", "look1"])
def test_uniform_kernel_binary_bytes(variant, cuda_device, ref):
    """Fixed-length strings over the whole byte range (UTF-8 pattern): the private-row
    kernel covers bytes < 128 only and must re-walk every word holding a byte >= 128."""
    import torch
    import pire_b200 as P
    sc_ref = ref.compile("привет|hello\\s+w.+d$".encode(), "iu")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    sc.set_variant(variant)
    rng = np.random.default_rng(17)
    n, length = 3000, 256
    alphabet = "привет ПРИВЕТ hello world HELLO WORLD\t".encode() + bytes(range(256))
    host = random_text(rng, n, length, alphabet)
    for i in range(0, n, 3):
        hit = "ПрИвЕт".encode() if i % 2 else b"HeLLo  WoRLd"
        host[i, -len(hit):] = np.frombuffer(hit, np.uint8)
    host = np.ascontiguousarray(host).reshape(-1)
    dev = torch.from_numpy(host).to("cuda:0")
    batch = P.Batch(dev, fixed_len=length, n=n)
    sc.Tune(batch, 512)
    r = P.Runner(sc).Begin().Run(batch).End()
    f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=length, n=n)
    assert (r.Matches().astype(np.uint8) == f_ref).all()
    assert (r.States() == s_ref).all()
    assert int(f_ref.sum()) >= n // 3


@pytest.mark.parametrize("length", [32, 64, 96, 480, 1024])
def test_look_variant_dense_near_misses(length, cuda_device, ref):
    """LOOK variant (one byte of look-ahead over the exit filter): text made almost only of the bytes that start
    or continue the ten patterns, so that nearly every position is an exit byte followed by a continuing or a
    non-continuing byte, strings that end on exit bytes and on half matches, every mark combination, static and
    tuned hot rows.  Everything must equal the reference (and the plain kernel)."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.glue_all(W.GLUE10)
    sc = P.Scanner(W.load_image("glue10"), cuda_device)
    rng = np.random.default_rng(length)
    n = 4096 + 5
    dense = b"(0123456789ABCXYZaefhilmorstuw)-: /GET"
    sparse = bytes(range(0x20, 0x7F))
    host = np.empty((n, length), np.uint8)
    for i in range(n):
        mix = rng.random()
        alphabet = dense if mix < 0.6 else dense + sparse
        row = rng.choice(np.frombuffer(alphabet, np.uint8), size=length)
        if i % 7 == 0:
            lit = W.GLUE10_PLANTS[(i // 7) % 10].lstrip(b"^$")
            cut = int(rng.integers(1, len(lit) + 1))                  # whole literals and proper prefixes of them
            at = int(rng.integers(0, max(1, length - cut))) if i % 14 else length - cut
            row[at:at + cut] = np.frombuffer(lit[:cut], np.uint8)[:length - at]
        host[i] = row
    host = np.ascontiguousarray(host).reshape(-1)
    dev = torch.from_numpy(host).to("cuda:0")
    batch = P.Batch(dev, fixed_len=length, n=n)
    for tuned in (False, True):
        if tuned:
            sc.Tune(batch, 2048)
        for begin in (True, False):
            for end in (True, False):
                f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=length, n=n, begin=begin, end=end, variant=1, threads=8)
                for variant in (1, 4, 5, 6):
                    sc.set_variant(variant)
                    r = P.Runner(sc)
                    r = r.Begin() if begin else r
                    r = r.Run(batch)
                    r = r.End() if end else r
                    assert (r.Matches().astype(np.uint8) == f_ref).all(), (variant, tuned, begin, end)
                    assert (r.AcceptMasks() == m_ref).all(), (variant, tuned, begin, end)
                    assert (r.States() == s_ref).all(), (variant, tuned, begin, end)


def test_auto_picks_the_shape_of_the_look_ahead_walk_by_batch_size(cuda_device, ref):
    """AUTO on a large automaton means the look-ahead filter: two strings per lane when the batch gives every resident
    warp a pair of units, one string per lane below that (capi.cu).  Both sides of the threshold, odd and partial last
    units, against the reference."""
    import torch
    import pire_b200 as P
    from pire_b200 import _native as N
    from pire_b200 import workloads as W
    sc_ref = ref.glue_all(W.GLUE10)
    sc = P.Scanner(W.load_image("glue10"), cuda_device)
    assert sc.info().variant == N.VARIANT_LOOK                      # AUTO, no timing run: > 64 states, look-ahead set complete
    length = 64
    for n in (33, 1000 + 7, 64 * 6000 + 32 + 5):                    # one pair, a few hundred pairs, more pairs than resident warps
        spec = W.SynthSpec(n, length, plants=[p[:40] for p in W.GLUE10_PLANTS], plant_every=3)
        dev = torch.empty(spec.total_bytes(), dtype=torch.uint8, device="cuda:0")
        spec.fill_device(dev)
        host = dev.cpu().numpy()
        f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=length, n=n, variant=1, threads=8)
        r = P.Runner(sc).Begin().Run(P.Batch(dev, fixed_len=length, n=n)).End()
        assert (r.Matches().astype(np.uint8) == f_ref).all(), n
        assert (r.AcceptMasks() == m_ref).all() and (r.States() == s_ref).all(), n


def test_noexit_early_stop_is_exact(cuda_device, ref):
    """multi.h:955-958: a state no byte can leave ends the walk early; End() must still be
    stepped.  'foo' un-anchored parks every matching string in an absorbing state."""
    import pire_b200 as P
    sc_ref = ref.compile(rb"foo", "")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    rng = np.random.default_rng(5)
    strings = [b"foo" + bytes(random_text(rng, 1, 4000)[0]) for _ in range(64)]      # whole warps park
    strings += [bytes(random_text(rng, 1, 4000)[0]) for _ in range(32)]
    strings += [b"x" * 100 + b"foo" + b"y" * 3000 for _ in range(16)] + [b"fo" * 900 for _ in range(16)]
    got = gpu_run(sc, strings)
    want = checker_run(None, strings, True, True, sc_ref)
    for g, w in zip(got, want):
        assert (g == w).all()


def test_host_buffer_entry_point(cuda_device, ref):
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.compile(*W.HEADLINE)
    sc = P.Scanner(sc_ref.save(), cuda_device)
    spec = W.SynthSpec(4096, 1024, plants=W.HEADLINE_PLANTS)
    host = spec.host_sample(0, 4096)
    bits, masks, states = sc.run_batch_host(host, fixed_len=1024, n=4096, want_masks=True, want_states=True)
    f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=1024, n=4096)
    got = np.unpackbits(bits.view(np.uint8), bitorder="little")[:4096]
    assert (got == f_ref).all() and (masks == m_ref).all() and (states == s_ref).all()
    # CSR through the same entry point
    strings = [bytes(host[i * 1024: i * 1024 + 100 + i]) for i in range(200)]
    corpus, offs = csr(strings)
    bits, masks, states = sc.run_batch_host(corpus, offsets=offs, want_masks=True, want_states=True)
    f_ref, m_ref, s_ref = sc_ref.run(corpus, offs)
    assert (np.unpackbits(bits.view(np.uint8), bitorder="little")[:200] == f_ref).all() and (states == s_ref).all()


def test_full_size_properties(cuda_device, ref):
    """BASELINE config 1 at full size (2^20 x 1 KiB): the match vector is bit-exact against
    the reference run on all host cores; at 4x that size only size-independent
    properties are checked (planted count, determinism, shard decomposition)."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    from pire_b200.dist import shard_bounds
    sc_ref = ref.compile(*W.HEADLINE)
    sc = P.Scanner(sc_ref.save(), cuda_device)
    n = 1 << 20
    spec = W.SynthSpec(n, 1024, plants=W.HEADLINE_PLANTS)
    dev = torch.empty(spec.total_bytes(), dtype=torch.uint8, device="cuda:0")
    spec.fill_device(dev)
    r = P.Runner(sc).Begin().Run(P.Batch(dev, fixed_len=1024, n=n)).End()
    got = r.Matches()
    host = dev.cpu().numpy()
    f_ref, _, _ = sc_ref.run(host, fixed_len=1024, n=n, variant=1, threads=ref.hardware_threads(), want=("final",))
    assert (got.astype(np.uint8) == f_ref).all()
    assert int(got.sum()) == n // 8
    del host
    # shards of the same corpus give the same bits as the whole
    whole = r.MatchBits().cpu().numpy()
    parts = []
    for rank in range(4):
        lo, hi = shard_bounds(n, rank, 4)
        sub = P.Batch(dev[lo * 1024: hi * 1024], fixed_len=1024, n=hi - lo)
        parts.append(P.Runner(sc).Begin().Run(sub).End().MatchBits().cpu().numpy())
    assert (np.concatenate(parts) == whole).all()


def test_length_binned_launch_mixed_utf8(cuda_device, ref):
    """BASELINE config 4 through the length-binned (ordered) launch: device- and host-generated
    corpora agree; match bits / masks / StateIndex, indexed by ORIGINAL string number, are
    bit-exact against the reference, with and without binning."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.compile(*W.HEADLINE_IU)
    sc = P.Scanner(W.load_image("headline_iu"), cuda_device)
    assert sc.Size() == sc_ref.size
    n = 6000
    spec = W.MixedSpec(n)
    corpus, offsets = spec.device_batch("cuda:0")
    h_corpus, h_offsets = spec.host_batch(0, n)
    assert (offsets.cpu().numpy().astype(np.uint64) == h_offsets).all()
    assert (corpus.cpu().numpy()[: int(h_offsets[-1])] == h_corpus[: int(h_offsets[-1])]).all()
    f_ref, m_ref, s_ref = sc_ref.run(h_corpus, h_offsets, variant=1, threads=8)
    assert int(f_ref.sum()) >= n // 8 * 0.9
    for binned in (False, True):
        batch = P.Batch(corpus, offsets, n=n)
        if binned:
            batch.bin_by_length()
            order = batch.order.cpu().numpy()
            lens = np.diff(h_offsets.astype(np.int64))
            assert sorted(order.tolist()) == list(range(n))
            sorted_lens = lens[order]
            msb = np.floor(np.log2(sorted_lens)).astype(int)
            bucket = 2 * msb + ((sorted_lens >> np.maximum(msb - 1, 0)) & 1)   # [2^k, 1.5*2^k) and [1.5*2^k, 2^(k+1))
            assert (np.diff(bucket) <= 0).all()                          # longest bucket first, corpus order inside
            same = np.diff(bucket) == 0
            assert (np.diff(order)[same] > 0).all()
        for variant in (1, 2, 4):
            sc.set_variant(variant)
            r = P.Runner(sc).Begin().Run(batch).End()
            assert (r.Matches().astype(np.uint8) == f_ref).all(), (binned, variant)
            assert (r.AcceptMasks() == m_ref).all() and (r.States() == s_ref).all(), (binned, variant)
    # the host-buffer entry point bins CSR batches itself
    bits, masks, states = sc.run_batch_host(h_corpus, offsets=h_offsets, want_masks=True, want_states=True)
    assert (np.unpackbits(bits.view(np.uint8), bitorder="little")[:n] == f_ref).all() and (states == s_ref).all()


def test_autoselect_keeps_results(cuda_device, ref):
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    sc_ref = ref.glue_all(W.GLUE10)
    sc = P.Scanner(W.load_image("glue10"), cuda_device)
    n = 32768
    spec = W.SynthSpec(n, 1024, plants=W.GLUE10_PLANTS)
    dev = torch.empty(spec.total_bytes(), dtype=torch.uint8, device="cuda:0")
    spec.fill_device(dev)
    batch = P.Batch(dev, fixed_len=1024, n=n)
    sc.Tune(batch, 4096)
    ms = sc.AutoSelect(batch)
    assert set(ms) >= {"plain", "pred"} and all(v > 0 for v in ms.values())
    assert sc.info().variant in (1, 2, 3, 4, 5)
    r = P.Runner(sc).Begin().Run(batch).End()
    f_ref, m_ref, _ = sc_ref.run(spec.host_sample(0, n), fixed_len=1024, n=n, variant=1, threads=8)
    assert (r.Matches().astype(np.uint8) == f_ref).all() and (r.AcceptMasks() == m_ref).all()


def test_prefix_scans_golden(cuda_device):
    """Pire::LongestPrefix / ShortestPrefix on the device against the reference's own
    ScanBoundaries@343 / ScanTermination@475 table."""
    import pire_b200 as P
    from conftest import GOLDEN_PREFIX
    for pat, image, text, shortest, longest in GOLDEN_PREFIX:
        sc = P.Scanner(image, cuda_device)
        batch = P.Batch.from_strings([b"junk", text, b"", text + b"tail"])
        s = P.ShortestPrefix(sc, batch)
        l = P.LongestPrefix(sc, batch)
        assert s[1] == shortest and l[1] == longest, (pat, s.tolist(), l.tolist())


def test_prefix_scans_vs_reference(cuda_device, ref):
    """Random text, all four mark combinations, hot sets small enough to force cold states;
    checker = the reference's byte-by-byte (NoMask) scanner and the oracle."""
    import pire_b200 as P
    from refpire import oracle_prefix
    rng = np.random.default_rng(33)
    for pat, opts in [(b"a+b", ""), (b"foo.*bar", "n"), (rb"[0-9]+\.[0-9]+", ""), (b"x*", "n"), (b"(ab)*c", "n"), (b".*z", "n"),
                      (b"^ab", ""), (b"[^x]*", "n")]:
        sc_ref = ref.compile(pat, opts)
        image = sc_ref.save()
        orc = Oracle(image)
        strs = [bytes(rng.choice(np.frombuffer(b"abfoxz019. r", np.uint8), size=int(n))) for n in rng.integers(0, 400, size=700)]
        strs += [b"a" * n for n in (15, 16, 17, 31, 32, 33, 64)]        # the 16-byte-boundary cases of the ExitMasks quirk
        corpus, offs = csr(strs)
        for max_hot in (255, 2):
            sc = P.Scanner(image, cuda_device)
            sc.set_max_hot(max_hot)
            batch = P.Batch.from_strings(strs)
            for tb in (False, True):
                for te in (False, True):
                    for shortest in (False, True):
                        fn = P.ShortestPrefix if shortest else P.LongestPrefix
                        got = fn(sc, batch, throughBeginMark=tb, throughEndMark=te)
                        want = sc_ref.prefix(corpus, offs, shortest=shortest, through_begin=tb, through_end=te, variant=2)
                        assert (got == want).all(), (pat, max_hot, tb, te, shortest, np.nonzero(got != want)[0][:5])
                        assert (got == oracle_prefix(orc, corpus, offs, shortest=shortest, through_begin=tb, through_end=te)).all()
    # fixed-length batch through the same entry point
    sc_ref = ref.compile(b"ab+c", "")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    host = rng.choice(np.frombuffer(b"abc ", np.uint8), size=(5000, 64)).reshape(-1)
    import torch
    got = P.LongestPrefix(sc, P.Batch(torch.from_numpy(host).to("cuda:0"), fixed_len=64, n=5000))
    assert (got == sc_ref.prefix(host, fixed_len=64, n=5000, variant=2)).all()


def _random_pattern(rng, depth=0):
    atoms = [b"a", b"b", b"c", b"x", b"0", b"\\d", b"\\s", b"\\w", b".", b"[a-c]", b"[^a]", b"ab", b"hello", b"\xd0\xb0", b" "]
    r = rng.random()
    if depth > 2 or r < 0.45:
        a = atoms[int(rng.integers(len(atoms)))]
    elif r < 0.65:
        a = b"(" + _random_pattern(rng, depth + 1) + b"|" + _random_pattern(rng, depth + 1) + b")"
    else:
        a = _random_pattern(rng, depth + 1) + _random_pattern(rng, depth + 1)
    q = rng.random()
    if q < 0.15:
        a = (b"(" + a + b")" if len(a) > 1 and not a.startswith(b"(") and not a.startswith(b"[") and not a.startswith(b"\\") else a) + b"*"
    elif q < 0.25:
        a = (b"(" + a + b")" if len(a) > 1 and not a.startswith(b"(") and not a.startswith(b"[") and not a.startswith(b"\\") else a) + b"+"
    elif q < 0.32:
        a = (b"(" + a + b")" if len(a) > 1 and not a.startswith(b"(") and not a.startswith(b"[") and not a.startswith(b"\\") else a) + b"{1,3}"
    return a


def test_fuzz_random_patterns(cuda_device, ref):
    """Differential fuzz: random patterns (alternation, classes, repetition, anchors, UTF-8,
    case-insensitive), singly and glued in threes, over random strings; every output of every
    kernel variant must equal the reference's."""
    import pire_b200 as P
    rng = np.random.default_rng(2024)
    alphabet = b"abcxABX 019\t." + "аб".encode()
    compiled = []
    while len(compiled) < 36:
        pat = _random_pattern(rng)
        if rng.random() < 0.2:
            pat = b"^" + pat
        if rng.random() < 0.2:
            pat = pat + b"$"
        opts = "".join(o for o in "iu" if rng.random() < 0.3)
        try:
            compiled.append((pat, opts, ref.compile(pat, opts)))
        except ValueError:
            continue
    scanners = [(p, o, sc) for p, o, sc in compiled]
    for k in range(0, 12, 3):                                    # glued triples
        try:
            g = ref.glue(ref.glue(compiled[k][2], compiled[k + 1][2]), compiled[k + 2][2])
        except ValueError:
            continue
        if not g.empty:
            scanners.append((b"glue", "", g))
    strings = [bytes(rng.choice(np.frombuffer(alphabet, np.uint8), size=int(n))) for n in rng.integers(0, 120, size=1500)]
    corpus, offs = csr(strings)
    batch = P.Batch.from_strings(strings)
    fixed = rng.choice(np.frombuffer(alphabet, np.uint8), size=(2048, 64)).reshape(-1)
    import torch
    fixed_batch = P.Batch(torch.from_numpy(fixed).to("cuda:0"), fixed_len=64, n=2048)
    for pat, opts, sc_ref in scanners:
        sc = P.Scanner(sc_ref.save(), cuda_device)
        sc.Tune(batch, 512)
        want = sc_ref.run(corpus, offs, variant=0)
        want_fixed = sc_ref.run(fixed, fixed_len=64, n=2048, variant=0)
        for variant in (1, 2, 3, 4, 5):
            sc.set_variant(variant)
            r = P.Runner(sc).Begin().Run(batch).End()
            ok = (r.Matches().astype(np.uint8) == want[0]).all() and (r.AcceptMasks() == want[1]).all()
            assert ok and (r.States() == want[2]).all(), (pat, opts, variant)
            r = P.Runner(sc).Begin().Run(fixed_batch).End()
            assert (r.Matches().astype(np.uint8) == want_fixed[0]).all() and (r.States() == want_fixed[2]).all(), (pat, opts, variant)
        for shortest in (False, True):
            fn = P.ShortestPrefix if shortest else P.LongestPrefix
            got = fn(sc, batch, throughBeginMark=True)
            assert (got == sc_ref.prefix(corpus, offs, shortest=shortest, through_begin=True, variant=2)).all(), (pat, opts, shortest)


def test_lines_front_end(cuda_device, ref):
    """samples/pigrep/pigrep.cpp:38-45: std::getline per line, then Runner(sc).Begin().Run(line).End().
    Lines are found on the device; the newline is not part of a line ('$' must see the line end);
    empty lines, a last line without newline and an empty text follow getline."""
    import torch
    import pire_b200 as P
    sc_ref = ref.compile(rb"timeout$|^GET |error", "")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    rng = np.random.default_rng(9)
    words = [b"GET /index", b"timeout", b"error 42", b"ok", b"", b"a timeout", b"timeout ", b"x" * 300, b"the error"]
    for ending in (b"\n", b""):
        lines = [words[int(k)] + bytes(rng.integers(0x20, 0x7F, size=int(rng.integers(0, 40)), dtype=np.uint8)) * int(rng.integers(0, 2))
                 for k in rng.integers(0, len(words), size=5000)]
        lines = [l.replace(b"\n", b" ") for l in lines]
        text = b"\n".join(lines) + ending
        expect_lines = text.split(b"\n")
        if text.endswith(b"\n") or text == b"":
            expect_lines = expect_lines[:-1]                      # std::getline: no empty line after a final newline
        batch = P.Batch.from_text(torch.from_numpy(np.frombuffer(text, np.uint8).copy()).to("cuda:0"))
        assert batch.n == len(expect_lines)
        offs = batch.offsets.cpu().numpy()
        for i in (0, 1, batch.n // 2, batch.n - 1):
            assert text[offs[i]: offs[i + 1] - 1] == expect_lines[i]
        corpus, o = csr(expect_lines)
        want = sc_ref.run(corpus, o, variant=0)
        for binned in (False, True):
            if binned:
                batch.bin_by_length()
            r = P.Runner(sc).Begin().Run(batch).End()
            assert (r.Matches().astype(np.uint8) == want[0]).all() and (r.AcceptMasks() == want[1]).all() and (r.States() == want[2]).all()
        # the other CSR entry points honour the line flag too (tune reads no byte past a line's end)
        sc.Tune(batch, 2048)
        assert (P.Runner(sc).Begin().Run(batch).End().AcceptMasks() == want[1]).all()
        got = P.LongestPrefix(sc, batch, throughBeginMark=True, throughEndMark=True)
        assert (got == sc_ref.prefix(corpus, o, through_begin=True, through_end=True, variant=2)).all()
    empty = P.Batch.from_text(torch.zeros(0, dtype=torch.uint8, device="cuda:0"))
    assert empty.n == 0
    one = P.Batch.from_text(torch.from_numpy(np.frombuffer(b"\n", np.uint8).copy()).to("cuda:0"))
    assert one.n == 1 and P.Runner(sc).Begin().Run(one).End().Matches().tolist() == [False]


def _text_of(rng, n_lines, ending):
    words = [b"GET /index", b"timeout", b"error 42", b"ok", b"", b"a timeout", b"$(555) 123-4567", b"fatal", b"https://x", b"hello \t world"]
    lens = [0, 0, 1, 2, 7, 15, 16, 17, 31, 32, 33, 47, 48, 63, 64, 65, 100, 200]
    lines = []
    for k in range(n_lines):
        r = rng.random()
        if r < 0.15:
            body = b""
        elif r < 0.25:
            body = bytes(rng.integers(0x20, 0x7F, size=int(rng.choice(lens)), dtype=np.uint8))
        else:
            body = bytes(rng.integers(0x20, 0x7F, size=int(rng.integers(0, 60)), dtype=np.uint8))
        w = words[int(rng.integers(0, len(words)))] if rng.random() < 0.4 else b""
        where = rng.random()
        lines.append(w + body if where < 0.4 else body + w if where < 0.8 else body[: len(body) // 2] + w + body[len(body) // 2:])
    # lines longer than a segment (1 KiB) and longer than a warp's unit of 32 segments, in the middle and at the end
    lines[n_lines // 3] = bytes(rng.integers(0x20, 0x7F, size=1500, dtype=np.uint8)) + b"error"
    lines[n_lines // 2] = bytes(rng.integers(0x20, 0x7F, size=40000, dtype=np.uint8)) + b" timeout"
    lines[-1] = bytes(rng.integers(0x20, 0x7F, size=5000, dtype=np.uint8))
    for k in range(n_lines // 4, n_lines // 4 + 50):
        lines[k] = b""                                             # a run of empty lines: several ends in one chunk
    return b"\n".join(lines) + ending, lines


def test_lines_in_stream(cuda_device, ref):
    """The in-stream lines kernel (one text segment per lane, the walk restarts behind every newline) against the
    reference line by line: lengths around the 16/32-byte chunk sizes, runs of empty lines, lines longer than a
    segment and than a warp's 32 segments, every alignment of the text in memory, with and without a last newline,
    plain and exit-filter walks, hot sets small enough that lanes leave the hot rows inside lines, and a scanner
    whose every line matches (atomics on every bitmap word)."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    rng = np.random.default_rng(77)
    cases = [(ref.glue_all(W.GLUE10), W.load_image("glue10")), ]
    one = ref.compile(rb"timeout$|^GET |error", "")
    cases.append((one, one.save()))
    every = ref.compile(rb".*", "")
    cases.append((every, every.save()))
    for sc_ref, image in cases:
        sc = P.Scanner(image, cuda_device)
        for ending in (b"\n", b""):
            text, lines = _text_of(rng, 3000, ending)
            corpus, o = csr(lines)
            want = sc_ref.run(corpus, o, variant=0)
            for shift in (0, 1, 7, 16, 31):
                buf = torch.zeros(len(text) + 64, dtype=torch.uint8, device="cuda:0")
                view = buf[shift: shift + len(text)]
                view.copy_(torch.from_numpy(np.frombuffer(text, np.uint8).copy()))
                batch = P.Batch.from_text(view)
                assert batch.n == len(lines)
                for max_hot in (255, 6, 2):
                    sc.set_max_hot(max_hot)
                    for variant in (1, 2):
                        sc.set_variant(variant)
                        r = P.Runner(sc).Begin().Run(batch).End()
                        assert (r.Matches().astype(np.uint8) == want[0]).all(), (shift, max_hot, variant, ending)
                        assert (r.AcceptMasks() == want[1]).all() and (r.States() == want[2]).all(), (shift, max_hot, variant, ending)
            sc.set_max_hot(255)
    # texts of a few bytes
    sc = P.Scanner(cases[1][1], cuda_device)
    for text in (b"\n", b"\n\n\n", b"error", b"error\n", b"x\nerror", b"\nGET \n", b"a" * 31 + b"\n" + b"timeout", b"a" * 32 + b"\ntimeout\n"):
        lines = text.split(b"\n")
        if text.endswith(b"\n"):
            lines = lines[:-1]
        corpus, o = csr(lines)
        want = cases[1][0].run(corpus, o, variant=0)
        batch = P.Batch.from_text(torch.from_numpy(np.frombuffer(text, np.uint8).copy()).to("cuda:0"))
        r = P.Runner(sc).Begin().Run(batch).End()
        assert batch.n == len(lines) and (r.Matches().astype(np.uint8) == want[0]).all() and (r.States() == want[2]).all(), text


def test_long_strings_split_over_a_warp(cuda_device, ref):
    """Length-ordered batches hand strings of 8 KiB and more to the split kernel: 32 lanes walk 32 pieces of one string
    from guessed states and stitch them.  Against the reference: lengths around the threshold and the piece sizes,
    every start alignment class, planted matches on piece boundaries, automata whose walks fall together (searches),
    one that needs eleven bytes to do so (a shift register) and one whose walks never do (parity of a run of a's: the
    stitching degenerates to the serial walk and must still be exact), absorbing accept states (NoExit short cut),
    small hot sets (pieces that leave the hot rows), plain and filtered walks, short strings in the same batch."""
    import torch
    import pire_b200 as P
    from pire_b200 import workloads as W
    rng = np.random.default_rng(4242)
    lens = [8191, 8192, 8193, 8192 + 31, 8192 + 32, 9000, 12345, 16384, 20000, 32 * 1024 - 1, 32 * 1024, 40000, 65536, 70001, 131072 + 17]
    cases = [
        (ref.glue_all(W.GLUE10), W.load_image("glue10"), bytes(range(0x20, 0x7F)), [p.lstrip(b"^$") for p in W.GLUE10_PLANTS]),
        (None, (rb"(a|b)*a(a|b)(a|b)(a|b)(a|b)(a|b)(a|b)(a|b)(a|b)(a|b)(a|b)", "n"), b"ab", [b"a"]),
        (None, (rb"^(aa)*$", "n"), b"a", [b"a"]),
        (None, (rb"timeout$|^GET |error", ""), b"abcdefg hijk", [b"error", b"timeout", b"GET "]),
    ]
    for sc_ref, image, alphabet, plants in cases:
        if sc_ref is None:
            sc_ref = ref.compile(*image)
            image = sc_ref.save()
        sc = P.Scanner(image, cuda_device)
        strs = []
        for k, n in enumerate(lens):
            row = rng.choice(np.frombuffer(alphabet, np.uint8), size=n)
            if k % 3 != 2:
                for j in range(1 + k % 4):
                    lit = np.frombuffer(plants[(k + j) % len(plants)], np.uint8)
                    piece = (n // 32) // 32 * 32                        # a piece of the split is about this long
                    at = min(n - len(lit), max(0, (j + 1) * piece * (3 + k % 5) - len(lit) // 2))
                    row[at:at + len(lit)] = lit                          # straddles a piece boundary
            strs.append(bytes(row))
            strs.append(bytes(rng.choice(np.frombuffer(alphabet, np.uint8), size=int(rng.integers(0, 300)))))
        strs += [b"", plants[0], bytes(rng.choice(np.frombuffer(alphabet, np.uint8), size=8192 * 3))]
        # odd gaps between the strings put them on every alignment
        pad = [bytes(int(rng.integers(0, 32))) for _ in strs]
        blob = b"".join(p_ + s_ for p_, s_ in zip(pad, strs))
        offs = np.zeros(2 * len(strs) + 1, np.int64)
        np.cumsum([len(x) for pair in zip(pad, strs) for x in pair], out=offs[1:])
        corpus, o = csr([x for pair in zip(pad, strs) for x in pair])
        want = sc_ref.run(corpus, o, variant=0)
        dev = torch.from_numpy(np.frombuffer(blob + bytes(64), np.uint8).copy()).to("cuda:0")
        batch = P.Batch(dev, torch.from_numpy(offs).to("cuda:0"), n=len(offs) - 1)
        batch.bin_by_length()
        for max_hot in (255, 6, 2):
            sc.set_max_hot(max_hot)
            for variant in (1, 2, 4):
                sc.set_variant(variant)
                for begin, end in ((True, True), (False, False)):
                    r = P.Runner(sc)
                    if begin:
                        r = r.Begin()
                    r = r.Run(batch)
                    if end:
                        r = r.End()
                    w = want if (begin and end) else sc_ref.run(corpus, o, variant=0, begin=begin, end=end)
                    assert (r.Matches().astype(np.uint8) == w[0]).all(), (image[:8], max_hot, variant, begin, end)
                    assert (r.AcceptMasks() == w[1]).all() and (r.States() == w[2]).all(), (image[:8], max_hot, variant, begin, end)


def test_half_final_counts_golden(cuda_device):
    """pire_gpu_count_batch against the numbers of count_ut.cpp HalfFinal@553 (committed fixtures)."""
    import pire_b200 as P
    from conftest import GOLDEN_COUNTS
    for case in GOLDEN_COUNTS:
        for max_hot, mode in ((255, 0), (255, 1), (255, 2), (255, 3), (3, 1), (3, 2), (3, 3)):
            sc = P.Scanner(case.image, cuda_device)
            sc.set_max_hot(max_hot)
            sc.set_count_mode(mode)           # accept lists / packed increments / packed on every chunk
            res = P.HalfFinalCount(sc, P.Batch.from_strings(case.strings))
            assert res.counts[0].tolist() == case.expect, (case, max_hot, mode)
            assert res.counts.tolist() == case.counts and res.final.astype(int).tolist() == case.final, (case, max_hot, mode)
            assert res.AcceptedRegexps(0) == [r for r, c in enumerate(case.expect) if c]
        if case.single:
            image, want, fin = case.single
            res = P.HalfFinalCount(P.Scanner(image, cuda_device), P.Batch.from_strings(case.strings))
            assert res.counts[:, 0].tolist() == want and res.final.astype(int).tolist() == fin


def test_half_final_counts_vs_reference(cuda_device, ref):
    """Random text, long and short strings, all mark combinations, hot sets small enough to force cold
    states, more than four glued counters (the register / global counter split), fixed-length batches."""
    import torch
    import pire_b200 as P
    from refpire import oracle_count
    rng = np.random.default_rng(44)
    alphabet = np.frombuffer(b"abcde z", np.uint8)
    for pat in (b"ab+", b"(ab)+", b"ab+c|b", rb"a\w+c|b", b"[a-c]+", rb"(\w\w)+"):
        scs = [ref.compile_half_final(pat, "un", mode) for mode in (1, 2, 3, 4, 5)]
        glued = scs[0]
        for sc in scs[1:] + [scs[3], scs[1]]:               # 7 counters
            glued = ref.glue_half_final(glued, sc)
        assert not glued.empty and glued.regexps == 7
        strs = [bytes(rng.choice(alphabet, size=int(k))) for k in rng.integers(0, 300, size=600)]
        strs += [bytes(rng.choice(alphabet, size=int(k))) for k in (4096, 5000, 15, 16, 17, 31, 32, 33)]
        corpus, offs = csr(strs)
        batch = P.Batch.from_strings(strs)
        for ref_sc in (glued, scs[3], ref.compile_half_final(pat, "u", 0)):
            image = ref_sc.save()
            orc = Oracle(image)
            for max_hot in (255, 2):
                sc = P.Scanner(image, cuda_device)
                sc.set_max_hot(max_hot)
                for begin, end in ((True, True), (False, False), (True, False), (False, True)):
                    want, wfin = ref_sc.count(corpus, offs, begin=begin, end=end)
                    for mode in (1, 2, 3):
                        sc.set_count_mode(mode)
                        res = P.HalfFinalCount(sc, batch, begin=begin, end=end)
                        assert (res.counts == want).all(), (pat, max_hot, mode, begin, end, np.argwhere(res.counts != want)[:4])
                        assert (res.final == wfin.astype(bool)).all()
                    got, _ = oracle_count(orc, corpus, offs, begin=begin, end=end)
                    assert (got == want).all()
        # 21 counters: too many for the packed form, the accept lists are walked whatever the mode says
        many = glued
        for _ in range(2):
            many = ref.glue_half_final(many, glued)
        assert many.regexps == 21
        sc = P.Scanner(many.save(), cuda_device)
        want, _ = many.count(corpus, offs)
        for mode in (0, 2):
            sc.set_count_mode(mode)
            assert (P.HalfFinalCount(sc, batch).counts == want).all()
        # long strings: the 16-bit stage of the packed counters is flushed before it can wrap
        long_strs = [bytes(rng.choice(np.frombuffer(b"ab", np.uint8), size=int(k))) for k in (70000, 66000, 1 << 17, 5)]
        lc, lo = csr(long_strs)
        want, _ = glued.count(lc, lo)
        sc = P.Scanner(glued.save(), cuda_device)
        for mode in (2, 3):
            sc.set_count_mode(mode)
            assert (P.HalfFinalCount(sc, P.Batch.from_strings(long_strs)).counts == want).all(), (pat, mode)
    # fixed-length strings, tuned hot rows
    ref_sc = ref.compile_half_final(b"ab+c|b", "un", 4)
    sc = P.Scanner(ref_sc.save(), cuda_device)
    host = rng.choice(np.frombuffer(b"abc ", np.uint8), size=(6000, 96)).reshape(-1)
    batch = P.Batch(torch.from_numpy(host).to("cuda:0"), fixed_len=96, n=6000)
    want, wfin = ref_sc.count(host, fixed_len=96, n=6000)
    for tuned in (False, True):
        if tuned:
            sc.Tune(batch, 6000)           # also measures how often final states are entered (AUTO -> every chunk)
        res = P.HalfFinalCount(sc, batch)
        assert (res.counts == want).all() and (res.final == wfin.astype(bool)).all()


def test_half_final_scanner_matches_like_scanner(cuda_device, ref):
    """A HalfFinalScanner image through the ordinary run entry point: pire_ut.cpp runs its Matches() vectors on
    HalfFinalScanner too (TestGlue@701-704, Serialization@576-579); Final() must agree with the reference's."""
    import pire_b200 as P
    rng = np.random.default_rng(45)
    for pat, opts in ((b"regexp", ""), (b"a.*b", ""), (b"^abc$", ""), (b"hello\\s+w.+d$", "")):
        ref_sc = ref.compile_half_final(pat, opts, 0)
        strs = [b"regexp", b"regxp", b"regexp t", b"abc", b"xabcx", b"hello  world", b"a--b", b""]
        strs += [bytes(rng.choice(np.frombuffer(b"abcreg xp", np.uint8), size=int(k))) for k in rng.integers(0, 80, size=200)]
        corpus, offs = csr(strs)
        _, wfin = ref_sc.count(corpus, offs)
        sc = P.Scanner(ref_sc.save(), cuda_device)
        final, _, _ = gpu_run(sc, strs)
        assert (final == wfin).all(), pat


def test_suffix_scans_golden(cuda_device):
    """Pire::LongestSuffix / ShortestSuffix on the device: PrefixSuffix@278 and, like ScanBoundaries@469-471, the
    prefix table through the suffix scans on the reversed text."""
    import pire_b200 as P
    from conftest import GOLDEN_PREFIX, GOLDEN_SUFFIX
    for pat, image, texts, shortest, longest in GOLDEN_SUFFIX:
        sc = P.Scanner(image, cuda_device)
        batch = P.Batch.from_strings(texts)
        assert P.ShortestSuffix(sc, batch).tolist() == shortest and P.LongestSuffix(sc, batch).tolist() == longest
    for pat, image, text, shortest, longest in GOLDEN_PREFIX:
        sc = P.Scanner(image, cuda_device)
        batch = P.Batch.from_strings([b"junk", text[::-1], b"", b"tail" + text[::-1]])
        s = P.ShortestSuffix(sc, batch)
        l = P.LongestSuffix(sc, batch)
        assert s[1] == shortest and l[1] == longest, (pat, s.tolist(), l.tolist())


def test_suffix_scans_vs_reference(cuda_device, ref):
    """Random text, every mark combination (incl. ShortestSuffix stepping BeginMark from where it stopped), every
    start alignment through ragged neighbours, hot sets small enough to force cold states; fixed-length batch."""
    import torch
    import pire_b200 as P
    from refpire import oracle_suffix
    rng = np.random.default_rng(34)
    for pat, opts in [(b"a+b", "n"), (b"a+b", "nr"), (b"foo.*bar", "n"), (rb"[0-9]+\.[0-9]+", "r"), (b"x*", "n"), (b"(ab)*c", "nr"),
                      (b".*z", "n"), (b"^ab", ""), (b"ab$", "r"), (b"[^x]*", "n")]:
        sc_ref = ref.compile(pat, opts)
        image = sc_ref.save()
        orc = Oracle(image)
        strs = [bytes(rng.choice(np.frombuffer(b"abfoxz019. r", np.uint8), size=int(n))) for n in rng.integers(0, 400, size=700)]
        strs += [b"a" * n for n in (15, 16, 17, 31, 32, 33, 64)] + [b"ab" * 40 + b"z" * k for k in range(0, 20)]
        corpus, offs = csr(strs)
        batch = P.Batch.from_strings(strs)
        for max_hot in (255, 2):
            sc = P.Scanner(image, cuda_device)
            sc.set_max_hot(max_hot)
            for te in (False, True):
                for tb in (False, True):
                    for shortest in (False, True):
                        fn = P.ShortestSuffix if shortest else P.LongestSuffix
                        got = fn(sc, batch, throughEndMark=te, throughBeginMark=tb)
                        want = sc_ref.suffix(corpus, offs, shortest=shortest, through_end=te, through_begin=tb, variant=2)
                        assert (got == want).all(), (pat, opts, max_hot, te, tb, shortest, np.nonzero(got != want)[0][:5])
                        assert (got == oracle_suffix(orc, corpus, offs, shortest=shortest, through_end=te, through_begin=tb)).all()
    sc_ref = ref.compile(b"ab+c", "r")
    sc = P.Scanner(sc_ref.save(), cuda_device)
    host = rng.choice(np.frombuffer(b"abc ", np.uint8), size=(5000, 72)).reshape(-1)
    batch = P.Batch(torch.from_numpy(host).to("cuda:0"), fixed_len=72, n=5000)
    for shortest in (False, True):
        got = (P.ShortestSuffix if shortest else P.LongestSuffix)(sc, batch)
        assert (got == sc_ref.suffix(host, fixed_len=72, n=5000, shortest=shortest, variant=2)).all()


def test_longest_prefix_vs_default_scanner_enumerated(cuda_device, ref):
    """run.h:277-292 through the default Scanner's skip loop (multi.h:966-989): the ExitMasks fast-forward does not
    call the predicate over the 16-byte words it jumps, so LongestPrefix comes out SHORT exactly when the string ends
    on a 16-byte boundary of the host address space after at least one whole aligned word walked in a final state
    with at most two exit bytes -- it then reports only the unaligned head.  The device (like the NoMask scanners)
    has no such artefact.  This test pins WHERE the two reference scanners differ, for every start alignment and
    length, and that the device agrees with the byte-by-byte answer everywhere."""
    import pire_b200 as P

    def aligned(nbytes):
        raw = np.zeros(nbytes + 64, np.uint8)
        off = (-raw.ctypes.data) % 64
        return raw[off:off + nbytes]

    cases = [(rb"[^x]*", b"a", True), (rb"a*b?", b"a", False), (rb"(ab)*", b"ab", False), (rb"[a-c]+x?", b"abc", False)]
    for pat, fill, has_artefact in cases:
        sc_ref = ref.compile(pat, "n")
        sc = P.Scanner(sc_ref.save(), cuda_device)
        strings, shifts = [], []
        differing = set()
        for shift in range(16):
            for ln in range(0, 70):
                buf = aligned(256)
                buf[:] = ord("z")
                text = (fill * 100)[:ln]
                if ln:
                    buf[shift:shift + ln] = np.frombuffer(text, np.uint8)
                offs = np.array([shift, shift + ln], np.uint64)
                default = int(sc_ref.prefix(buf, offs, variant=0)[0])
                nomask = int(sc_ref.prefix(buf, offs, variant=2)[0])
                if default != nomask:
                    differing.add((shift, ln))
                    head = (-shift) % 16
                    assert default == (head if head else 0) and default < nomask      # only the unaligned head is seen
                strings.append(text)
                shifts.append((shift, ln, nomask))
        predicted = set()
        for shift in range(16):
            for ln in range(0, 70):
                end, first = shift + ln, (shift + 15) // 16 * 16
                if has_artefact and end % 16 == 0 and end >= first + 16:
                    predicted.add((shift, ln))
        assert differing == predicted, (pat, sorted(differing ^ predicted)[:8])
        # the device: every string at every device alignment (CSR, back to back) equals the byte-by-byte reference
        got = P.LongestPrefix(sc, P.Batch.from_strings(strings))
        assert got.tolist() == [w for _, _, w in shifts], pat


def test_accept_sets_beyond_32_regexps(cuda_device, ref):
    """multi.h:149-158 returns accept lists of any length; the scan kernels' mask holds ids 0..31.  Forty end-anchored
    literals glued into one scanner: every id, also 32..39, must come back through pire_gpu_accept_sets."""
    import ctypes as C
    import torch
    import pire_b200 as P
    from pire_b200 import _native as N
    pats = [(("[a-z]*w%02d" % k).encode(), "n") for k in range(40)]       # not surrounded: lowercase text ending in wNN
    sc_ref = ref.glue_all(pats)
    sc = P.Scanner(sc_ref.save(), cuda_device)
    assert sc.RegexpsCount() == 40 and N.lib.pire_gpu_accept_words(sc._h) == 2
    rng = np.random.default_rng(40)
    n, length = 4096, 64
    host = rng.integers(0x61, 0x7B, size=(n, length), dtype=np.uint8)
    want_ids = []
    for i in range(n):
        if i % 3:
            k = int(rng.integers(0, 40))
            host[i, -3:] = np.frombuffer(b"w%02d" % k, np.uint8)
            want_ids.append([k])
        else:
            host[i, int(rng.integers(0, length))] = ord("!")
            want_ids.append([])
    dev = torch.from_numpy(np.ascontiguousarray(host).reshape(-1)).to("cuda:0")
    batch = P.Batch(dev, fixed_len=length, n=n)
    f_ref, m_ref, s_ref = sc_ref.run(np.ascontiguousarray(host).reshape(-1), fixed_len=length, n=n, begin=False, end=False)
    assert [sc_ref.accepted(int(st)) for st in s_ref[:64]] == want_ids[:64]      # the reference agrees with the construction
    for variant in (1, 2, 4, 5):
        sc.set_variant(variant)
        r = P.Runner(sc).Run(batch)              # patterns without Surround() do not consume the marks (run.h:396-400)
        assert (r.States() == s_ref).all() and (r.AcceptMasks() == m_ref).all()
        states = torch.from_numpy(r.States().astype(np.int32)).to("cuda:0")
        sets = torch.zeros((n, 2), dtype=torch.int32, device="cuda:0")
        N.check(N.lib.pire_gpu_accept_sets(sc._h, states.data_ptr(), n, sets.data_ptr(), None), "pire_gpu_accept_sets")
        sets = sets.cpu().numpy().view(np.uint32)
        masks = r.AcceptMasks()
        for i in range(n):
            ids = [k for k in range(40) if (int(sets[i, k // 32]) >> (k % 32)) & 1]
            assert ids == want_ids[i], (variant, i, ids, want_ids[i])
            assert int(masks[i]) == int(sets[i, 0])                              # the 32-bit mask is the first word
            assert ids == sc.AcceptedRegexps(int(r.States()[i]))                 # and the host accessor agrees
        assert (r.Matches() == np.array([bool(w) for w in want_ids])).all()
    # a state index outside the scanner yields an empty set
    bad = torch.tensor([sc.Size() + 5], dtype=torch.int32, device="cuda:0")
    out = torch.full((1, 2), -1, dtype=torch.int32, device="cuda:0")
    N.check(N.lib.pire_gpu_accept_sets(sc._h, bad.data_ptr(), 1, out.data_ptr(), None), "pire_gpu_accept_sets")
    assert out.cpu().tolist() == [[0, 0]]


def test_host_entry_streams_chunks(cuda_device, ref, monkeypatch):
    """pire_gpu_run_batch_host with pageable buffers (numpy): chunks of 1 MiB force a dozen trips round the three-slot
    ring for a fixed-length and a ragged CSR batch; two threads on one handle run concurrently; bad offsets are
    refused.  Results equal the reference."""
    import threading
    import pire_b200 as P
    from pire_b200 import _native as N
    from pire_b200 import workloads as W
    monkeypatch.setenv("PIRE_B200_HOST_CHUNK_MB", "1")
    sc_ref = ref.glue_all(W.GLUE10)
    sc = P.Scanner(W.load_image("glue10"), cuda_device)
    n = 12 * 1024 + 37
    spec = W.SynthSpec(n, 1024, plants=W.GLUE10_PLANTS)
    host = spec.host_sample(0, n)                                  # pageable
    f_ref, m_ref, s_ref = sc_ref.run(host, fixed_len=1024, n=n, threads=8)
    bits, masks, states = sc.run_batch_host(host, fixed_len=1024, n=n, want_masks=True, want_states=True)
    assert (np.unpackbits(bits.view(np.uint8), bitorder="little")[:n] == f_ref).all()
    assert (masks == m_ref).all() and (states == s_ref).all()
    # ragged CSR incl. empty strings, a string longer than a chunk, lengths not multiples of anything
    rng = np.random.default_rng(8)
    lens = np.concatenate([rng.integers(0, 3000, size=5000), [0, 0, 3 << 20, 1, 17]])
    rng.shuffle(lens)
    total = int(lens.sum())
    corpus = rng.integers(0x20, 0x7F, size=total, dtype=np.uint8)
    offs = np.zeros(len(lens) + 1, np.uint64)
    np.cumsum(lens, out=offs[1:])
    for k in range(0, len(lens), 7):                               # plant a few hits
        if lens[k] >= 8:
            corpus[int(offs[k + 1]) - 5:int(offs[k + 1])] = np.frombuffer(b"error", np.uint8)
    f2, m2, s2 = sc_ref.run(corpus, offs, threads=8)
    bits, masks, states = sc.run_batch_host(corpus, offsets=offs, want_masks=True, want_states=True)
    assert (np.unpackbits(bits.view(np.uint8), bitorder="little")[:len(lens)] == f2).all()
    assert (masks == m2).all() and (states == s2).all()
    assert int(f2.sum()) > 100
    # two threads, one handle
    results = [None, None]

    def work(k):
        results[k] = sc.run_batch_host(host, fixed_len=1024, n=n, want_masks=True)
    ts = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for b, m, _ in results:
        assert (np.unpackbits(b.view(np.uint8), bitorder="little")[:n] == f_ref).all() and (m == m_ref).all()
    # refused: offsets that step back, offsets past the buffer, n * fixed_len past the buffer
    bad = offs.copy()
    bad[10], bad[11] = bad[11], bad[10]
    with pytest.raises(P.PireGpuError):
        sc.run_batch_host(corpus, offsets=bad)
    with pytest.raises(P.PireGpuError):
        sc.run_batch_host(corpus[: total // 2], offsets=offs)
    with pytest.raises(P.PireGpuError):
        sc.run_batch_host(host[:4096], fixed_len=1024, n=5)


@pytest.mark.parametrize("length", [32, 160, 1024])
def test_uniform_bodies_of_prefix_and_count(length, cuda_device, ref, monkeypatch):
    """Fixed-length, 32-byte aligned batches take the register-streaming bodies of PrefixKernel / CountKernel (no
    staging ring).  Every mark combination, longest and shortest, a pattern with dead states, all counting modes:
    equal to the reference and to the ring path on the same bytes."""
    import torch
    import pire_b200 as P
    rng = np.random.default_rng(1000 + length)
    n = 3000 + 11
    host = rng.choice(np.frombuffer(b"abcx 01.", np.uint8), size=(n, length))
    host[::5, : min(length, 24)] = np.frombuffer((b"ab" * 12)[: min(length, 24)], np.uint8)
    host = np.ascontiguousarray(host).reshape(-1)
    dev = torch.from_numpy(host).to("cuda:0")
    batch = P.Batch(dev, fixed_len=length, n=n)
    for pat, opts in [(b"(ab)*c?", "n"), (b"a+b", ""), (rb"[0-9]+\.[0-9]+", ""), (b"[^x]*", "n")]:
        sc_ref = ref.compile(pat, opts)
        sc = P.Scanner(sc_ref.save(), cuda_device)
        for tb in (False, True):
            for te in (False, True):
                for shortest in (False, True):
                    fn = P.ShortestPrefix if shortest else P.LongestPrefix
                    want = sc_ref.prefix(host, fixed_len=length, n=n, shortest=shortest, through_begin=tb, through_end=te, variant=2)
                    monkeypatch.delenv("PIRE_B200_NO_UNIFORM_BODY", raising=False)
                    got = fn(sc, batch, throughBeginMark=tb, throughEndMark=te)
                    monkeypatch.setenv("PIRE_B200_NO_UNIFORM_BODY", "1")
                    ring = fn(sc, batch, throughBeginMark=tb, throughEndMark=te)
                    assert (got == want).all() and (ring == want).all(), (pat, tb, te, shortest)
    monkeypatch.delenv("PIRE_B200_NO_UNIFORM_BODY", raising=False)
    for pat in (b"ab", b"[ab]+", b"a.*b|c"):
        hf = ref.compile_half_final(pat, "n", 0)
        sc = P.Scanner(hf.save(), cuda_device)
        for begin in (True, False):
            for end in (True, False):
                want, wfin = hf.count(host, fixed_len=length, n=n, begin=begin, end=end)
                for mode in (1, 2, 3):
                    sc.set_count_mode(mode)
                    res = P.HalfFinalCount(sc, batch, begin=begin, end=end)
                    assert (res.counts == want).all() and (res.final == wfin.astype(bool)).all(), (pat, begin, end, mode)
