"""The reference's recorded answers, for the tests that compare with it (TEST INFRASTRUCTURE).

The reference (oracle/_ref, compiled from the original project's sources by oracle/build_ref.sh) is not part of this
repository, so the tests that compare with it read its answers from tests/golden/reference_answers.json.xz:

* every scanner the reference compiled or glued for those tests, as its Scanner::Save() image with Size(),
  RegexpsCount() and Empty() -- or the error it raised;
* for every test, one digest over the questions it put to the reference (the scanner, the arguments, the bytes
  scanned) and the reference's answers, in the order asked.

``GoldenRef`` has the face of refpire.Ref.  Its scanners answer run / prefix / suffix / count through the oracle port
(oracle/pire_oracle.c) over the recorded image; the few answers in which the reference and the port differ (prefix
scans through the default Scanner, whose ExitMasks skip depends on the host address) and the accept lists, which the
port does not compute, are stored as they are.  When a test ends, the digest of what it asked and was told must equal
the recorded one: the port answered as the reference did, on the same bytes.

With PIRE_REF_RECORD=<file> the real reference answers instead (needs oracle/_ref), and the recording, merged into
the committed one, is written to <file> after every test:

    PIRE_REF_RECORD=/tmp/answers.json.xz python -m pytest tests/test_oracle.py tests/test_gpu_parity.py
    cp /tmp/answers.json.xz tests/golden/reference_answers.json.xz
"""
import hashlib
import json
import lzma
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from refpire import Oracle, oracle_count, oracle_prefix, oracle_suffix

HERE = os.path.dirname(os.path.abspath(__file__))
ANSWERS = os.path.join(HERE, "golden", "reference_answers.json.xz")
DATA = os.path.join(os.path.dirname(HERE), "pire_b200", "data")
STORED_MAX = 4096          # answer elements that may be stored as they are (the rest must come from the port)


class MissingAnswer(LookupError):
    pass


class Store:
    """The recording: images by content hash, scanner questions, per-test digests."""

    def __init__(self, path=ANSWERS):
        d = {}
        if os.path.exists(path):
            with open(path, "rb") as f:
                d = json.loads(lzma.decompress(f.read()))
        self.images = d.get("images", {})          # sha1 -> {"meta": {...}, "hex": image} or {"meta": {...}, "data": name}
        self.scanners = d.get("scanners", {})      # question -> sha1 or {"error": message}
        self.tests = d.get("tests", {})            # test id -> {"questions": n, "digest": hex, "stored": {index: answer}}
        self._decoded = {}
        self._data = None

    def image(self, sha):
        if sha not in self._decoded:
            e = self.images[sha]
            if "data" in e:
                with open(os.path.join(DATA, e["data"] + ".pire.xz"), "rb") as f:
                    img = lzma.decompress(f.read())
            else:
                img = bytes.fromhex(e["hex"])
            assert hashlib.sha1(img).hexdigest() == sha
            self._decoded[sha] = img
        return self._decoded[sha]

    def put_image(self, image, meta):
        sha = hashlib.sha1(image).hexdigest()
        if self._data is None:          # the images shipped under pire_b200/data are named, not copied
            self._data = {}
            for name in sorted(os.listdir(DATA)):
                with open(os.path.join(DATA, name), "rb") as f:
                    self._data[hashlib.sha1(lzma.decompress(f.read())).hexdigest()] = name[:-len(".pire.xz")]
        if sha not in self.images:
            self.images[sha] = {"meta": meta, "data": self._data[sha]} if sha in self._data else {"meta": meta, "hex": image.hex()}
            self._decoded[sha] = image
        return sha

    def save(self, path):
        used = {v for v in self.scanners.values() if isinstance(v, str)}
        d = {"note": "answers of the reference (oracle/_ref) recorded by tests/refgolden.py; see its docstring",
             "scanners": dict(sorted(self.scanners.items())), "tests": dict(sorted(self.tests.items())),
             "images": {k: v for k, v in sorted(self.images.items()) if k in used}}
        with open(path, "wb") as f:
            f.write(lzma.compress(json.dumps(d, indent=0).encode(), preset=9 | lzma.PRESET_EXTREME))


_STORE = None


def store():
    global _STORE
    if _STORE is None:
        _STORE = Store()
    return _STORE


def _n_of(corpus, offsets, fixed_len, n):
    if offsets is not None:
        return len(offsets) - 1 if n is None else n
    if n is None:
        return len(corpus) // fixed_len if fixed_len else 0
    return n


def _inputs(corpus, offsets, fixed_len, n):
    """The bytes a batch call reads, as (corpus, offsets) arrays to hash."""
    corpus = np.ascontiguousarray(corpus, dtype=np.uint8)
    if offsets is not None:
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)[: n + 1]
        return corpus[: int(offsets[-1]) if n else 0], offsets
    return corpus[: n * fixed_len], None


def _answer(values):
    return tuple(np.ascontiguousarray(v) for v in values)


def _port_run(orc, corpus, offsets, fixed_len, n, begin, end):
    """The port over slices of the batch on a few threads (the C call drops the GIL)."""
    final, mask, state = np.zeros(n, np.uint8), np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    parts = max(1, min(os.cpu_count() or 1, 16, n // 4096))

    def part(k):
        lo, hi = n * k // parts, n * (k + 1) // parts
        if offsets is not None:
            out = orc.run(corpus, offsets[lo:hi + 1], n=hi - lo, begin=begin, end=end, shortcuts=True)
        else:
            out = orc.run(corpus[lo * fixed_len:hi * fixed_len], fixed_len=fixed_len, n=hi - lo, begin=begin, end=end, shortcuts=True)
        final[lo:hi], mask[lo:hi], state[lo:hi] = out
    with ThreadPoolExecutor(parts) as pool:
        list(pool.map(part, range(parts)))
    return final, mask, state


class _Scanner:
    """A scanner the reference made: its image, and (recording) the reference's own handle."""

    def __init__(self, owner, sha, real=None):
        self._owner, self.sha, self._real = owner, sha, real
        self._orc = None
        meta = owner.store.images[sha]["meta"]
        self.size, self.regexps, self.empty = meta["size"], meta["regexps"], bool(meta["empty"])

    def save(self):
        return self._owner.store.image(self.sha)

    def _port(self):
        if self._orc is None:
            self._orc = Oracle(self.save())
        return self._orc

    def run(self, corpus, offsets=None, fixed_len=0, n=None, begin=True, end=True, variant=1, threads=1,
            want=("final", "mask", "state")):
        """Runner(sc).[Begin()].Run(str).[End()] per string: (final u8, mask u32, state u32), None where not wanted."""
        n = _n_of(corpus, offsets, fixed_len, n)
        corpus, offsets = _inputs(corpus, offsets, fixed_len, n)
        args = dict(fixed_len=fixed_len, n=n, begin=begin, end=end, variant=variant)
        out = self._owner.ask(
            "run", self, args, (corpus, offsets),
            lambda: _port_run(self._port(), corpus, offsets, fixed_len, n, begin, end),
            lambda: self._real.run(corpus, offsets, fixed_len=fixed_len, n=n, begin=begin, end=end, variant=variant,
                                   threads=self._owner.threads()))
        return tuple(a if k in want else None for k, a in zip(("final", "mask", "state"), out))

    def prefix(self, corpus, offsets=None, fixed_len=0, n=None, shortest=False, through_begin=False, through_end=False,
               variant=2):
        n = _n_of(corpus, offsets, fixed_len, n)
        corpus, offsets = _inputs(corpus, offsets, fixed_len, n)
        args = dict(fixed_len=fixed_len, n=n, shortest=shortest, through_begin=through_begin, through_end=through_end, variant=variant)
        return self._owner.ask(
            "prefix", self, args, (corpus, offsets),
            lambda: (oracle_prefix(self._port(), corpus, offsets, fixed_len, n, shortest, through_begin, through_end),),
            lambda: (self._real.prefix(corpus, offsets, fixed_len, n, shortest, through_begin, through_end, variant),))[0]

    def suffix(self, corpus, offsets=None, fixed_len=0, n=None, shortest=False, through_end=False, through_begin=False,
               variant=2):
        n = _n_of(corpus, offsets, fixed_len, n)
        corpus, offsets = _inputs(corpus, offsets, fixed_len, n)
        args = dict(fixed_len=fixed_len, n=n, shortest=shortest, through_end=through_end, through_begin=through_begin, variant=variant)
        return self._owner.ask(
            "suffix", self, args, (corpus, offsets),
            lambda: (oracle_suffix(self._port(), corpus, offsets, fixed_len, n, shortest, through_end, through_begin),),
            lambda: (self._real.suffix(corpus, offsets, fixed_len, n, shortest, through_end, through_begin, variant),))[0]

    def count(self, corpus, offsets=None, fixed_len=0, n=None, begin=True, end=True, threads=1):
        """HalfFinalScanner counting per string: (counts[n, regexps] u32, final[n] u8)."""
        n = _n_of(corpus, offsets, fixed_len, n)
        corpus, offsets = _inputs(corpus, offsets, fixed_len, n)
        args = dict(fixed_len=fixed_len, n=n, begin=begin, end=end)
        return self._owner.ask(
            "count", self, args, (corpus, offsets),
            lambda: oracle_count(self._port(), corpus, offsets, fixed_len, n, begin, end),
            lambda: self._real.count(corpus, offsets, fixed_len, n, begin, end, self._owner.threads()))

    def accepted(self, state):
        """AcceptedRegexps(state): the port does not compute accept lists, so they are stored."""
        out = self._owner.ask("accepted", self, dict(state=int(state)), (), None,
                              lambda: (np.array(self._real.accepted(state), np.int64),))
        return [int(x) for x in out[0]]


class GoldenRef:
    """refpire.Ref's face over the recording (or, recording, over the real reference) for one test."""

    def __init__(self, test_id, record_to=None):
        self.test_id, self.record_to = test_id, record_to
        self.store = store()
        self.real = None
        if record_to:
            import refpire
            self.real = refpire.Ref()
        self._hash = hashlib.sha1()
        self._asked = 0
        self._stored = {}
        want = self.store.tests.get(test_id)
        if not record_to and want is None:
            raise MissingAnswer("no recorded reference answers for %s: record them with PIRE_REF_RECORD (tests/refgolden.py)" % test_id)
        self._want = want

    # --- scanners ----------------------------------------------------------------------------------------------------
    def _scanner(self, question, make):
        if self.real is not None:
            try:
                sc = make()
            except ValueError as e:
                self.store.scanners[question] = {"error": str(e)}
                raise
            meta = {"size": int(sc.size), "regexps": int(sc.regexps), "empty": bool(sc.empty)}
            sha = self.store.put_image(sc.save(), meta)
            self.store.scanners[question] = sha
            return _Scanner(self, sha, sc)
        got = self.store.scanners.get(question)
        if got is None:
            raise MissingAnswer("no recorded reference scanner for %s: record it with PIRE_REF_RECORD (tests/refgolden.py)" % question)
        if isinstance(got, dict):
            raise ValueError(got["error"])
        return _Scanner(self, got)

    @staticmethod
    def _pat(pattern):
        return (pattern.encode("latin-1") if isinstance(pattern, str) else bytes(pattern)).hex()

    def compile(self, pattern, opts=""):
        return self._scanner("compile %s %s" % (self._pat(pattern), opts), lambda: self.real.compile(pattern, opts))

    def glue(self, a, b, max_size=0):
        return self._scanner("glue %s %s %d" % (a.sha, b.sha, max_size), lambda: self.real.glue(a._real, b._real, max_size))

    def glue_all(self, patterns):
        """tools/bench/bench.cpp:108-132: glue left to right (only the result is recorded)."""
        key = " ".join("%s/%s" % (self._pat(p), o) for p, o in patterns)
        return self._scanner("glue_all " + key, lambda: self.real.glue_all(patterns))

    def compile_half_final(self, pattern, opts="", mode=0):
        return self._scanner("compile_half_final %s %s %d" % (self._pat(pattern), opts, mode),
                             lambda: self.real.compile_half_final(pattern, opts, mode))

    def glue_half_final(self, a, b, max_size=0):
        return self._scanner("glue_half_final %s %s %d" % (a.sha, b.sha, max_size),
                             lambda: self.real.glue_half_final(a._real, b._real, max_size))

    def hardware_threads(self):
        return self.threads()

    @staticmethod
    def threads():
        return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    # --- questions ---------------------------------------------------------------------------------------------------
    def ask(self, what, sc, args, inputs, port, real):
        """One question to the reference: the stored answer, the port's, or (recording) the reference's own."""
        k = self._asked
        self._asked += 1
        if self.real is not None:
            answer = _answer(real())
            mine = _answer(port()) if port is not None else None
            if mine is None or len(mine) != len(answer) or not all(np.array_equal(a, b) for a, b in zip(answer, mine)):
                assert sum(a.size for a in answer) <= STORED_MAX, \
                    "%s: the oracle port differs from the reference on a large answer (%s %s)" % (self.test_id, what, args)
                self._stored[str(k)] = [[a.dtype.str, a.tolist()] for a in answer]
        elif self._want["stored"].get(str(k)) is not None:
            answer = tuple(np.array(v, dtype=np.dtype(t)) for t, v in self._want["stored"][str(k)])
        else:
            if port is None:
                raise MissingAnswer("%s: question %d (%s) has no stored answer" % (self.test_id, k, what))
            answer = _answer(port())
        h = self._hash
        h.update(json.dumps([k, what, sc.sha, args], sort_keys=True).encode())
        for a in inputs:
            if a is not None:
                h.update(memoryview(a).cast("B"))
        for a in answer:
            h.update(a.dtype.str.encode() + repr(a.shape).encode())
            h.update(memoryview(a).cast("B"))
        return answer

    def finish(self):
        """At the end of a test that passed: record, or check that the answers given were the reference's."""
        if self.real is not None:
            self.store.tests[self.test_id] = {"questions": self._asked, "digest": self._hash.hexdigest(), "stored": self._stored}
            self.store.save(self.record_to)
            return
        assert self._asked == self._want["questions"], "%s: %d questions to the reference, the recording has %d" % (
            self.test_id, self._asked, self._want["questions"])
        assert self._hash.hexdigest() == self._want["digest"], (
            "%s: the questions asked or the answers the oracle port gave differ from the reference's recorded ones" % self.test_id)
