import base64
import json
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


class GoldenCase:
    def __init__(self, d):
        self.name = d["name"]
        self.patterns = [(bytes.fromhex(p), o) for p, o in d["patterns"]]
        self.image = base64.b64decode(d["image"])
        self.strings = [bytes.fromhex(s) for s in d["strings"]]
        self.final = d["final"]
        self.ids = d["ids"]
        self.state = d["state"]
        self.begin = bool(d["begin"])
        self.end = bool(d["end"])
        self.states, self.letters, self.regexps = d["states"], d["letters"], d["regexps"]

    def mask(self):
        return [sum(1 << i for i in ids if i < 32) for ids in self.ids]

    def __repr__(self):
        return "GoldenCase(%s)" % self.name


def load_golden():
    with open(os.path.join(HERE, "golden", "pire_golden.json")) as f:
        return [GoldenCase(c) for c in json.load(f)["cases"]]


def load_golden_prefix():
    with open(os.path.join(HERE, "golden", "pire_golden.json")) as f:
        return [(bytes.fromhex(c["pattern"]), base64.b64decode(c["image"]), bytes.fromhex(c["text"]), c["shortest"], c["longest"])
                for c in json.load(f)["prefix_cases"]]


class CountCase:
    """count_ut.cpp HalfFinal@553: the glue of the five HalfFinalFsm counters of one pattern."""

    def __init__(self, d):
        import lzma
        self.pattern = bytes.fromhex(d["pattern"])
        self.image = lzma.decompress(base64.b64decode(d["image_xz"]))
        self.strings = [bytes.fromhex(s) for s in d["strings"]]
        self.counts, self.final, self.expect = d["counts"], d["final"], d["expect"]
        self.states, self.regexps = d["states"], d["regexps"]
        self.single = None
        if "single" in d:
            self.single = (lzma.decompress(base64.b64decode(d["single"]["image_xz"])), d["single"]["counts"], d["single"]["final"])

    def __repr__(self):
        return "CountCase(%r, %r)" % (self.pattern, self.strings[0])


def load_golden_counts():
    with open(os.path.join(HERE, "golden", "pire_golden.json")) as f:
        return [CountCase(c) for c in json.load(f)["count_cases"]]


def load_golden_suffix():
    with open(os.path.join(HERE, "golden", "pire_golden.json")) as f:
        return [(bytes.fromhex(c["pattern"]), base64.b64decode(c["image"]), [bytes.fromhex(t) for t in c["texts"]], c["shortest"],
                 c["longest"]) for c in json.load(f)["suffix_cases"]]


GOLDEN = load_golden()
GOLDEN_SUFFIX = load_golden_suffix()
GOLDEN_COUNTS = load_golden_counts()
GOLDEN_PREFIX = load_golden_prefix()


@pytest.fixture(scope="session")
def golden():
    return GOLDEN


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    # the `ref` fixture checks its answers against the recording only for a test body that passed: a failed test has
    # already said what went wrong, and asked only part of its questions
    outcome = yield
    if call.when == "call":
        item.call_failed = outcome.get_result().failed


@pytest.fixture
def ref(request):
    """The reference's answers, as recorded in tests/golden/reference_answers.json.xz (tests/refgolden.py); with
    PIRE_REF_RECORD=<file> the real reference (oracle/_ref) answers and the recording is written to <file>."""
    import refgolden
    r = refgolden.GoldenRef("%s::%s" % (request.module.__name__, request.node.name), os.environ.get("PIRE_REF_RECORD"))
    yield r
    if not getattr(request.node, "call_failed", True):
        r.finish()


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("this test is marked gpu but no CUDA device is visible")
    return 0
