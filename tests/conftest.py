import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    from tools.datafiles import inflate_data      # index files that travelled as zstd frames (tools/datafiles.py)
    inflate_data()


def read_fastx(path):
    """(names, seqs) the way kseq tokenises: name = header up to first whitespace."""
    names, seqs = [], []
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    i = 0
    while i < len(lines):
        ln = lines[i]
        if ln.startswith(b">"):
            names.append(ln[1:].split()[0].decode())
            seqs.append(lines[i + 1].strip())
            i += 2
        elif ln.startswith(b"@"):
            names.append(ln[1:].split()[0].decode())
            seqs.append(lines[i + 1].strip())
            i += 4
        else:
            i += 1
    return names, seqs


@pytest.fixture(scope="session")
def golden():
    return GOLDEN


@pytest.fixture(scope="session")
def small_index(tmp_path_factory):
    """Prefix of the `small` benchmark index (1 Mbp x 16 haplotypes): data/small when it has been built, else the same
    files built once per session without the reference (tools/synth.build_index_gpu, about a minute; needs a GPU)."""
    prefix = os.path.join(ROOT, "data", "small", "small")
    if os.path.exists(prefix + ".mab"):
        return prefix
    from tools import synth
    prefix = str(tmp_path_factory.mktemp("small") / "small")
    synth.build_index_gpu(synth.make_panel(*synth.CONFIGS["small"]), prefix, markers=True)
    return prefix


FIXTURES = {
    # name: (dir, prefix, query files, has markers)
    "toy": ("toy", "small.fa", ["simple_query.fq", "error_query.fq", "edge_query.fq"], True),
    "greedy": ("greedy", "ref.fa", ["query.fq"], False),
    "tiny": ("tiny", "tiny", ["exact.fq", "noisy.fq", "short.fq", "marked.fq"], True),
}
FLAGSETS = [("count", False, False), ("s", True, False), ("m", False, True), ("sm", True, True)]


def fixture_cases():
    for name, (d, pre, fqs, has_ma) in FIXTURES.items():
        for fq in fqs:
            for tag, sa, ma in FLAGSETS:
                if ma and not has_ma:
                    continue
                yield pytest.param(d, pre, fq, tag, sa, ma, id="%s-%s-%s" % (name, fq, tag))
