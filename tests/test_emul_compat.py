"""The htslib-compatible iterator tier (samtools_b200/csrc/host/plp_compat.cpp) on the emulation harness: the host logic of
bam_plp_* / bam_mplp_* (contig buffering, k-way merge, slab paging, hooks) against the oracle's restatement of htslib's
iterator, without a GPU.  The same cases run on the CUDA engine in tests/test_gpu_parity.py::test_htslib_compat_iterator."""
import hashlib, json, os, subprocess
import pytest
import golden_cases
from conftest import ROOT


@pytest.fixture(scope='module')
def dump_emul():
    subprocess.run([os.path.join(ROOT, 'tests', 'emul', 'build.sh')], check=True)
    return os.path.join(ROOT, 'tests', 'emul', '_build', 'plp_dump_emul')


@pytest.mark.parametrize('args,files', golden_cases.COMPAT_CASES, ids=golden_cases.COMPAT_IDS)
def test_iterator_tier_host_logic(args, files, dump_emul, oracle_bin, corpus):
    paths = [os.path.join(corpus, f) for f in files]
    got = subprocess.run([dump_emul, *args, *paths], capture_output=True)
    want = subprocess.run([oracle_bin, 'pileup-dump', *args, *paths], capture_output=True)
    assert got.returncode == 0, got.stderr[-300:]
    assert got.stdout == want.stdout
    assert len(got.stdout) > 100


@pytest.mark.parametrize('args,files', golden_cases.COMPAT_CASES[:7], ids=golden_cases.COMPAT_IDS[:7])
def test_iterator_hooks_and_kstring_insertion(args, files, dump_emul, oracle_bin, corpus):
    """-c: constructor/destructor hooks (client data carried by every entry, one destructor call per constructed read)
    and htslib's kstring signature of bam_plp_insertion; the dump itself must not change."""
    paths = [os.path.join(corpus, f) for f in files]
    got = subprocess.run([dump_emul, '-c', *args, *paths], capture_output=True)
    want = subprocess.run([oracle_bin, 'pileup-dump', *args, *paths], capture_output=True)
    assert got.returncode == 0, got.stderr[-300:]
    assert got.stdout == want.stdout
    assert b'hooks: ctor=' in got.stderr and b'bad=0' in got.stderr


PLBUF_GOLDEN = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'plbuf_dumps.json')))


@pytest.mark.parametrize('f', sorted(PLBUF_GOLDEN))
def test_reference_bam_plbuf_rides_on_the_tier(f, dump_emul, oracle_bin, corpus):
    """samtools' own bam_plbuf layer (bam_plbuf.h:32-51) drives the iterator tier through bam_plp_push / bam_plp64_next.
    plp_dump -p drives it the same way (drain after every push, NULL push at the end) and must yield byte for byte the
    columns bam_plbuf.c saw when it was compiled unmodified against the compatibility header
    (tests/golden/plbuf_dumps.json, written by tests/golden/make_plbuf_golden.py) and those of htslib's iterator."""
    got = subprocess.run([dump_emul, '-p', os.path.join(corpus, f)], capture_output=True)
    want = subprocess.run([oracle_bin, 'pileup-dump', os.path.join(corpus, f)], capture_output=True)
    assert got.returncode == 0, got.stderr[-300:]
    assert got.stdout == want.stdout and len(got.stdout) > 100
    assert {'sha256': hashlib.sha256(got.stdout).hexdigest(), 'bytes': len(got.stdout)} == PLBUF_GOLDEN[f]


@pytest.mark.parametrize('budget', ['1', '400', '5000'])
@pytest.mark.parametrize('args,files', golden_cases.COMPAT_CASES, ids=golden_cases.COMPAT_IDS)
def test_iterator_tier_windows(args, files, budget, dump_emul, oracle_bin, corpus, monkeypatch):
    """B200_PLP_WINDOW_BYTES: the tier cuts a reference sequence into windows once the collected reads exceed a payload budget
    (cut at the start of the read that exceeded it, halo reads staged again, columns served window by window).  With budgets of
    1 / 400 / 5000 bases every case is cut many times -- mate overlaps across a cut, deletions, the max-depth case, the k-way
    merge of three files, the hooks -- and must dump exactly what htslib's iterator yields."""
    monkeypatch.setenv('B200_PLP_WINDOW_BYTES', budget)
    paths = [os.path.join(corpus, f) for f in files]
    got = subprocess.run([dump_emul, '-c', *args, *paths], capture_output=True)
    want = subprocess.run([oracle_bin, 'pileup-dump', *args, *paths], capture_output=True)
    assert got.returncode == 0, got.stderr[-300:]
    assert got.stdout == want.stdout
    assert b'bad=0' in got.stderr
