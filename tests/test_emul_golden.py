"""Host drivers + per-column / per-read arithmetic, single-stepped on the CPU.

tests/emul/emul_engine.cpp implements the C ABI by calling the very same
__host__ __device__ functions the CUDA kernels call (plp_core.h, plp_stage.h)
and the engine's host-side policy (stage_host.h: max-depth sweep, sortedness,
column domain, text bounds).  What it does on its own is only the control flow:
sequential loops in place of the kernel grids and a host prefix max in place of
the device scans.  So the b200samtools driver code (option handling, -a/-aa
sequencing, packing, BED / RG / BQ-tag host bits), the column formatters and
the output bounds can be checked against the reference's golden outputs without
a GPU.  This harness is a debugging aid, not a product path: it is never linked
into libb200pileup.so / b200samtools.
The BAQ kernel (warp-cooperative) is not emulated: those cases run in -m gpu."""
import os, subprocess
import pytest
import golden_cases
from conftest import ROOT

CASES = golden_cases.all_cases()


@pytest.fixture(scope='module')
def emul_bin():
    subprocess.run([os.path.join(ROOT, 'tests', 'emul', 'build.sh')], check=True)
    return os.path.join(ROOT, 'tests', 'emul', '_build', 'b200samtools_emul')


@pytest.mark.parametrize('case', CASES, ids=[c['id'] for c in CASES])
def test_host_drivers_and_column_code(case, emul_bin, oracle_bin, corpus):
    if case['skip']:
        pytest.skip(case['skip'])
    ok, out, err = golden_cases.run_case(case, emul_bin, oracle_bin, corpus)
    if not ok and b'BAQ kernel is not emulated' in err:
        pytest.skip('needs the BAQ kernel (covered by -m gpu)')
    if not ok and b'not available on the device path' in err:
        pytest.skip('--output-extra/QNAME/mods: host-string columns not on the device path yet')
    assert ok, f"{case['cmd']}\nstderr: {err[-300:]!r}\nstdout head: {out[:200]!r}"


@pytest.mark.parametrize('cmd', [c for c in golden_cases.EX1_CMDS if ' -B ' in c])
def test_c1_ex1_host_path(cmd, emul_bin, oracle_bin, corpus):
    """BASELINE config 1 plumbing (headerless SAM + .fai contig list) through the host drivers, no GPU."""
    cwd = os.path.join(corpus, 'examples')
    want = subprocess.run(f'{oracle_bin} {cmd}', shell=True, cwd=cwd, capture_output=True)
    got = subprocess.run(f'{emul_bin} {cmd}', shell=True, cwd=cwd, capture_output=True)
    assert len(want.stdout) > 1000 and got.stdout == want.stdout


def test_column_windows_with_halo(emul_bin, oracle_bin, corpus, monkeypatch):
    """The drivers cut every reference sequence into column windows and stage, per window, the records overlapping it
    (halo = reads reaching in from the left, the -r rule bam_plcmd.c:550-554,609).  With 97-column windows every golden
    mpileup / depth / coverage case crosses dozens of window edges -- reads, mate overlaps, deletions, -a / -aa rows,
    BED filters, depth -s clips, coverage read counts -- and must still reproduce the reference's bytes."""
    from concurrent.futures import ThreadPoolExecutor
    monkeypatch.setenv('B200_WINDOW_COLS', '97')
    todo = [c for c in CASES if not c['skip'] and '>' not in c['cmd']]

    def run(c):
        ok, out, err = golden_cases.run_case(c, emul_bin, oracle_bin, corpus)
        if not ok and (b'BAQ kernel is not emulated' in err or b'not available on the device path' in err):
            return None
        return None if ok else (c['id'], c['cmd'], err[-200:])
    with ThreadPoolExecutor(max_workers=6) as ex:
        bad = [r for r in ex.map(run, todo) if r]
    assert not bad, bad[:3]


def test_coverage_histogram_views(emul_bin, oracle_bin, corpus, tmp_path, monkeypatch):
    """`coverage -m / -A / -D / -w` (per-bin counters b200_coverage_hist + the host-side print_hist) against the oracle, on the
    reference's sample.sam and on a synthetic 30 kb contig cut into 997-column windows (bins accumulate across windows)."""
    import hist_cases
    from samtools_b200 import synth
    soa = synth.make_batch(length=30_000, depth=12, seed=21)
    sam = str(tmp_path / 'h.sam')
    synth.write_sam(sam, soa)
    assert not hist_cases.run_all(emul_bin, oracle_bin, corpus, tmp_path, sam)
    assert not hist_cases.run_all(emul_bin, oracle_bin, corpus, tmp_path, sam, {'B200_WINDOW_COLS': '997'})


def test_swar_entry_formatter_exhaustive(tmp_path):
    """ent_group8_swar (plp_core.h: eight bases formatted SIMD-in-word by the device entry pass) == ent_plain for every
    quality byte x base code x strand x -Q 0..127 x reference equal / different / absent, at every position of a group"""
    exe = str(tmp_path / 'swar_check')      # built here: pytest-xdist workers rebuild tests/emul/_build concurrently
    subprocess.run(['g++', '-std=c++17', '-O2', '-Wno-parentheses', '-o', exe, os.path.join(ROOT, 'tests', 'emul', 'swar_check.cpp')], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and ' 0 mismatches' in r.stdout, r.stdout + r.stderr


def test_window_workers(emul_bin, oracle_bin, corpus, monkeypatch):
    """B200_DEVICES / B200_HANDLES: the mpileup driver hands the column windows of a reference sequence round-robin to several
    engine handles (one per listed device; threads) and writes their text in window order.  Every golden mpileup / depth case with
    97-column windows over three workers must still reproduce the reference's bytes."""
    from concurrent.futures import ThreadPoolExecutor
    monkeypatch.setenv('B200_WINDOW_COLS', '97')
    monkeypatch.setenv('B200_DEVICES', '0,0,0')
    todo = [c for c in CASES if not c['skip'] and '>' not in c['cmd'] and ('mpileup' in c['cmd'] or 'depth' in c['cmd'])]

    def run(c):
        ok, out, err = golden_cases.run_case(c, emul_bin, oracle_bin, corpus)
        if not ok and (b'BAQ kernel is not emulated' in err or b'not available on the device path' in err):
            return None
        return None if ok else (c['id'], c['cmd'], err[-200:])
    with ThreadPoolExecutor(max_workers=4) as ex:
        bad = [r for r in ex.map(run, todo) if r]
    assert len(todo) > 100 and not bad, bad[:3]
