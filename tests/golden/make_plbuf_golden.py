#!/usr/bin/env python3
"""Record what samtools' own bam_plbuf layer sees on top of the iterator tier: tests/golden/plbuf_dumps.json.

bam_plbuf.c (bam_plbuf.h:32-51) is compiled UNMODIFIED from a samtools 1.23.1 source tree against
tests/compat/shim/htslib/sam.h -> include/b200_htslib_compat.h and linked with tests/compat/plbuf_dump.cpp on the
emulation harness (tests/emul/emul_engine.cpp).  Its column dump of each file in PLBUF_FILES is stored as a sha256
digest and a length; tests/test_emul_compat.py::test_reference_bam_plbuf_rides_on_the_tier checks the tier's push
interface against them.  Nothing of the samtools source is stored.  Run:

    python tests/golden/make_plbuf_golden.py <samtools source tree>
"""
import hashlib, json, os, subprocess, sys, tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
import golden_cases  # noqa: E402

OUT = os.path.join(HERE, 'plbuf_dumps.json')
PLBUF_FILES = ['test/mpileup/mp_DI.sam', 'test/mpileup/mp_N2.sam', 'test/mpileup/mpileup.1.bam']


def main(ref):
    if not os.path.isfile(os.path.join(ref, 'bam_plbuf.c')):
        raise SystemExit(f'{ref}: no bam_plbuf.c (usage: make_plbuf_golden.py <samtools source tree>)')
    host = os.path.join(ROOT, 'samtools_b200', 'csrc', 'host')
    inc = ['-I' + os.path.join(ROOT, 'include'), '-I' + os.path.join(ROOT, 'tests', 'compat', 'shim'), '-I' + ref]
    with tempfile.TemporaryDirectory() as td:
        obj, exe = os.path.join(td, 'bam_plbuf.o'), os.path.join(td, 'plbuf_dump')
        subprocess.run(['gcc', '-c', '-O1', *inc, '-o', obj, os.path.join(ref, 'bam_plbuf.c')], check=True)
        subprocess.run(['g++', '-std=c++17', '-O1', *inc, '-o', exe, os.path.join(ROOT, 'tests', 'compat', 'plbuf_dump.cpp'), obj,
                        os.path.join(host, 'plp_compat.cpp'), os.path.join(host, 'hts_io.cpp'),
                        os.path.join(ROOT, 'tests', 'emul', 'emul_engine.cpp'), '-lz'], check=True)
        corpus = golden_cases.prepare(td)
        rec = {}
        for f in PLBUF_FILES:
            out = subprocess.run([exe, os.path.join(corpus, f)], capture_output=True, check=True).stdout
            rec[f] = {'sha256': hashlib.sha256(out).hexdigest(), 'bytes': len(out)}
    with open(OUT, 'w') as o:
        json.dump(rec, o, indent=1)
        o.write('\n')
    print(json.dumps(rec, indent=1))


if __name__ == '__main__':
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
