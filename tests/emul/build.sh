#!/bin/sh
# Builds the DEBUG-ONLY emulation harness (see emul_engine.cpp).  Not part of the product build.
set -e
# every output is linked under a temporary name and renamed into place: pytest-xdist workers run this script concurrently
# while others execute the binaries ("text file busy" otherwise)
cd "$(dirname "$0")/../.."
mkdir -p tests/emul/_build
# up to date?  (every output present and no source newer than the oldest of them: four test modules call this script)
stamp=tests/emul/_build/.stamp
if [ -f "$stamp" ] && [ -f tests/emul/_build/b200samtools_emul ] && [ -f tests/emul/_build/plp_dump_emul ] && [ -f tests/emul/_build/baq_host ] && \
   [ -z "$(find samtools_b200/csrc include tests/emul tests/compat oracle -maxdepth 2 -type f \( -name '*.cpp' -o -name '*.h' -o -name '*.hpp' -o -name '*.cuh' -o -name '*.c' -o -name '*.sh' -o -name Makefile \) -newer "$stamp" 2>/dev/null | head -1)" ]; then
    exit 0
fi
touch tests/emul/_build/.stamp.new.$$
g++ -std=c++17 -O1 -g -ffp-contract=off -Wall -Wno-unused-function -o tests/emul/_build/b200samtools_emul.tmp$$ \
    samtools_b200/csrc/host/cli.cpp samtools_b200/csrc/host/hts_io.cpp tests/emul/emul_engine.cpp -lz
# the htslib-compatible iterator tier (plp_compat.cpp) + its test client, on the emulation harness
g++ -std=c++17 -O1 -g -ffp-contract=off -Wall -Wno-unused-function -Iinclude -o tests/emul/_build/plp_dump_emul.tmp$$ \
    tests/compat/plp_dump.cpp samtools_b200/csrc/host/plp_compat.cpp samtools_b200/csrc/host/hts_io.cpp tests/emul/emul_engine.cpp -lz
# the register-band BAQ arithmetic (samtools_b200/csrc/baq_reg.h) single-stepped on the CPU against the oracle's sam_prob_realn
make -s -C oracle
g++ -std=c++17 -O2 -ffp-contract=off -Wno-unknown-pragmas -o tests/emul/_build/baq_host.tmp$$ tests/emul/baq_host.cpp \
    -Loracle/_build -loracle -Wl,-rpath,"$PWD/oracle/_build" -lz -lm

for f in b200samtools_emul baq_host plp_dump_emul; do mv -f tests/emul/_build/$f.tmp$$ tests/emul/_build/$f; done
mv -f tests/emul/_build/.stamp.new.$$ tests/emul/_build/.stamp
