"""Builds tests/simt/liblt_emu.so: the CUDA sources of the package compiled with g++ against the
SIMT emulator (simt.h) — TEST INFRASTRUCTURE.  The product only ever loads liblt_b200.so.

Several processes may build at once (pytest-xdist workers that all find the library missing or stale):
each compiles and links under names of its own and moves the finished library into place with one
rename, so a process that loads the library never sees a partly written file."""

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, 'lattice_based_tagger_b200', 'csrc')
LIB = os.path.join(HERE, 'liblt_emu.so')


def sources():
    out = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(('.cu', '.cuh'))]
    out += [os.path.join(HERE, 'simt.h'), os.path.join(HERE, 'simt.cpp'), os.path.join(ROOT, 'include', 'lt_b200.h')]
    return out


def build(force=False, opt='-O1'):
    if not force and os.path.exists(LIB) and all(os.path.getmtime(s) <= os.path.getmtime(LIB) for s in sources()):
        return LIB
    cxx = os.environ.get('CXX', 'g++')
    common = [cxx, '-std=c++17', opt, '-g', '-fPIC', '-DLT_SIMT_EMU', '-ffp-contract=off', '-fno-strict-aliasing',
              '-Wno-unknown-pragmas', '-Wno-attributes', '-I', HERE, '-I', CSRC]
    own = '.%d' % os.getpid()
    obj_k = os.path.join(HERE, 'lt_emu%s.o' % own)
    obj_s = os.path.join(HERE, 'simt%s.o' % own)
    lib = os.path.join(HERE, 'liblt_emu%s.so' % own)
    try:
        subprocess.run(common + ['-x', 'c++', '-c', os.path.join(CSRC, 'lt_b200.cu'), '-o', obj_k], check=True)
        subprocess.run(common + ['-c', os.path.join(HERE, 'simt.cpp'), '-o', obj_s], check=True)
        subprocess.run([cxx, '-shared', '-o', lib, obj_k, obj_s], check=True)
        os.replace(lib, LIB)
    finally:
        for path in (obj_k, obj_s, lib):
            if os.path.exists(path):
                os.remove(path)
    return LIB


if __name__ == '__main__':
    import sys
    print(build(force='--force' in sys.argv))
