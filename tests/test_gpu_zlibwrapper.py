"""-m gpu: the ZlibInflator drop-in (antiz_b200/host/ZlibWrapper.h, reference interface ZlibWrapper.h:25-100) driven the way the
reference's scanner drives it (tests/zlibwrapper_scan.cpp: operator() / continuePrev / refillInput / totalInputByte / avail_in / avail_out /
lastRetVal, chunk by chunk with the duplicated overlap byte) must find exactly the streams the reference binary finds."""
import os
import subprocess
import tempfile

import pytest

import antiz_b200 as az
import corpus
import zref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def scanner(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("scanner") / "atz_zlibwrapper_scan")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "antiz_b200", "host"),
                           os.path.join(ROOT, "tests", "zlibwrapper_scan.cpp"), "-o", exe, "-L", os.path.join(ROOT, "antiz_b200"), "-lantiz_b200",
                           "-Wl,-rpath," + os.path.join(ROOT, "antiz_b200")])
    return exe


@pytest.mark.parametrize("chunksize", [524288, 20000, 3000])
def test_scanner_over_zlibinflator_finds_the_reference_streams(scanner, chunksize):
    data = corpus.c2(10, 55, 1 << 10, 40 << 10) + corpus.c4(40, 56) + corpus.junk(5000, 57)
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        out = subprocess.run([scanner, f, str(chunksize)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr
        got = [tuple(int(x) for x in line.split()) for line in out.stdout.splitlines()]
        # the product's own scan (proven against the reference through the byte-identical .atz files of test_gpu_e2e.py) ...
        c = az.Context(0); c.load(data); c.scan(chunksize)
        want = [(s.offset, s.offsetType, s.streamLength, s.inflatedLength) for s in c.streams()]
        c.close()
        assert got == want
        # ... and the reference binary's count for the same chunk size
        if os.path.exists(zref.REF_BIN):
            ref = subprocess.run([zref.REF_BIN, "-i", f, "-o", f + ".atz", "--notest", "--chunksize", str(chunksize)], capture_output=True, text=True)
            line = [l for l in ref.stdout.splitlines() if l.startswith("Total zlib headers found")][0]
            assert int(line.split(":")[1]) == len(got)
