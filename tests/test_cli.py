"""The `uncomp` host program's argument handling and ATZ1 reader errors (no GPU needed for these paths)."""
import json
import os
import struct
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")


def run(*a):
    # started as `uncomp` (argv[0]) wherever the checkout lies: TCLAP wraps the usage text relative to the program name
    return subprocess.run(["uncomp"] + list(a), executable=UNCOMP, capture_output=True, text=True)


def test_missing_input_is_a_parse_error():
    p = run()
    assert p.returncode == 1 and "AntiZ 0.1.6-git" in p.stdout
    assert "PARSE ERROR" in p.stderr and "Required argument missing: input" in p.stderr


def test_unknown_flag_and_version():
    assert run("--bogus").returncode == 1
    v = run("--version")
    assert v.returncode == 0 and "0.1.6-git" in v.stdout
    h = run("--help")
    assert h.returncode == 0 and "--brute-window" in h.stdout and "--shortcut-len" in h.stdout


def test_reconstruct_rejects_bad_atz():
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "x.atz")
        open(f, "wb").write(b"NOPE" + bytes(40))
        p = run("-r", "-i", f)
        assert p.returncode == 255 and "Invalid file: ATZ1 header not found" in p.stdout          # main.cpp:1018-1021, main() returns -1
        open(f, "wb").write(b"ATZ\x01" + struct.pack("<QQQ", 999, 10, 0) + b"0123456789")
        p = run("-r", "-i", f)
        assert p.returncode == 255 and "Invalid file: ATZ file size mismatch" in p.stdout        # main.cpp:1022-1025
        # an ATZ with no recompressed streams is a plain copy from offset 28 (main.cpp:941-948); needs no GPU
        body = b"hello world, no streams here"
        open(f, "wb").write(b"ATZ\x01" + struct.pack("<QQQ", 28 + len(body), len(body), 0) + body)
        p = run("-r", "-i", f, "-o", f + ".rec")
        assert p.returncode == 0 and open(f + ".rec", "rb").read() == body
        assert "reconstructing from" in p.stdout and "Original file size: %d" % len(body) in p.stdout


REF = os.path.join(ROOT, "oracle", "_ref", "uncomp_ref")
CLI_CASES = ["", "--bogus", "--version", "-i", "--input", "-r", "-i x --recomp-tresh abc", "-i x --recomp-tresh 12abc", "-i x --chunksize", "-i x -i y",
             "-i x extra", "-i x --notest --notest", "-i nosuchfile -- foo bar", "-o y", "-i x -o", "--shortcut-len 5 --shortcut-len 6 -i x"]


GOLDEN_CLI = os.path.join(ROOT, "tests", "golden", "cli_reference.json")
EXTENSIONS = "antiz_b200 extensions: "


def cli_texts(exe, tmp):
    """{args: [exit code, stdout, stderr]} of `./uncomp args` for CLI_CASES and --help, with `exe` started as ./uncomp (the usage
    line is wrapped relative to the program name).  This project's --help goes on after the reference's text with its extensions:
    only the reference's part is kept."""
    d = os.path.join(tmp, os.path.basename(exe) + "_dir")
    os.mkdir(d); os.symlink(exe, os.path.join(d, "uncomp"))
    out = {}
    for args in CLI_CASES + ["--help"]:
        p = subprocess.run(["./uncomp"] + args.split(), cwd=d, capture_output=True, text=True)
        out[args] = [p.returncode, p.stdout.split(EXTENSIONS)[0] if args == "--help" else p.stdout, p.stderr]
    return out


def test_cli_texts_equal_the_reference_binary():
    """usage, help, version and parse-error texts (stdout, stderr, exit code) against the reference's TCLAP front end: the
    reference binary where it has been built, else the stored record of its texts"""
    with tempfile.TemporaryDirectory() as tmp:
        want = cli_texts(REF, tmp) if os.path.exists(REF) else json.load(open(GOLDEN_CLI))
        for args in CLI_CASES:
            p = subprocess.run(["./uncomp"] + args.split(), cwd=tmp, executable=UNCOMP, capture_output=True, text=True)
            assert [p.returncode, p.stdout, p.stderr] == want[args], args
        # --help: the reference's text, then the extensions of this implementation
        r = want["--help"]
        u = subprocess.run(["./uncomp", "--help"], cwd=tmp, executable=UNCOMP, capture_output=True, text=True)
        assert r[0] == u.returncode == 0 and u.stdout.startswith(r[1]) and r[2] == u.stderr
        rest = u.stdout[len(r[1]):]
        assert rest.startswith(EXTENSIONS) and all(f in rest for f in ("--gpus <integer>", "--device <integer>", "--exact-records", "--stats"))


def test_cli_layout_without_the_reference():
    """the same layout rules, pinned on literal text (runs where oracle/_ref is absent)"""
    p = run("--bogus")
    assert p.returncode == 1 and p.stdout == "AntiZ 0.1.6-git\n"
    lines = p.stderr.split("\n")
    assert lines[0] == "PARSE ERROR: Argument: --bogus" and lines[1] == "             Couldn't find match for argument" and lines[3] == "Brief USAGE: "
    assert all(len(l) <= 75 for l in lines) and lines[4].startswith("   uncomp  [--brute-window] [--notest] [-r]")
    assert p.stderr.endswith("For complete USAGE and HELP type: \n   uncomp --help\n\n")
    assert run().stderr.startswith("PARSE ERROR:  \n             Required argument missing: input\n")
    assert run("-i").stderr.startswith("PARSE ERROR: Argument: -i (--input)\n             Missing a value for this argument!\n")
    assert run("-i", "x", "--mismatch-tol", "q").stderr.startswith("PARSE ERROR: Argument: (--mismatch-tol)\n             Couldn't read argument value from string 'q'\n")
    h = run("--help").stdout
    assert h.startswith("AntiZ 0.1.6-git\n\nUSAGE: \n\n   ") and "\n\nWhere: \n\n   --brute-window\n     Bruteforce deflate window size" in h
    assert "   -i <string>,  --input <string>\n     (required)  Input file name\n" in h and all(len(l) <= 75 for l in h.split("\n"))
