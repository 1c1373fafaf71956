"""Generates tests/golden/atz_reference.json and cli_reference.json: what the reference binary writes for every input that
test_gpu_e2e.py and test_host_logic.py compare with it - the sha256 of the input and of the .atz file with the summary lines, or the
headers found and the recompressed streams - and the texts test_cli.py compares with it.  They come from oracle/_ref/uncomp_ref where it
has been built; elsewhere from this project's uncomp, which the same tests found to write the reference binary's .atz files and texts
(the .atz files need a GPU; `--cli` writes cli_reference.json alone).
Run: python tests/golden/make_atz_golden.py [--cli] [output directory]"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import zref  # noqa: E402
from test_gpu_e2e import KEEP, UNCOMP, reference_inputs, sha256  # noqa: E402
from test_cli import cli_texts  # noqa: E402
from test_host_logic import atz_streams, fold_inputs  # noqa: E402

args = [a for a in sys.argv[1:] if a != "--cli"]
dest = args[0] if args else HERE
exe = zref.REF_BIN if os.path.exists(zref.REF_BIN) else UNCOMP
src = os.path.basename(exe)
with tempfile.TemporaryDirectory() as tmp:
    json.dump(cli_texts(exe, tmp), open(os.path.join(dest, "cli_reference.json"), "w"), indent=1, sort_keys=True)
if "--cli" in sys.argv:
    sys.exit(0)
out = {}
for key, (make, flags) in reference_inputs().items():
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "in.bin")
        open(f, "wb").write(make())
        r = subprocess.run([exe, "-i", f, "-o", f + ".atz", "--notest"] + flags, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out[key] = {"input_sha256": sha256(f), "flags": flags, "atz_sha256": sha256(f + ".atz"),
                    "lines": [l for l in r.stdout.splitlines() if l.startswith(KEEP)], "source": src}
        print(key, out[key]["lines"], flush=True)
for key, (data, S) in fold_inputs().items():
    with tempfile.TemporaryDirectory() as tmp:
        found, recs = atz_streams(exe, data, S, tmp)
    out[key] = {"input_sha256": hashlib.sha256(data).hexdigest(), "chunksize": S, "found": found, "records": recs, "source": src}
    print(key, found, len(recs), flush=True)
json.dump(out, open(os.path.join(dest, "atz_reference.json"), "w"), indent=1, sort_keys=True)
