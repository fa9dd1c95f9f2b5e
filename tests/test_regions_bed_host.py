"""CPU: compress_b200 --decompress --regions= refuses a malformed BED file before it touches the device: the line
number and the fault on stderr, exit status 1, no output file."""
import subprocess

import pytest

from conftest import ROOT

COMPRESS = ROOT / "genome-compression_b200" / "host" / "compress_b200"

MALFORMED = [
    ("chr1 0 10\nchr1 5 x\n", "line 2: "),
    ("chr1 -1 10\n", "line 1: "),
    ("chr1 0 1e3\n", "line 1: "),
    ("# header\nchr1 20 10\n", "line 2: "),
    ("chr1 0 10 name 0 *\n", "line 1: "),
    ("track a\n\nchr1 0\n", "line 3: "),
    ("chr1 0 99999999999999999999\n", "line 1: "),
]


@pytest.mark.parametrize("bed,message", MALFORMED)
def test_malformed_bed_is_refused_before_the_device(stb, tmp_path, bed, message):
    assert COMPRESS.exists(), "genome-compression_b200/host/compress_b200 missing: run __graft_entry__.build()"
    dag = tmp_path / "in.dag"
    dag.write_bytes(b"not read: the BED file is parsed first")
    (tmp_path / "r.bed").write_text(bed)
    out = tmp_path / "out.fa"
    res = subprocess.run([COMPRESS, "--decompress", "--dna-size=12", f"--regions={tmp_path / 'r.bed'}", f"--output={out}", dag],
                         capture_output=True, text=True, timeout=60)
    assert res.returncode == 1, res.stdout + res.stderr
    assert res.stderr.startswith(message), res.stderr
    assert not out.exists() and not (tmp_path / "in.fa").exists()
