"""`rsicnv ... -crc`: the CRC32 of every BGZF block decoded on the GPU is checked (rsigpu_set_bgzf_crc) on every route that feeds
BAM bytes to a GPU decoder.  Without the flag a block whose only damage is its CRC footer decodes as before; with it the contig
that holds the block fails like a corrupt deflate stream does: no rows for it, the error on stderr, a non-zero exit status."""
import os
import shutil
import struct
import subprocess

import pytest

from rsicnv_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    return CLI


def _table(path):
    return [ln for ln in open(path).read().splitlines() if not ln.startswith("#input")]


def test_crc_flag_is_parsed_and_listed(cli, tmp_path):
    out = subprocess.run([cli], capture_output=True, text=True)
    assert "-crc" in out.stderr, out.stderr
    out = subprocess.run([cli, "rsi", "-b", str(tmp_path / "x.bam"), "-f", str(tmp_path / "x.fa"), "-crc"], capture_output=True, text=True)
    assert "unknown option" not in out.stderr, out.stderr
    out = subprocess.run([cli, "stat", "-b", str(tmp_path / "x.bam"), "-v", str(tmp_path / "x.txt"), "-crc"], capture_output=True, text=True)
    assert "unknown option" not in out.stderr, out.stderr


@pytest.fixture(scope="module")
def two_contigs(tmp_path_factory):
    d = tmp_path_factory.mktemp("crc")
    lens = [4_300_000, 4_200_000]
    fas = [synth.make_fasta(L, 90 + i) for i, L in enumerate(lens)]
    reads = {i: synth.make_reads(L, 90 + i, fas[i], coverage=8, n_events=4, lens=(4000, 9000, 20000), tid=i)[0] for i, L in enumerate(lens)}
    bam = str(d / "t.bam"); fasta = str(d / "t.fa")
    synth.write_bam(bam, [("1", lens[0]), ("2", lens[1])], reads, level=1, random_seq=5)
    synth.write_fasta_multi(fasta, [("1", fas[0]), ("2", fas[1])])
    synth.write_bai(bam)
    return d, bam, fasta


def _run(cli, args, out, env=None):
    return subprocess.run([cli] + args + ["-o", out], capture_output=True, text=True, env=dict(os.environ, **(env or {})))


def _rsi(bam, fasta):
    return ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]


@pytest.mark.gpu
def test_cli_crc_footer_damage(cli, two_contigs, tmp_path):
    d, bam, fasta = two_contigs
    good = _run(cli, _rsi(bam, fasta), str(tmp_path / "good.txt"))
    assert good.returncode == 0, good.stderr
    want = _table(str(tmp_path / "good.txt"))
    rows = [ln for ln in want if not ln.startswith("#")]
    assert {ln.split("\t")[0] for ln in rows} == {"1", "2"}
    first = [ln for ln in rows if ln.split("\t")[0] == "1"]
    # one bit of the CRC footer of the BGZF block that holds the file's 80 % point (well inside contig 2)
    data = bytearray(open(bam, "rb").read())
    off = 0; at = int(len(data) * 0.8)
    while True:
        bsize = struct.unpack_from("<H", data, off + 16)[0] + 1
        if off + bsize > at:
            break
        off += bsize
    data[off + bsize - 7] ^= 0x08
    bad = str(tmp_path / "bad.bam")
    open(bad, "wb").write(bytes(data))
    shutil.copy(bam + ".bai", bad + ".bai")
    # without -crc: today's behaviour, the same table
    out = _run(cli, _rsi(bad, fasta), str(tmp_path / "nocrc.txt"))
    assert out.returncode == 0, out.stderr
    assert _table(str(tmp_path / "nocrc.txt")) == want
    # with -crc: contig 2 fails on the indexed and the one-pass route, contig 1 is untouched on the indexed one
    for env in ({}, {"RSICNV_NO_INDEX": "1"}):
        out = _run(cli, _rsi(bad, fasta) + ["-crc"], str(tmp_path / "crc.txt"), env)
        assert out.returncode != 0, (env, out.stderr)
        assert any("CRC32" in ln for ln in out.stderr.splitlines()), (env, out.stderr)
        got = [ln for ln in _table(str(tmp_path / "crc.txt")) if not ln.startswith("#")]
        assert not [ln for ln in got if ln.split("\t")[0] == "2"], (env, out.stderr)
        if not env:
            assert got == first, out.stderr
    # the host decoder always checks: the damaged block is reported and contig 2 gets no rows
    out = _run(cli, _rsi(bad, fasta) + ["-hostdecode"], str(tmp_path / "host.txt"))
    assert "CRC" in out.stderr, out.stderr
    if os.path.exists(str(tmp_path / "host.txt")):
        assert not [ln for ln in _table(str(tmp_path / "host.txt")) if ln.split("\t")[0] == "2"], out.stderr


@pytest.mark.gpu
def test_cli_crc_intact_file_same_table(cli, two_contigs, tmp_path):
    d, bam, fasta = two_contigs
    for extra, env in (([], {}), ([], {"RSICNV_NO_INDEX": "1"})):
        a = _run(cli, _rsi(bam, fasta) + extra, str(tmp_path / "a.txt"), env)
        b = _run(cli, _rsi(bam, fasta) + extra + ["-crc"], str(tmp_path / "b.txt"), env)
        assert a.returncode == 0 and b.returncode == 0, (extra, env, a.stderr, b.stderr)
        assert _table(str(tmp_path / "a.txt")) == _table(str(tmp_path / "b.txt")), (extra, env)
    # stat with the table just written as its list of calls
    calls = str(tmp_path / "a.txt")
    for env in ({}, {"RSICNV_NO_INDEX": "1"}):
        a = _run(cli, ["stat", "-b", bam, "-v", calls], str(tmp_path / "sa.txt"), env)
        b = _run(cli, ["stat", "-b", bam, "-v", calls, "-crc"], str(tmp_path / "sb.txt"), env)
        assert a.returncode == 0 and b.returncode == 0, (env, a.stderr, b.stderr)
        sa = open(str(tmp_path / "sa.txt")).read()
        assert "RP=" in sa and sa == open(str(tmp_path / "sb.txt")).read(), env


@pytest.mark.gpu
def test_cli_crc_two_gpus(cli, two_contigs, tmp_path):
    if api.load_library().rsigpu_num_devices() < 2:
        pytest.skip("needs two GPUs")
    d, bam, fasta = two_contigs
    a = _run(cli, _rsi(bam, fasta) + ["-gpus", "2"], str(tmp_path / "a.txt"))
    b = _run(cli, _rsi(bam, fasta) + ["-gpus", "2", "-crc"], str(tmp_path / "b.txt"))
    assert a.returncode == 0 and b.returncode == 0, (a.stderr, b.stderr)
    assert _table(str(tmp_path / "a.txt")) == _table(str(tmp_path / "b.txt"))
