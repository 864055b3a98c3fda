"""CPU dry run of ``gc_bias`` and the ``gc-bias`` command: the public-API bodies of tests/test_gpu_gc_bias.py with the
kernel wrappers swapped for the oracle (tests/host_shim.py) and ``device.gc_observed`` / ``device.gc_expected`` for
the numpy definition (tests/gc_oracle.py).  Covers region parsing, merging and warnings, the writer, errors, the CLI,
the C ABI's argument checks and a world-size-2 run where no GPU exists; the ``-m gpu`` run covers the kernels."""
import inspect
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import bam_replay as R
import gc_oracle as GO
import host_shim
import test_gpu_gc_bias as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class HostRef:
    """Stand-in for ``device.PackedContig``."""

    def __init__(self, codes, nmask):
        self.codes, self.nmask, self.length = codes, nmask, int(codes.shape[0])
        self.device = torch.device("cpu")


def host_gc_observed(frags, ref, reg_start, reg_stop, min_length, max_length, quality_threshold=30, out=None):
    from finaletoolkit_b200.device import gc_check
    gc_check(min_length, max_length)
    fr = frags.fr
    got = torch.from_numpy(GO.observed(fr.start, fr.stop, fr.mapq, ref.codes, ref.nmask, ref.length, list(reg_start),
                                       list(reg_stop), int(min_length), int(max_length), quality_threshold))
    return got if out is None else out.add_(got)


def host_gc_expected(ref, reg_start, reg_stop, min_length, max_length, out=None):
    from finaletoolkit_b200.device import gc_check
    gc_check(min_length, max_length)
    got = torch.from_numpy(GO.expected(ref.codes, ref.nmask, ref.length, list(reg_start), list(reg_stop),
                                       int(min_length), int(max_length)))
    return got if out is None else out.add_(got)


def install(monkeypatch):
    from finaletoolkit_b200 import device
    from finaletoolkit_b200.io.reference import ReferenceWrapper
    host_shim.install(monkeypatch, {})
    monkeypatch.setattr(ReferenceWrapper, "device_contig", lambda self, contig, device=None: HostRef(*self.contig_arrays(contig)))
    monkeypatch.setattr(device, "gc_observed", host_gc_observed)
    monkeypatch.setattr(device, "gc_expected", host_gc_expected)
    monkeypatch.setattr(device, "require_cuda", lambda device=None: torch.device("cpu"))


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    install(monkeypatch)
    yield
    fragments._CACHE.clear()


test_gc_bias_api = G.test_gc_bias_api
test_gc_bias_fasta_iupac = G.test_gc_bias_fasta_iupac
test_gc_bias_errors = G.test_gc_bias_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_region_parsing(tmp_path):
    from finaletoolkit_b200.frag._gc_bias import read_regions
    bed = tmp_path / "r.bed"
    bed.write_text("# c\ntrack x\nbrowser y\n\nA\t50\t60\nA\t10\t20\nA\t20\t25\nA\t-5\t3\nA\t55\t58\nB\t90\t200\n"
                   "A\t70\t70\nZ\t1\t2\nA\t95\t400\nY\t0\t1\nZ\t4\t5\n")
    with pytest.warns(UserWarning, match="lacks were skipped: Z, Y$") as rec:
        got = read_regions(str(bed), {"A": 100, "B": 150})
    assert len([w for w in rec if issubclass(w.category, UserWarning)]) == 1
    assert {c: (s.tolist(), e.tolist()) for c, (s, e) in got.items()} == \
        {"A": ([0, 10, 50, 95], [3, 25, 60, 100]), "B": ([90], [150])}
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert read_regions(str(bed), {"A": 100, "B": 150, "Y": 9, "Z": 9})["Z"][0].tolist() == [1, 4]
    bed.write_text("A\t5\t4\n")
    with pytest.raises(ValueError, match="invalid"):
        read_regions(str(bed), {"A": 100})


def test_writer_text(tmp_path):
    from finaletoolkit_b200.frag._gc_bias import GCBias, gc_ratio, gc_text
    O = np.array([[0, 3, 1, 0], [0, 0, 0, 0], [1, 2, 0, 5]], np.int64)
    E = np.array([[4, 4, 0, 0], [1, 1, 1, 0], [3, 3, 7, 1]], np.int64)
    R_ = gc_ratio(O, E)
    assert np.array_equal(R_, GO.ratio(O, E), equal_nan=True)
    text = gc_text(GCBias(O, E, R_, 1, 3))
    assert text == GO.text(O, E, R_, 1)
    assert text.splitlines()[:4] == ["length\tgc\tobserved\texpected\tratio", "1\t0\t0\t4\t0.0", "1\t1\t3\t4\t1.5",
                                     "2\t0\t0\t1\tnan"]
    assert text.splitlines()[-1] == f"3\t3\t5\t1\t{(5 / 8) / (1 / 14)!r}"
    assert len(text.splitlines()) == 1 + 2 + 3 + 4


def test_cli_flags_and_kwargs(tmp_path, manifest, golden):
    from finaletoolkit_b200.cli.main_cli import BIAS_COMMANDS, COMMANDS, EXTRA_COMMANDS, SITE_COMMANDS, main_cli
    from finaletoolkit_b200.frag import gc_bias
    assert set(BIAS_COMMANDS) == {"gc-bias"}
    assert not set(BIAS_COMMANDS) & (set(COMMANDS) | set(EXTRA_COMMANDS) | set(SITE_COMMANDS))
    module, func, _, spec = BIAS_COMMANDS["gc-bias"]
    assert (module, func) == ("finaletoolkit_b200.frag", "gc_bias")
    assert CliRunner().invoke(main_cli, ["gc-bias", "--help"]).exit_code == 0
    sig = inspect.signature(gc_bias).parameters
    assert {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec} == set(sig)
    flags = {f: names[-1] for kind, names, _ in spec if kind == "opt" for f in names[:-1]}
    assert flags == {"--regions": "interval_file", "-r": "reference_file", "--reference": "reference_file",
                     "-o": "output_file", "--output": "output_file", "--min-length": "min_length",
                     "--max-length": "max_length", "-q": "quality_threshold", "--min-mapq": "quality_threshold",
                     "-t": "workers", "--threads": "workers", "-v": "verbose", "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    assert defaults.pop("output_file") == "-" and sig["output_file"].default is None   # the CLI writes to stdout
    for name, d in defaults.items():
        assert sig[name].default == d, name
    frag, tb, _, _ = G.motif_files(tmp_path, manifest, golden)
    out = str(tmp_path / "cli.tsv.gz")
    r = CliRunner().invoke(main_cli, ["gc-bias", frag, tb, "-o", out, "--min-length", "60", "--max-length", "90",
                                      "-q", "10", "-t", "3"])
    assert r.exit_code == 0, r.output
    import gzip
    res = gc_bias(frag, tb, min_length=60, max_length=90, quality_threshold=10)
    with gzip.open(out, "rt") as fh:
        assert fh.read() == GO.text(res.observed, res.expected, res.ratio, 60)
    r = CliRunner().invoke(main_cli, ["gc-bias", frag, tb, "-o", "x.txt"])
    assert isinstance(r.exception, ValueError)


def test_gc_abi_argument_validation():
    """ftk_gc_observed_u64 / ftk_gc_expected_u64 check their arguments before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import lib
    build()
    o, e = lib().ftk_gc_observed_u64, lib().ftk_gc_expected_u64
    #       start stop mapq n_frag maxL seq nm clen rs re n_reg min max q splits scratch out stream
    assert o(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 50, 500, 30, 1, 0, 0, 0) == 0               # no regions: zero work
    assert o(8, 8, 0, 0, 0, 8, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == 0             # no fragments: zero work
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 0, 0, 3, 50, 500, 30, 1, 8, 8, 0) == -1            # regions, no tables
    assert o(0, 0, 0, 5, 0, 8, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -1            # fragments, no columns
    assert o(8, 8, 0, -1, 0, 8, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -1           # n_frag < 0
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, -3, 50, 500, 30, 1, 8, 8, 0) == -1           # n_reg < 0
    assert o(8, 8, 0, 5, 0, 0, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -1            # no reference
    assert o(8, 8, 0, 5, 0, 4, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -1            # seq words not 8-byte aligned
    assert o(8, 8, 0, 5, 0, 8, 8, -1, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -1             # contig_len < 0
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 3, 0, 500, 30, 1, 8, 8, 0) == -1             # min_len < 1
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 3, 200, 100, 30, 1, 8, 8, 0) == -1           # max_len < min_len
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 3, 50, 500, 30, 0, 8, 8, 0) == -1            # splits < 1
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 3, 50, 1025, 30, 1, 8, 8, 0) == -3           # max_len > 1024
    assert o(8, 8, 0, 5, 0, 8, 8, 2 ** 31, 8, 8, 3, 50, 500, 30, 1, 8, 8, 0) == -3        # contig_len > 2^31 - 1
    assert o(8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 2 ** 30, 50, 500, 30, 4, 8, 8, 0) == -3      # 2^32 units
    #       seq nm clen lo hi n_tiles cap min max out stream
    assert e(0, 0, 0, 0, 0, 0, 0, 50, 500, 0, 0) == 0                                     # no tiles: zero work
    assert e(8, 8, 100, 0, 8, 3, 10, 50, 500, 8, 0) == -1                                 # no tile table
    assert e(8, 8, 100, 8, 8, -1, 10, 50, 500, 8, 0) == -1                                # n_tiles < 0
    assert e(8, 8, 100, 8, 8, 3, 0, 50, 500, 8, 0) == -1                                  # tile_cap < 1
    assert e(8, 8, 100, 8, 8, 3, 10, 50, 500, 0, 0) == -1                                 # no output
    assert e(8, 0, 100, 8, 8, 3, 10, 50, 500, 8, 0) == -1                                 # no N mask
    assert e(8, 8, 100, 8, 8, 3, 10, 0, 500, 8, 0) == -1                                  # min_len < 1
    assert e(8, 8, 100, 8, 8, 3, 10, 60, 50, 8, 0) == -1                                  # max_len < min_len
    assert e(8, 8, 100, 8, 8, 3, 10, 50, 1025, 8, 0) == -3                                # max_len > 1024
    assert e(8, 8, 100, 8, 8, 3, 16385, 50, 500, 8, 0) == -3                              # tile_cap > 16384
    assert e(8, 8, 2 ** 31, 8, 8, 3, 10, 50, 500, 8, 0) == -3                             # contig_len > 2^31 - 1


_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
repo = os.environ["FTK_REPO"]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from _pytest.monkeypatch import MonkeyPatch
import test_gc_bias_dryrun as GD
import finaletoolkit_b200 as F
mp = MonkeyPatch()
GD.install(mp)
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank = dist.get_rank()
d = os.environ["FTK_DIR"]
r = F.gc_bias(os.path.join(d, "read1.bam"), os.path.join(d, "read1.2bit"), os.path.join(d, "regions.bed"),
              output_file=os.path.join(d, "g%d.tsv" % rank), min_length=50, max_length=300, quality_threshold=0)
from finaletoolkit_b200.distributed import owned_contigs
from finaletoolkit_b200.io.fragments import load_fragments
np.save(os.path.join(d, "o%d.npy" % rank), r.observed); np.save(os.path.join(d, "e%d.npy" % rank), r.expected)
print(json.dumps({"rank": rank, "mine": owned_contigs(load_fragments(os.path.join(d, "read1.bam")))}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2(tmp_path, golden):
    import finaletoolkit_b200 as F
    bam = R.make_fixture(tmp_path, golden)
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    (tmp_path / "regions.bed").write_text("".join(f"{t[0]}\t{t[1]}\t{t[2]}\n" for t in tiles[::2]))
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(35500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", FTK_REPO=REPO, FTK_PORT=port, FTK_DIR=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-2000:] for o in outs]
    got = [json.loads(o[0].strip().splitlines()[-1]) for o in outs]
    assert sorted(got[0]["mine"] + got[1]["mine"]) == ["chrA", "chrB"] and got[0]["mine"] and got[1]["mine"]
    single = F.gc_bias(bam["path"], bam["tb"], str(tmp_path / "regions.bed"), min_length=50, max_length=300,
                       quality_threshold=0)
    assert single.observed.sum() > 0
    for r in range(2):
        assert np.array_equal(np.load(tmp_path / f"o{r}.npy"), single.observed), r
        assert np.array_equal(np.load(tmp_path / f"e{r}.npy"), single.expected), r
    assert open(tmp_path / "g0.tsv").read() == GO.text(single.observed, single.expected, single.ratio, 50)
    assert not (tmp_path / "g1.tsv").exists()
