"""CPU dry run of ``ocf`` and the ``ocf`` command: the public-API bodies of tests/test_gpu_ocf.py with the kernel
wrappers swapped for the oracle (tests/host_shim.py) and ``device.ocf_sites`` for the numpy definition
(tests/ocf_oracle.py).  Covers site sets, BAM fetch grouping, writers, errors, the CLI, the C ABI's argument checks
and a world-size-2 run where no GPU exists; the ``-m gpu`` run covers the kernel."""
import inspect
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import bam_replay as R
import host_shim
import ocf_oracle as OO
import test_gpu_ocf as G
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_ocf_sites(frags, site_center, site_flip, site_set, n_sets, flank, min_length=None, max_length=None,
                   quality_threshold=30, out=None):
    """Stand-in for ``device.ocf_sites`` on ``host_shim.HostFrags``."""
    from finaletoolkit_b200.device import _ocf_shape, ocf_length_check
    _ocf_shape(flank, n_sets)
    ocf_length_check(min_length, max_length)
    fr = frags.fr
    got = torch.from_numpy(OO.ends(fr.start, fr.stop, fr.mapq, list(site_center), list(site_flip), list(site_set),
                                   int(n_sets), int(flank), min_length, max_length, quality_threshold))
    return got if out is None else out.add_(got)


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200 import device
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    host_shim.install(monkeypatch, {})
    monkeypatch.setattr(device, "ocf_sites", host_ocf_sites)
    yield
    fragments._CACHE.clear()


test_ocf_api_fx = G.test_ocf_api_fx
test_ocf_api_syn = G.test_ocf_api_syn
test_ocf_errors = G.test_ocf_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_ocf_values_match_the_oracle():
    """The host OCF formula against the oracle's explicit loops and exact fractions, on random counts and on
    hand-made ones."""
    from finaletoolkit_b200.frag._ocf import ocf_values
    rng = np.random.default_rng(3)
    for flank, o, w in [(1000, 60, 20), (69, 60, 20), (1, 1, 1), (37, 10, 7), (500, 200, 301)]:
        counts = rng.integers(0, 10 ** 12, (5, 2, 2 * flank + 1))
        counts[1] = 0
        counts[2, 0] = 0
        got = ocf_values(counts, flank, o, w)
        for k in range(5):
            exp = OO.ocf_value(counts[k, 0], counts[k, 1], flank, o, w)
            assert (np.isnan(got[k]) and np.isnan(exp)) or got[k] == exp, (flank, o, w, k)
    c = np.zeros((1, 2, 2001), np.int64)
    c[0, 0, 1000 + 55] = 3      # U in P+
    c[0, 1, 1000 - 60] = 1      # D in P-
    assert ocf_values(c, 1000, 60, 20)[0] == 4 * 2 * 2001 / 4


def test_cli_flags_and_kwargs():
    import finaletoolkit_b200.cli.main_cli
    M = sys.modules["finaletoolkit_b200.cli.main_cli"]
    from finaletoolkit_b200.frag import ocf
    tables = [M.COMMANDS, M.EXTRA_COMMANDS, M.SITE_COMMANDS, M.BIAS_COMMANDS, M.CORRECTION_COMMANDS,
              M.SPECTRUM_COMMANDS]
    assert set(M.ORIENTATION_COMMANDS) == {"ocf"}
    assert not set(M.ORIENTATION_COMMANDS) & set().union(*map(set, tables))
    module, func, _, spec = M.ORIENTATION_COMMANDS["ocf"]
    assert (module, func) == ("finaletoolkit_b200.frag", "ocf")
    assert CliRunner().invoke(M.main_cli, ["ocf", "--help"]).exit_code == 0
    params = {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec}
    sig = inspect.signature(ocf).parameters
    assert params == set(sig)
    args = {names[0]: kw for kind, names, kw in spec if kind == "arg"}
    assert args["site_beds"]["nargs"] == -1 and args["site_beds"]["required"] is True
    flags = {f: names[-1] for kind, names, _ in spec if kind == "opt" for f in names[:-1]}
    assert flags == {"-r": "reference_file", "--reference": "reference_file", "-o": "output_file",
                     "--output": "output_file", "--profiles": "profile_file", "--flank": "flank",
                     "--peak-offset": "peak_offset", "--peak-width": "peak_width", "--min-length": "min_length",
                     "--max-length": "max_length", "-q": "quality_threshold", "--min-mapq": "quality_threshold",
                     "-t": "workers", "--threads": "workers", "-v": "verbose", "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    assert defaults.pop("output_file") == "-" and sig["output_file"].default is None   # the CLI writes to stdout
    assert defaults == {"reference_file": None, "profile_file": None, "flank": 1000, "peak_offset": 60,
                        "peak_width": 20, "min_length": None, "max_length": None, "quality_threshold": 30, "workers": 1,
                        "verbose": 0}
    for name, d in defaults.items():
        assert sig[name].default == d, name
    r = CliRunner().invoke(M.main_cli, ["ocf", "in.frag.gz"])
    assert r.exit_code != 0 and "SITES" in r.output                  # at least one site file


def test_cli_writes_files(fx, tmp_path):
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.cli.main_cli import main_cli
    a = tmp_path / "a.bed"; a.write_text(G._FX_SITES)
    b = tmp_path / "b.bed"; b.write_text(G._FX_SITES_B)
    out, prof = str(tmp_path / "cli.tsv"), str(tmp_path / "prof.tsv")
    r = CliRunner().invoke(main_cli, ["ocf", fx["frag"], str(a), str(b), "-o", out, "--profiles", prof, "--flank", "80",
                                      "--peak-offset", "40", "--peak-width", "9", "-q", "0", "-t", "3"])
    assert r.exit_code == 0, r.output
    res = F.ocf(fx["frag"], [str(a), str(b)], flank=80, peak_offset=40, peak_width=9, quality_threshold=0)
    counts = np.stack([res.upstream, res.downstream], axis=1)
    summary, profile = G.expected_texts(["a", "b"], res.n_sites.tolist(), counts, 80, 40, 9)
    assert open(out).read() == summary and open(prof).read() == profile
    r = CliRunner().invoke(main_cli, ["ocf", fx["frag"], str(a), "-o", "x.txt"])
    assert isinstance(r.exception, ValueError)


def test_ocf_abi_argument_validation():
    """ftk_ocf_u64 checks its arguments before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import FTK_NONE, lib
    build()
    f = lib().ftk_ocf_u64
    N = FTK_NONE
    T = 2 ** 32 - 1

    def call(start=1, stop=1, mapq=0, n_frag=5, max_frag_len=0, lo=1, hi=1, flip=1, sset=1, n_sites=3, n_sets=2,
             flank=10, min_len=N, max_len=N, q=30, splits=1, bounds=1, n_cta=1, flush=T, scratch=1, out=1):
        return f(start, stop, mapq, n_frag, max_frag_len, lo, hi, flip, sset, n_sites, n_sets, flank, min_len, max_len,
                 q, splits, bounds, n_cta, flush, scratch, out, 0)

    assert call(start=0, stop=0, lo=0, hi=0, flip=0, sset=0, bounds=0, scratch=0, out=0, n_sites=0, n_frag=0) == 0
    assert call(start=0, stop=0, n_frag=0) == 0                            # no fragments: zero work
    assert call(n_frag=5, min_len=300, max_len=300, max_frag_len=200) == 0  # no fragment can pass: zero work
    assert call(lo=0, hi=0, flip=0, sset=0, bounds=0, scratch=0, out=0) == -1   # sites, no tables
    for kw in ({"lo": 0}, {"hi": 0}, {"flip": 0}, {"sset": 0}, {"bounds": 0}, {"scratch": 0}, {"out": 0}):
        assert call(**kw) == -1, kw
    assert call(start=0, stop=0) == -1                                     # fragments, no columns
    for kw in ({"n_frag": -1}, {"n_sites": -3}, {"n_sets": 0}, {"n_cta": 0}, {"flank": -1}, {"splits": 0},
               {"flush": 0}, {"min_len": -1}, {"max_len": -2}, {"min_len": 200, "max_len": 100}):
        assert call(**kw) == -1, kw
    assert call(flank=8193) == -3                                          # flank > FTK_OCF_MAX_FLANK
    assert call(flush=T + 1) == -3                                         # a 32-bit counter could overflow
    assert call(n_sets=4096, flank=8192) == -3                             # 4096 x 2 x 16385 > 2^27 cells
    assert call(n_sites=2 ** 30, splits=4) == -3                           # 2^32 units
    assert call(n_sets=4095, flank=8192, n_frag=0) == 0                    # 4095 x 2 x 16385 cells fit


_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
repo = os.environ["FTK_REPO"]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from _pytest.monkeypatch import MonkeyPatch
import host_shim
import test_ocf_dryrun as OD
import finaletoolkit_b200 as F
import finaletoolkit_b200.device as D
mp = MonkeyPatch()
host_shim.install(mp, {})
mp.setattr(D, "ocf_sites", OD.host_ocf_sites)
mp.setattr(D, "require_cuda", lambda device=None: torch.device("cpu"))
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank = dist.get_rank()
d = os.environ["FTK_DIR"]
res = F.ocf(os.path.join(d, "read1.bam"), [os.path.join(d, "s0.bed"), os.path.join(d, "s1.bed")],
            output_file=os.path.join(d, "o%d.tsv" % rank), profile_file=os.path.join(d, "p%d.tsv" % rank),
            flank=150, min_length=50, max_length=300, quality_threshold=0)
from finaletoolkit_b200.distributed import owned_contigs
from finaletoolkit_b200.io.fragments import load_fragments
np.save(os.path.join(d, "m%d.npy" % rank), np.stack([res.upstream, res.downstream], axis=1))
np.save(os.path.join(d, "v%d.npy" % rank), np.concatenate([res.ocf, res.n_sites.astype(np.float64)]))
print(json.dumps({"rank": rank, "mine": owned_contigs(load_fragments(os.path.join(d, "read1.bam")))}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2(tmp_path, golden):
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.frag._ocf import ocf_profile_text, ocf_summary_text
    bam = R.make_fixture(tmp_path, golden)
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    for j in range(2):
        (tmp_path / f"s{j}.bed").write_text("".join(f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n"
                                                   for k, t in enumerate(tiles) if k % 2 == j))
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
    single = F.ocf(bam["path"], [str(tmp_path / "s0.bed"), str(tmp_path / "s1.bed")], flank=150, min_length=50,
                   max_length=300, quality_threshold=0)
    counts = np.stack([single.upstream, single.downstream], axis=1)
    assert counts.sum() > 0
    for r in range(2):
        assert np.array_equal(np.load(tmp_path / f"m{r}.npy"), counts), r
        v = np.load(tmp_path / f"v{r}.npy")
        assert np.array_equal(v, np.concatenate([single.ocf, single.n_sites.astype(np.float64)]), equal_nan=True), r
    assert open(tmp_path / "o0.tsv").read() == ocf_summary_text(single)   # written by rank 0 only
    assert open(tmp_path / "p0.tsv").read() == ocf_profile_text(single)
    assert not (tmp_path / "o1.tsv").exists() and not (tmp_path / "p1.tsv").exists()
