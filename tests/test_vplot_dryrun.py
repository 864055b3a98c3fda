"""CPU dry run of ``vplot`` and the ``vplot`` command: the public-API bodies of tests/test_gpu_vplot.py with the kernel
wrappers swapped for the oracle (tests/host_shim.py) and ``device.vplot_sites`` for the numpy definition
(tests/vplot_oracle.py).  Covers site parsing, BAM fetch grouping, writers, errors, the CLI, the C ABI's argument
checks and a world-size-2 run where no GPU exists; the ``-m gpu`` run covers the kernel."""
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
import test_gpu_vplot as G
import vplot_oracle as VO
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_vplot_sites(frags, site_center, site_flip, flank, min_length, max_length, quality_threshold=30, out=None):
    """Stand-in for ``device.vplot_sites`` on ``host_shim.HostFrags``."""
    from finaletoolkit_b200.device import vplot_check
    vplot_check(flank, min_length, max_length)
    fr = frags.fr
    got = torch.from_numpy(VO.vplot(fr.start, fr.stop, fr.mapq, list(site_center), list(site_flip), int(flank),
                                    int(min_length), int(max_length), quality_threshold))
    return got if out is None else out.add_(got)


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200 import device
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    host_shim.install(monkeypatch, {})
    monkeypatch.setattr(device, "vplot_sites", host_vplot_sites)
    yield
    fragments._CACHE.clear()


test_vplot_api_fx = G.test_vplot_api_fx
test_vplot_api_syn = G.test_vplot_api_syn
test_vplot_errors = G.test_vplot_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_cli_flags_and_kwargs():
    from finaletoolkit_b200.cli.main_cli import COMMANDS, EXTRA_COMMANDS, SITE_COMMANDS, main_cli
    from finaletoolkit_b200.frag import vplot
    assert set(SITE_COMMANDS) == {"vplot"} and not set(SITE_COMMANDS) & (set(COMMANDS) | set(EXTRA_COMMANDS))
    module, func, _, spec = SITE_COMMANDS["vplot"]
    assert (module, func) == ("finaletoolkit_b200.frag", "vplot")
    assert CliRunner().invoke(main_cli, ["vplot", "--help"]).exit_code == 0
    params = {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec}
    sig = inspect.signature(vplot).parameters
    assert params == set(sig)
    flags = {f: names[-1] for kind, names, _ in spec if kind == "opt" for f in names[:-1]}
    assert flags == {"-r": "reference_file", "--reference": "reference_file", "-o": "output_file",
                     "--output": "output_file", "--flank": "flank", "--min-length": "min_length",
                     "--max-length": "max_length", "-q": "quality_threshold", "--min-mapq": "quality_threshold",
                     "-t": "workers", "--threads": "workers", "-v": "verbose", "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    assert defaults.pop("output_file") == "-" and sig["output_file"].default is None   # the CLI writes to stdout
    assert defaults == {"reference_file": None, "flank": 1000, "min_length": 0, "max_length": 500,
                        "quality_threshold": 30, "workers": 1, "verbose": 0}
    for name, d in defaults.items():
        assert sig[name].default == d, name


def test_cli_writes_files(fx, tmp_path):
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.cli.main_cli import main_cli
    bed = tmp_path / "s.bed"; bed.write_text(G._FX_SITES)
    out = str(tmp_path / "cli.tsv")
    r = CliRunner().invoke(main_cli, ["vplot", fx["frag"], str(bed), "-o", out, "--flank", "50", "-q", "0", "-t", "3"])
    assert r.exit_code == 0, r.output
    M = F.vplot(fx["frag"], str(bed), flank=50, quality_threshold=0)
    assert open(out).read() == G.expected_text(M, 50, 0)
    r = CliRunner().invoke(main_cli, ["vplot", fx["frag"], str(bed), "-o", "x.txt"])
    assert isinstance(r.exception, ValueError)


def test_vplot_abi_argument_validation():
    """ftk_vplot_u64 checks its arguments before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import lib
    build()
    f = lib().ftk_vplot_u64
    #       start stop mapq n_frag maxL lo hi flip n_sites flank min max q splits scratch out stream
    assert f(0, 0, 0, 0, 0, 0, 0, 0, 0, 10, 0, 500, 30, 1, 0, 0, 0) == 0             # no sites: zero work
    assert f(1, 1, 0, 0, 0, 1, 1, 1, 3, 10, 0, 500, 30, 1, 1, 1, 0) == 0             # no fragments: zero work
    assert f(0, 0, 0, 0, 0, 0, 0, 0, 3, 10, 0, 500, 30, 1, 0, 0, 0) == -1            # sites, no tables
    assert f(0, 0, 0, 5, 0, 1, 1, 1, 3, 10, 0, 500, 30, 1, 1, 1, 0) == -1            # fragments, no columns
    assert f(1, 1, 0, -1, 0, 1, 1, 1, 3, 10, 0, 500, 30, 1, 1, 1, 0) == -1           # n_frag < 0
    assert f(1, 1, 0, 5, 0, 1, 1, 1, -3, 10, 0, 500, 30, 1, 1, 1, 0) == -1           # n_sites < 0
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, -1, 0, 500, 30, 1, 1, 1, 0) == -1            # flank < 0
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, 10, -1, 500, 30, 1, 1, 1, 0) == -1           # min_len < 0
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, 10, 200, 100, 30, 1, 1, 1, 0) == -1          # max_len < min_len
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, 10, 0, 500, 30, 0, 1, 1, 0) == -1            # splits < 1
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, 2 ** 20 + 1, 0, 0, 30, 1, 1, 1, 0) == -3     # flank > 2^20
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 3, 2 ** 20, 0, 63, 30, 1, 1, 1, 0) == -3        # 64 x 2097153 > 2^27 cells
    assert f(1, 1, 0, 5, 0, 1, 1, 1, 2 ** 30, 10, 0, 500, 30, 4, 1, 1, 0) == -3      # 2^32 units
    assert f(1, 1, 0, 0, 0, 1, 1, 1, 3, 2 ** 20, 0, 62, 30, 1, 1, 1, 0) == 0         # 63 x 2097153 cells fit


_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
repo = os.environ["FTK_REPO"]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from _pytest.monkeypatch import MonkeyPatch
import host_shim
import test_vplot_dryrun as VD
import finaletoolkit_b200 as F
import finaletoolkit_b200.device as D
mp = MonkeyPatch()
host_shim.install(mp, {})
mp.setattr(D, "vplot_sites", VD.host_vplot_sites)
mp.setattr(D, "require_cuda", lambda device=None: torch.device("cpu"))
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank = dist.get_rank()
d = os.environ["FTK_DIR"]
M = F.vplot(os.path.join(d, "read1.bam"), os.path.join(d, "sites.bed"), output_file=os.path.join(d, "v%d.tsv" % rank),
            flank=150, min_length=50, max_length=300, quality_threshold=0)
from finaletoolkit_b200.distributed import owned_contigs
from finaletoolkit_b200.io.fragments import load_fragments
np.save(os.path.join(d, "m%d.npy" % rank), M)   # a file, not stdout: the matrix would fill the pipe before the barrier
print(json.dumps({"rank": rank, "mine": owned_contigs(load_fragments(os.path.join(d, "read1.bam")))}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2(tmp_path, golden):
    import finaletoolkit_b200 as F
    bam = R.make_fixture(tmp_path, golden)
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    (tmp_path / "sites.bed").write_text("".join(f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n" for k, t in enumerate(tiles)))
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(33500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", FTK_REPO=REPO, FTK_PORT=port, FTK_DIR=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-2000:] for o in outs]
    got = [json.loads(o[0].strip().splitlines()[-1]) for o in outs]
    assert sorted(got[0]["mine"] + got[1]["mine"]) == ["chrA", "chrB"] and got[0]["mine"] and got[1]["mine"]
    single = F.vplot(bam["path"], str(tmp_path / "sites.bed"), flank=150, min_length=50, max_length=300,
                     quality_threshold=0)
    assert single.sum() > 0
    for r in range(2):
        assert np.array_equal(np.load(tmp_path / f"m{r}.npy"), single), r
    assert open(tmp_path / "v0.tsv").read() == G.expected_text(single, 150, 50)   # written by rank 0 only
    assert not (tmp_path / "v1.tsv").exists()
