"""CPU dry run of coverage_profile / multi_coverage_profile and the ``coverage-profile`` command: the public-API
bodies of tests/test_gpu_coverage_profile.py with the kernel wrappers swapped for the oracle (tests/host_shim.py)
and ``device.depth_intervals`` for the numpy definition (tests/depth_oracle.py).  Covers interval handling, BAM
fetch grouping, scaling, writers, errors and the CLI where no GPU exists; the ``-m gpu`` run covers the kernel."""
import inspect

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import bam_replay as R
import depth_oracle as DO
import host_shim
import test_gpu_coverage_profile as G
from helpers import read_gz
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)


def host_depth_intervals(frags, ivl_start, ivl_stop, chrom_size, min_length=None, max_length=None,
                         quality_threshold=30, midpoint=False):
    """Stand-in for ``device.depth_intervals`` on ``host_shim.HostFrags``."""
    fr = frags.fr
    out, off = DO.depth_intervals(fr.start, fr.stop, fr.mapq, ivl_start, ivl_stop, min_length, max_length,
                                  quality_threshold, midpoint)
    return torch.from_numpy(out.astype(np.int32)), off


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200 import device
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    host_shim.install(monkeypatch, {})
    monkeypatch.setattr(device, "depth_intervals", host_depth_intervals)
    yield
    fragments._CACHE.clear()


test_coverage_profile_api = G.test_coverage_profile_api
test_multi_coverage_profile_api = G.test_multi_coverage_profile_api


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_bedgraph_text(syn, tmp_path):
    import finaletoolkit_b200 as F
    bed = tmp_path / "one.bed"; bed.write_text("chrC\t100\t103\n")
    out = str(tmp_path / "one.bed.gz")
    F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file=out, quality_threshold=0)
    lines = read_gz(out).splitlines()
    assert [ln.split("\t")[:3] for ln in lines] == [["chrC", "100", "101"], ["chrC", "101", "102"], ["chrC", "102", "103"]]
    vals = [float(ln.split("\t")[3]) for ln in lines]
    assert all(v == int(v) and ln.endswith(".0") for v, ln in zip(vals, lines))   # depth * 1.0, float64 repr


def test_cli_matches_api(syn, manifest, tmp_path):
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.cli.main_cli import main_cli
    bed = tmp_path / "ivl.bed"; bed.write_text(manifest["cleavage"]["bed"])
    args = [["-q", "0", "--midpoint", "--pad-left", "40", "--pad-right", "7"],
            ["--min-length", "100", "--max-length", "220", "--scale-factor", "3", "-n"],
            ["-t", "4", "-v"]]
    kwargs = [dict(quality_threshold=0, midpoint=True, left=40, right=7),
              dict(min_length=100, max_length=220, scale_factor=3.0, normalize=True),
              dict(workers=4, verbose=1)]
    for j, (a, kw) in enumerate(zip(args, kwargs)):
        cli_out, api_out = str(tmp_path / f"cli{j}.bed.gz"), str(tmp_path / f"api{j}.bed.gz")
        with pytest.warns(UserWarning):
            r = CliRunner().invoke(main_cli, ["coverage-profile", syn["frag"], str(bed), syn["cs"], "-o", cli_out] + a)
        assert r.exit_code == 0, r.output
        with pytest.warns(UserWarning):
            F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file=api_out, **kw)
        assert read_gz(cli_out) == read_gz(api_out), a
    r = CliRunner().invoke(main_cli, ["coverage-profile", syn["frag"], str(bed), syn["cs"], "-o", "x.txt"])
    assert isinstance(r.exception, ValueError)


def test_cli_flags_and_kwargs():
    from finaletoolkit_b200.cli.main_cli import COMMANDS, EXTRA_COMMANDS, main_cli
    from finaletoolkit_b200.frag import multi_coverage_profile
    assert set(EXTRA_COMMANDS) == {"coverage-profile"} and not set(EXTRA_COMMANDS) & set(COMMANDS)
    module, func, _, spec = EXTRA_COMMANDS["coverage-profile"]
    assert (module, func) == ("finaletoolkit_b200.frag", "multi_coverage_profile")
    assert CliRunner().invoke(main_cli, ["coverage-profile", "--help"]).exit_code == 0
    params = {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec}
    accepted = set(inspect.signature(multi_coverage_profile).parameters)
    assert params == accepted
    flags = {f: names[-1] for kind, names, _ in spec if kind == "opt" for f in names[:-1]}
    assert flags == {"-r": "reference_file", "--reference": "reference_file", "-o": "output_file",
                     "--output": "output_file", "--min-length": "min_length", "--max-length": "max_length",
                     "-q": "quality_threshold", "--min-mapq": "quality_threshold", "--pad-left": "left",
                     "--pad-right": "right", "--midpoint": "midpoint", "--scale-factor": "scale_factor",
                     "-n": "normalize", "--normalize": "normalize", "-t": "workers", "--threads": "workers",
                     "-v": "verbose", "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    sig = inspect.signature(multi_coverage_profile).parameters
    for name, d in defaults.items():
        assert sig[name].default == d, name


def test_depth_abi_argument_validation():
    """ftk_depth_tiles_i32 checks its arguments like ftk_cleavage_tiles_f64, before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import lib
    build()
    L = lib()
    assert L.ftk_depth_tiles_i32(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0) == 0           # zero work
    assert L.ftk_depth_tiles_i32(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 3, 0, 0, 0, 1, 0, 0, 0) == -1          # tiles, no tables
    assert L.ftk_depth_tiles_i32(0, 0, 0, 5, 0, 1, 1, 1, 1, 1, 3, 0, 0, 0, 0, 1, 1, 0) == -1          # fragments, no columns
    assert L.ftk_depth_tiles_i32(1, 1, 0, -1, 0, 1, 1, 1, 1, 1, 3, 0, 0, 0, 0, 1, 1, 0) == -1         # n_frag < 0
    assert L.ftk_depth_tiles_i32(1, 1, 0, 5, 0, 1, 1, 1, 1, 1, 2 ** 31, 0, 0, 0, 0, 1, 1, 0) == -3   # too many tiles
