"""CPU dry run of ``wps_spectrum``, the ``wps-spectrum`` command and ``distributed.wps_spectrum_genome``: the
public-API bodies of tests/test_gpu_spectrum.py with ``device.spectrum_segments`` swapped for the numpy direct sum
(tests/spectrum_oracle.py) and the WPS / adjust wrappers for the oracle (tests/host_shim.py).  Also covers the CLI
table, the C ABI's argument checks and a world-size-2 run where no GPU exists; the ``-m gpu`` run covers the kernel."""
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
import spectrum_oracle as SO
import test_gc_bias_dryrun as GD
import test_gpu_spectrum as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_spectrum_segments(x, offsets, min_period=120, max_period=280, out=None):
    from finaletoolkit_b200.device import spectrum_check
    n_p = spectrum_check(min_period, max_period)
    x = np.asarray(x.cpu() if torch.is_tensor(x) else x)
    off = np.asarray(offsets, np.int64)
    rows = [SO.spectrum(x[a:b], int(min_period), int(max_period)) for a, b in zip(off[:-1], off[1:])]
    return torch.from_numpy(np.array(rows, np.float64).reshape(len(rows), n_p))


def install(monkeypatch):
    from finaletoolkit_b200 import device
    GD.install(monkeypatch)
    monkeypatch.setattr(device, "spectrum_segments", host_spectrum_segments)


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    install(monkeypatch)
    yield
    fragments._CACHE.clear()


test_api_text_and_cli = G.test_api_text_and_cli
test_api_errors = G.test_api_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_genome_driver_body():
    """Adjusted series when the results hold them, the raw WPS otherwise; empty series give NaN rows."""
    from finaletoolkit_b200.distributed import ContigWps, wps_spectrum_genome
    rng = np.random.default_rng(5)
    off = np.array([0, 3000, 3000, 4500], np.int64)
    raw = ContigWps("a", None, None, off, torch.from_numpy(rng.integers(-50, 50, 4500).astype(np.int32)))
    adj = ContigWps("b", None, None, off, torch.from_numpy(rng.integers(-50, 50, 4500).astype(np.int32)))
    adj.adj_offsets = np.array([0, 2000, 2000, 2500], np.int64)
    adj.adjusted = torch.from_numpy(rng.normal(size=2500))
    short = ContigWps("c", None, None, off, torch.from_numpy(np.zeros(4500, np.int32)))
    short.adj_offsets = np.zeros(4, np.int64)
    got = wps_spectrum_genome({"a": raw, "b": adj, "c": short}, 130, 250)
    for k in range(3):
        SO.check_row(got["a"][k].numpy(), raw.wps.numpy()[off[k]: off[k + 1]], 130, 250)
        SO.check_row(got["b"][k].numpy(), adj.adjusted.numpy()[adj.adj_offsets[k]: adj.adj_offsets[k + 1]], 130, 250)
    assert np.isnan(got["a"][1].numpy()).all() and np.isnan(got["c"].numpy()).all()
    lost = ContigWps("d", None, None, off, raw.wps)
    lost.adj_offsets = adj.adj_offsets
    with pytest.raises(ValueError):
        wps_spectrum_genome({"d": lost})
    with pytest.raises(ValueError):
        wps_spectrum_genome({"a": raw}, 2, 1025)


def test_output_lengths_match_adjust_plan():
    """The series lengths wps_spectrum reports are the outputs AdjustPlan(skip_short=True) plans."""
    from finaletoolkit_b200.device import AdjustPlan
    seg = np.array([0, 1, 999, 1000, 1001, 1020, 1021, 1022, 5000])
    plan = AdjustPlan(seg, 1000, True, 21, 2, skip_short=True)
    assert list(plan.n_out) == list(AdjustPlan.output_lengths(seg, 1000, True, 21)) == [0, 0, 0, 0, 0, 0, 21, 22, 4000]
    assert list(AdjustPlan.output_lengths(seg, 1000, False, 21)) == [0, 0, 0, 0, 1, 20, 21, 22, 4000]


def test_cli_table_and_flags():
    from finaletoolkit_b200.cli.main_cli import (BIAS_COMMANDS, COMMANDS, CORRECTION_COMMANDS, EXTRA_COMMANDS,
                                                 SITE_COMMANDS, SPECTRUM_COMMANDS, main_cli)
    from finaletoolkit_b200 import frag
    assert set(SPECTRUM_COMMANDS) == {"wps-spectrum"}
    assert not set(SPECTRUM_COMMANDS) & (set(COMMANDS) | set(EXTRA_COMMANDS) | set(SITE_COMMANDS) | set(BIAS_COMMANDS)
                                         | set(CORRECTION_COMMANDS))
    module, f, _, spec = SPECTRUM_COMMANDS["wps-spectrum"]
    assert (module, f) == ("finaletoolkit_b200.frag", "wps_spectrum")
    assert CliRunner().invoke(main_cli, ["wps-spectrum", "--help"]).exit_code == 0
    sig = inspect.signature(frag.wps_spectrum).parameters
    named = {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec}
    assert named == set(sig) - {"fraction_low", "fraction_high"}
    assert {fl: names[-1] for kind, names, _ in spec if kind == "opt" for fl in names[:-1]} == {
        "-r": "reference_file", "--reference": "reference_file", "--chrom-sizes": "chrom_sizes", "-o": "output_file",
        "--output": "output_file", "--min-period": "min_period", "--max-period": "max_period",
        "--adjust/--no-adjust": "adjust", "-m": "median_window_size", "--median-window-size": "median_window_size",
        "--savgol/--no-savgol": "savgol", "--savgol-window-size": "savgol_window_size",
        "--savgol-poly-deg": "savgol_poly_deg", "-W": "window_size", "--window-size": "window_size",
        "--min-length": "min_length", "--max-length": "max_length", "-q": "quality_threshold",
        "--min-mapq": "quality_threshold", "-t": "workers", "--threads": "workers", "-v": "verbose",
        "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    assert defaults.pop("output_file") == "-" and sig["output_file"].default is None   # the CLI writes to stdout
    for k, d in defaults.items():
        assert sig[k].default == d, k


def test_spectrum_abi_argument_validation():
    """ftk_spectrum_i32_f64 / ftk_spectrum_f64_f64 check their arguments before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import lib
    build()
    for fn in (lib().ftk_spectrum_i32_f64, lib().ftk_spectrum_f64_f64):
        #      x  off n_seg lo  hi  out stream
        ok = [8, 8, 0, 120, 280, 8, 0]

        def call(**kw):
            a = list(ok)
            for k, v in kw.items():
                a[int(k[1:])] = v
            return fn(*a)
        assert call() == 0                                     # no segments: no launch
        assert call(a3=2, a4=2) == 0 and call(a3=2, a4=1024) == 0
        for k, v in [(0, 0), (1, 0), (5, 0), (2, -1), (3, 1), (3, 281), (4, 119)]:
            assert call(**{f"a{k}": v}) == -1, k               # FTK_E_INVALID
        assert call(a4=1025) == -3                             # FTK_E_RANGE
        assert call(a2=2 ** 31, a3=120, a4=280) == -3          # more CTAs than a grid holds
        assert call(a2=2 ** 27, a3=2, a4=1024) == -3


_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
repo = os.environ["FTK_REPO"]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from _pytest.monkeypatch import MonkeyPatch
import test_spectrum_dryrun as SD
import finaletoolkit_b200 as F
mp = MonkeyPatch()
SD.install(mp)
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank = dist.get_rank()
d = os.environ["FTK_DIR"]
r = F.wps_spectrum(os.path.join(d, "read1.bam"), os.path.join(d, "w.bed"), output_file=os.path.join(d, "s%d.tsv" % rank),
                   min_length=100, max_length=220, min_period=150, max_period=200)
np.save(os.path.join(d, "i%d.npy" % rank), r.intensity)
print(json.dumps({"rank": rank, "n": r.n.tolist()}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2(tmp_path, golden):
    import finaletoolkit_b200 as F
    bam = R.make_fixture(tmp_path, golden)
    rows = ["chrA\t0\t12000\ta\n", "chrB\t100\t20000\tb\n", "chrA\t30000\t45000\tc\n", "chrB\t24000\t30000\td\n",
            "chrQ\t0\t5000\tq\n", "chrA\t5000\t5500\te\n"]
    (tmp_path / "w.bed").write_text("".join(rows))
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(38500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", FTK_REPO=REPO, FTK_PORT=port, FTK_DIR=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-2000:] for o in outs]
    got = [json.loads(o[0].strip().splitlines()[-1]) for o in outs]
    single = F.wps_spectrum(bam["path"], str(tmp_path / "w.bed"), min_length=100, max_length=220, min_period=150,
                            max_period=200)
    assert list(single.n) == [11000, 18900, 14000, 0, 0, 0]
    assert np.nansum(single.intensity[:3]) > 0 and np.isnan(single.intensity[3:]).all()
    for r in range(2):
        assert got[r]["n"] == single.n.tolist()
        assert np.array_equal(np.load(tmp_path / f"i{r}.npy").view(np.int64), single.intensity.view(np.int64)), r
    assert open(tmp_path / "s0.tsv").read() == SO.text(single.intervals, single.n, single.periods, single.intensity)
    assert not (tmp_path / "s1.tsv").exists()
