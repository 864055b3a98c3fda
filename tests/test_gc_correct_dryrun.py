"""CPU dry run of ``gc_corrected_coverage`` / ``gc_corrected_profile`` and their commands: the public-API bodies of
tests/test_gpu_gc_correct.py with the kernel wrappers swapped for the numpy definitions (tests/gc_correct_oracle.py,
tests/gc_oracle.py) through tests/host_shim.py.  Also covers the ``read_gc_bias`` round trip, the CLI table, the C
ABI's argument checks and a world-size-2 run where no GPU exists; the ``-m gpu`` run covers the kernels."""
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
import gc_correct_oracle as CO
import test_gc_bias_dryrun as GD
import test_gpu_gc_correct as G

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _w(weights):
    return weights.cpu().numpy() if torch.is_tensor(weights) else np.asarray(weights, np.float64)


def _into(out, got):
    if out is None:
        return got
    out[0].add_(got[0]); out[1].add_(got[1])
    return out


def host_gc_weighted_intervals(frags, ref, ivl_start, ivl_stop, weights, min_length, max_length, quality_threshold=30,
                               out=None):
    from finaletoolkit_b200.device import gc_check
    gc_check(min_length, max_length)
    fr = frags.fr
    c, w = CO.intervals(fr.start, fr.stop, fr.mapq, ref.codes, ref.nmask, ref.length, list(ivl_start), list(ivl_stop),
                        _w(weights), int(min_length), int(max_length), quality_threshold)
    return _into(out, (torch.from_numpy(c), torch.from_numpy(w)))


def host_gc_weighted_sites(frags, ref, site_center, site_flip, flank, weights, min_length, max_length,
                           quality_threshold=30, out=None):
    from finaletoolkit_b200.device import gc_check
    gc_check(min_length, max_length)
    fr = frags.fr
    c, w = CO.sites(fr.start, fr.stop, fr.mapq, ref.codes, ref.nmask, ref.length, list(site_center), list(site_flip),
                    int(flank), _w(weights), int(min_length), int(max_length), quality_threshold)
    return _into(out, (torch.from_numpy(c), torch.from_numpy(w)))


def install(monkeypatch):
    from finaletoolkit_b200 import device
    GD.install(monkeypatch)
    monkeypatch.setattr(device, "gc_weighted_intervals", host_gc_weighted_intervals)
    monkeypatch.setattr(device, "gc_weighted_sites", host_gc_weighted_sites)


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    install(monkeypatch)
    yield
    fragments._CACHE.clear()


test_api_models_text_and_cli = G.test_api_models_text_and_cli
test_api_errors = G.test_api_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_read_gc_bias_round_trip(tmp_path):
    from finaletoolkit_b200.frag import read_gc_bias
    from finaletoolkit_b200.frag._gc_bias import GCBias, gc_ratio, gc_text
    from finaletoolkit_b200.frag._gc_correct import gc_weights
    rng = np.random.default_rng(3)
    lo, hi = 3, 40
    O = rng.integers(0, 50, (hi - lo + 1, hi + 1)); E = rng.integers(0, 7, O.shape) * rng.integers(0, 2, O.shape)
    for i in range(O.shape[0]):
        O[i, lo + i + 1:] = 0; E[i, lo + i + 1:] = 0
    O[5] = 0
    res = GCBias(O, E, gc_ratio(O, E), lo, hi)
    assert np.isnan(res.ratio).any() and (res.ratio == 0).any()
    for name in ("m.tsv", "m.tsv.gz"):
        path = tmp_path / name
        from finaletoolkit_b200.frag._common import write_text
        write_text(str(path), gc_text(res))
        back = read_gc_bias(path)
        assert (back.min_length, back.max_length) == (lo, hi)
        assert np.array_equal(back.observed, O) and np.array_equal(back.expected, E)
        assert np.array_equal(back.ratio, res.ratio, equal_nan=True)
        assert np.array_equal(gc_weights(back), gc_weights(res)) and np.array_equal(gc_weights(res), CO.weights(res.ratio))
        assert gc_text(back) == gc_text(res)
    good = gc_text(res).splitlines()
    bad_tables = ["", "length\tgc\tobserved\n", good[0] + "\n",
                  "\n".join(good[:-1]) + "\n",                                  # a row short
                  "\n".join(good[:1] + good[2:] + good[1:2]) + "\n",            # rows out of order
                  "\n".join(good + ["40\t40\t1\t1\t1.0"]) + "\n",              # a row extra
                  "\n".join(good[:3] + ["3\t2\tx\t1\t1.0"] + good[4:]) + "\n",  # not an integer
                  "\n".join(good[:3] + ["3\t2\t1\t1"] + good[4:]) + "\n",       # a column short
                  "length\tgc\tobserved\texpected\tratio\n0\t0\t1\t1\t1.0\n"]    # length 0
    for k, text in enumerate(bad_tables):
        (tmp_path / "bad.tsv").write_text(text)
        with pytest.raises(ValueError):
            read_gc_bias(tmp_path / "bad.tsv")


def test_cli_table_and_flags():
    from finaletoolkit_b200.cli.main_cli import (BIAS_COMMANDS, COMMANDS, CORRECTION_COMMANDS, EXTRA_COMMANDS,
                                                 SITE_COMMANDS, main_cli)
    from finaletoolkit_b200 import frag
    assert set(CORRECTION_COMMANDS) == {"gc-corrected-coverage", "gc-corrected-profile"}
    assert not set(CORRECTION_COMMANDS) & (set(COMMANDS) | set(EXTRA_COMMANDS) | set(SITE_COMMANDS) | set(BIAS_COMMANDS))
    common = {"-r": "reference_file", "--reference": "reference_file", "-o": "output_file", "--output": "output_file",
              "--gc-bias": "gc_bias", "--gc-regions": "gc_regions", "--min-length": "min_length",
              "--max-length": "max_length", "-q": "quality_threshold", "--min-mapq": "quality_threshold",
              "-t": "workers", "--threads": "workers", "-v": "verbose", "--verbose": "verbose"}
    for name, func, extra in (("gc-corrected-coverage", "gc_corrected_coverage", {}),
                              ("gc-corrected-profile", "gc_corrected_profile", {"--flank": "flank"})):
        module, f, _, spec = CORRECTION_COMMANDS[name]
        assert (module, f) == ("finaletoolkit_b200.frag", func)
        assert CliRunner().invoke(main_cli, [name, "--help"]).exit_code == 0
        sig = inspect.signature(getattr(frag, func)).parameters
        assert {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec} == set(sig)
        assert {fl: names[-1] for kind, names, _ in spec if kind == "opt" for fl in names[:-1]} == {**common, **extra}
        defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
        assert defaults.pop("output_file") == "-" and sig["output_file"].default is None   # the CLI writes to stdout
        for k, d in defaults.items():
            assert sig[k].default == d, (name, k)


def test_weighted_abi_argument_validation():
    """ftk_gc_weighted_intervals_f64 / ftk_gc_weighted_sites_f64 check their arguments before touching CUDA."""
    from finaletoolkit_b200.csrc.build import build
    from finaletoolkit_b200._lib import lib
    build()
    iv, si = lib().ftk_gc_weighted_intervals_f64, lib().ftk_gc_weighted_sites_f64
    #      st sp mq n_frag maxL seq nm clen lo hi n min max q splits scratch w cnt corr stream
    ok = [8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 3, 50, 500, 30, 1, 8, 8, 8, 8, 0]

    def I(**kw):
        a = list(ok)
        for k, v in kw.items():
            a[int(k[1:])] = v
        return iv(*a)
    assert I(a10=0, a0=0, a1=0, a5=0, a16=0) == 0          # no intervals: zero work
    assert I(a3=0) == 0                                     # no fragments: zero work
    assert I(a3=0, a5=4) == -1                              # ... but the arguments are still checked
    for k, v in [(0, 0), (1, 0), (3, -1), (5, 0), (6, 0), (5, 4), (7, -1), (8, 0), (9, 0), (10, -3), (11, 0),
                 (12, 40), (14, 0), (15, 0), (16, 0), (17, 0), (18, 0)]:
        assert I(**{f"a{k}": v}) == -1, k                   # FTK_E_INVALID
    for k, v in [(12, 1025), (7, 2 ** 31), (10, 2 ** 30)]:
        assert I(**{f"a{k}": v}) == -3, k                   # FTK_E_RANGE
    assert I(a10=2 ** 20, a14=4096) == -3                   # 2^32 units
    #        st sp mq n_frag maxL seq nm clen lo hi flip n flank min max q splits scratch w cnt corr stream
    sok = [8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 8, 3, 1000, 50, 500, 30, 1, 8, 8, 8, 8, 0]

    def S(**kw):
        a = list(sok)
        for k, v in kw.items():
            a[int(k[1:])] = v
        return si(*a)
    assert S(a11=0, a0=0, a10=0, a18=0) == 0                # no sites: zero work
    assert S(a3=0) == 0
    for k, v in [(0, 0), (3, -1), (5, 0), (5, 4), (8, 0), (10, 0), (11, -1), (12, -1), (13, 0), (14, 40), (16, 0),
                 (17, 0), (18, 0), (19, 0), (20, 0)]:
        assert S(**{f"a{k}": v}) == -1, k
    for k, v in [(12, 2 ** 20 + 1), (14, 1025), (7, 2 ** 31), (11, 2 ** 30)]:
        assert S(**{f"a{k}": v}) == -3, k


_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
repo = os.environ["FTK_REPO"]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from _pytest.monkeypatch import MonkeyPatch
import test_gc_correct_dryrun as CD
import finaletoolkit_b200 as F
mp = MonkeyPatch()
CD.install(mp)
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank = dist.get_rank()
d = os.environ["FTK_DIR"]
bam, tb = os.path.join(d, "read1.bam"), os.path.join(d, "read1.2bit")
r = F.gc_corrected_coverage(bam, tb, os.path.join(d, "ivl.bed"), output_file=os.path.join(d, "c%d.tsv" % rank),
                            min_length=50, max_length=300, quality_threshold=0)
p = F.gc_corrected_profile(bam, tb, os.path.join(d, "sites.bed"), output_file=os.path.join(d, "p%d.tsv" % rank),
                           flank=300, min_length=50, max_length=300, quality_threshold=0)
np.save(os.path.join(d, "pc%d.npy" % rank), p.count); np.save(os.path.join(d, "pw%d.npy" % rank), p.corrected)
print(json.dumps({"rank": rank, "rows": [list(x) for x in r], "n_sites": p.n_sites}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2(tmp_path, golden):
    import finaletoolkit_b200 as F
    bam = R.make_fixture(tmp_path, golden)
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    (tmp_path / "ivl.bed").write_text("".join(f"{t[0]}\t{t[1]}\t{t[2]}\tt{k}\n" for k, t in enumerate(tiles[::2])))
    (tmp_path / "sites.bed").write_text("".join(f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n"
                                                for k, t in enumerate(tiles[::3])))
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(37500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", FTK_REPO=REPO, FTK_PORT=port, FTK_DIR=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-2000:] for o in outs]
    got = [json.loads(o[0].strip().splitlines()[-1]) for o in outs]
    kw = dict(min_length=50, max_length=300, quality_threshold=0)
    single = F.gc_corrected_coverage(bam["path"], bam["tb"], str(tmp_path / "ivl.bed"), **kw)
    prof = F.gc_corrected_profile(bam["path"], bam["tb"], str(tmp_path / "sites.bed"), flank=300, **kw)
    assert sum(x.count for x in single) > 0 and prof.corrected.sum() > 0
    for r in range(2):
        assert [tuple(x) for x in got[r]["rows"]] == [tuple(x) for x in single], r   # bit-identical per interval
        assert got[r]["n_sites"] == prof.n_sites
        assert np.array_equal(np.load(tmp_path / f"pc{r}.npy"), prof.count)
        assert np.allclose(np.load(tmp_path / f"pw{r}.npy"), prof.corrected, rtol=1e-12, atol=0)
    assert open(tmp_path / "c0.tsv").read() == CO.coverage_text(single)
    assert (tmp_path / "p0.tsv").exists() and not (tmp_path / "c1.tsv").exists() and not (tmp_path / "p1.tsv").exists()
