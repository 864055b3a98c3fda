"""CPU dry run of ``gc_corrected_coverage_profile`` / ``multi_gc_corrected_coverage_profile`` and the
``gc-corrected-coverage-profile`` command: the public-API bodies of tests/test_gpu_gc_track.py with the kernel
wrappers swapped for the numpy definitions (tests/gc_track_oracle.py, and those of the GC-correction dry run).  Also
covers the CLI table and the C ABI's argument checks where no GPU exists; the ``-m gpu`` run covers the kernel."""
import inspect

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import bam_replay as R
import gc_track_oracle as TO
import test_gc_correct_dryrun as CD
import test_gpu_gc_track as G


def host_gc_depth_intervals(frags, ref, ivl_start, ivl_stop, chrom_size, weights, min_length, max_length,
                            quality_threshold=30, midpoint=False):
    """Stand-in for ``device.gc_depth_intervals`` on ``host_shim.HostFrags`` and ``HostRef``."""
    from finaletoolkit_b200.device import gc_check, gc_quantise_weights
    gc_quantise_weights(weights, gc_check(min_length, max_length))   # the device layer's checks
    fr = frags.fr
    out, off = TO.track_intervals(fr.start, fr.stop, fr.mapq, ref.codes, ref.nmask, ref.length, list(ivl_start),
                                  list(ivl_stop), CD._w(weights), int(min_length), int(max_length), quality_threshold,
                                  midpoint)
    return torch.from_numpy(out), off


@pytest.fixture(autouse=True)
def _oracle_device_layer(monkeypatch):
    from finaletoolkit_b200 import device
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    CD.install(monkeypatch)
    monkeypatch.setattr(device, "gc_depth_intervals", host_gc_depth_intervals)
    yield
    fragments._CACHE.clear()


test_api_models_text_and_cli = G.test_api_models_text_and_cli
test_api_errors = G.test_api_errors


def test_bam_fetch_semantics(tmp_path, golden):
    G.check_bam(R.make_fixture(tmp_path, golden))


def test_quantisation():
    """rint(W * 2^32) with ties to even; 2^30 and more refused."""
    from finaletoolkit_b200.device import gc_quantise_weights
    W = np.array([[0.0, 1.0, 2.0 ** -33, 3 * 2.0 ** -33, 2.0 ** 30 - 2.0 ** -20, 1 / 3]])
    q = gc_quantise_weights(W, W.shape)
    assert q.dtype == np.int64
    assert q.tolist() == [[0, 2 ** 32, 0, 2, 2 ** 62 - 2 ** 12, 1431655765]]
    assert np.array_equal(gc_quantise_weights(torch.from_numpy(W), W.shape), q)
    with pytest.raises(ValueError):
        gc_quantise_weights(np.full((1, 1), 2.0 ** 30), (1, 1))


def test_cli_table_and_flags():
    import importlib
    from finaletoolkit_b200 import frag
    M = importlib.import_module("finaletoolkit_b200.cli.main_cli")
    assert set(M.GC_TRACK_COMMANDS) == {"gc-corrected-coverage-profile"}
    others = [M.COMMANDS, M.EXTRA_COMMANDS, M.SITE_COMMANDS, M.BIAS_COMMANDS, M.CORRECTION_COMMANDS,
              M.SPECTRUM_COMMANDS, M.ORIENTATION_COMMANDS]
    assert not any(set(M.GC_TRACK_COMMANDS) & set(t) for t in others)
    module, func, _, spec = M.GC_TRACK_COMMANDS["gc-corrected-coverage-profile"]
    assert (module, func) == ("finaletoolkit_b200.frag", "multi_gc_corrected_coverage_profile")
    assert CliRunner().invoke(M.main_cli, ["gc-corrected-coverage-profile", "--help"]).exit_code == 0
    sig = inspect.signature(frag.multi_gc_corrected_coverage_profile).parameters
    assert {names[-1] if kind == "opt" else names[0] for kind, names, _ in spec} == set(sig)
    assert [names[0] for kind, names, _ in spec if kind == "arg"] == ["input_file", "refseq_file", "interval_file",
                                                                      "chrom_sizes"]
    assert {fl: names[-1] for kind, names, _ in spec if kind == "opt" for fl in names[:-1]} == {
        "-r": "reference_file", "--reference": "reference_file", "-o": "output_file", "--output": "output_file",
        "--gc-bias": "gc_bias", "--gc-regions": "gc_regions", "--min-length": "min_length",
        "--max-length": "max_length", "-q": "quality_threshold", "--min-mapq": "quality_threshold",
        "--pad-left": "left", "--pad-right": "right", "--midpoint": "midpoint", "--scale-factor": "scale_factor",
        "-n": "normalize", "--normalize": "normalize", "-t": "workers", "--threads": "workers", "-v": "verbose",
        "--verbose": "verbose"}
    defaults = {names[-1]: kw.get("default") for kind, names, kw in spec if kind == "opt" and "default" in kw}
    for k, d in defaults.items():
        assert sig[k].default == d, k


def test_gc_depth_abi_argument_validation():
    """ftk_gc_depth_tiles_f64 checks its arguments before touching CUDA."""
    from finaletoolkit_b200._lib import lib
    from finaletoolkit_b200.csrc.build import build
    build()
    f = lib().ftk_gc_depth_tiles_f64
    #     st sp mq n maxL seq nm clen p0 len lo hi off n_tiles min max q mid w maxw scratch flag out stream
    ok = [8, 8, 0, 5, 0, 8, 8, 100, 8, 8, 8, 8, 8, 3, 50, 500, 30, 0, 8, 2 ** 32, 8, 8, 8, 0]

    def F(**kw):
        a = list(ok)
        for k, v in kw.items():
            a[int(k[1:])] = v
        return f(*a)
    assert F(a13=0, a0=0, a5=0, a18=0, a21=0) == 0                 # no tiles: zero work
    for k, v in [(0, 0), (1, 0), (3, -1), (5, 0), (5, 4), (6, 0), (7, -1), (8, 0), (12, 0), (13, -2), (14, 0),
                 (15, 40), (18, 0), (19, -1), (20, 0), (21, 0), (22, 0), (22, 12)]:
        assert F(**{f"a{k}": v}) == -1, k                             # FTK_E_INVALID
    for k, v in [(15, 1025), (7, 2 ** 31), (19, 2 ** 62), (13, 2 ** 31)]:
        assert F(**{f"a{k}": v}) == -3, k                             # FTK_E_RANGE
