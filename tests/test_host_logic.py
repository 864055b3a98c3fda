"""CPU-only tests: host logic of the product, the C ABI surface, and the N>1 sharding path (gloo)."""
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

from helpers import write_2bit, write_text_gz
from oracle import oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_library_exports_every_declared_symbol():
    """include/ftk_b200.h <-> libftk_b200.so <-> the ctypes table (no compute calls)."""
    from finaletoolkit_b200 import _lib
    from finaletoolkit_b200.csrc.build import build
    build()
    hdr = open(os.path.join(REPO, "include", "ftk_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(ftk_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    h = _lib.lib()
    for name in declared:
        assert hasattr(h, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    assert h.ftk_abi_version() == 2
    assert h.ftk_error_string(-1) == b"invalid argument"
    # the host-only planner is callable without a GPU
    import ctypes
    s = np.array([0, 10_000, 7], np.int64); e = np.array([5000, 22_000, 7], np.int64); off = np.array([0, 5000, 17000], np.int64)
    p = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))
    n = h.ftk_wps_plan_tiles(p(s, ctypes.c_int64), p(e, ctypes.c_int64), p(off, ctypes.c_int64), 3, 100_000, 180,
                             None, None, None, None, None)
    assert n == 1 + 3  # 5000 -> 1 tile, 12000 -> 3 tiles, degenerate -> 0


def test_no_cpu_fallback():
    """Without CUDA every feature fails loudly instead of computing on the host.  On a machine with a GPU
    the checks run in a child process that sees no device."""
    import torch
    if not torch.cuda.is_available():
        _check_no_cpu_fallback()
        return
    code = (f"import sys; sys.path[:0] = {[REPO, os.path.join(REPO, 'tests')]!r}\n"
            "import test_host_logic as t; t._check_no_cpu_fallback(); print('no cpu fallback ok')")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "no cpu fallback ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def _check_no_cpu_fallback():
    import torch
    assert not torch.cuda.is_available()
    import finaletoolkit_b200 as F
    from finaletoolkit_b200._lib import FtkLibraryError
    cols = {"c": (np.array([1, 5]), np.array([150, 170]), np.array([60, 60]), np.array([1, 0]))}
    with pytest.raises(FtkLibraryError):
        F.wps(cols, "c", 0, 100, 1000)
    with pytest.raises(FtkLibraryError):
        F.single_coverage(cols, "c", 0, 100)
    with pytest.raises(FtkLibraryError):
        F.frag_length_bins(cols)


def test_product_never_imports_oracle():
    for root, _, files in os.walk(os.path.join(REPO, "finaletoolkit_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|ftk_oracle|libftk_oracle", txt, flags=re.M), \
                    f"{f} references the oracle"


def test_read_sites_matches_oracle(tmp_path, manifest):
    from finaletoolkit_b200.frag._multi_wps import _read_sites
    from finaletoolkit_b200.frag._adjust_wps import _read_adjust_sites
    m = manifest["synth_small"]
    sizes = dict(m["contigs"])
    bed = tmp_path / "s.bed"; bed.write_text(m["sites_bed"])
    for isz in (5000, 2000, 600, 2):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            c, s, e = _read_sites(str(bed), isz, list(sizes), sizes)
        order = {k: i for i, k in enumerate(sizes)}
        got = sorted(zip(c, s, e), key=lambda t: (order[t[0]], t[1]))
        assert got == O.read_sites(m["sites_bed"].splitlines(), isz, sizes)
    ab = tmp_path / "a.bed"; ab.write_text(manifest["adjust"]["tile_bed"])
    assert _read_adjust_sites(str(ab), 5000, 1000) == O.adjust_sites(manifest["adjust"]["tile_bed"].splitlines(keepends=True), 5000, 1000)
    with pytest.raises(ValueError):
        _read_adjust_sites("x.txt", 5000, 1000)


def test_fragment_loader(tmp_path, manifest):
    from finaletoolkit_b200.exceptions import MissingIndexError, UnsupportedFormatError
    from finaletoolkit_b200.io import load_fragments
    m = manifest["fixture17"]
    p = write_text_gz(tmp_path / "a.frag.gz", m["frag_gz_text"])
    t = load_fragments(p)
    assert t.contigs == ["12"] and t.n_fragments() == 17
    st, sp, mq, sd = t.host("12")
    assert st[0] == 34443118 and sp[0] == 34443284 and mq[4] == 54 and sd[3] == 0 and st.dtype == np.int32
    assert load_fragments(p) is t  # cached
    # malformed rows are skipped, BED6 is detected with a warning
    bad = m["frag_gz_text"].splitlines()
    bad.insert(2, "12\tx\t5\t60\t+"); bad.insert(5, "12\t7")
    t2 = load_fragments(write_text_gz(tmp_path / "b.frag.gz", "\n".join(bad) + "\n"))
    assert t2.n_fragments() == 17
    with pytest.warns(UserWarning):
        assert load_fragments(write_text_gz(tmp_path / "c.bed.gz", m["frag_bed_gz_text"])).n_fragments() == 17
    with pytest.raises(FileNotFoundError):
        load_fragments(str(tmp_path / "missing.frag.gz"))
    (tmp_path / "noidx.frag.gz").write_bytes(open(p, "rb").read())
    with pytest.raises(MissingIndexError):
        load_fragments(str(tmp_path / "noidx.frag.gz"))
    (tmp_path / "x.txt").write_text("hi")
    with pytest.raises(UnsupportedFormatError):
        load_fragments(str(tmp_path / "x.txt"))


def test_reference_wrapper(tmp_path):
    from finaletoolkit_b200.exceptions import ContigNotFoundError, OutOfBoundsError
    from finaletoolkit_b200.io import ReferenceWrapper
    from finaletoolkit_b200.synth import pack_twobit, synth_twobit
    codes, nm = synth_twobit(5003, 0, telomere=100, n_blocks=2, block_len=50)
    tb = write_2bit(tmp_path / "r.2bit", [("chrZ", codes, nm), ("s", codes[:7], nm[:7] & False)])
    r = ReferenceWrapper(tb)
    assert r.chroms == {"chrZ": 5003, "s": 7}
    seq = np.frombuffer(b"ACGT", np.uint8)[codes].copy(); seq[nm] = ord("N")
    assert r.sequence("chrZ") == seq.tobytes().decode() and r.sequence("chrZ", 120, 131) == seq[120:131].tobytes().decode()
    assert r["chrZ"][200:204] == seq[200:204].tobytes().decode() and len(r["chrZ"]) == 5003
    with pytest.raises(OutOfBoundsError):
        r.sequence("chrZ", 5000, 5004)
    assert r.sequence("chrZ", 5000, 5004, fail_on_excess_range=False) == seq[5000:5003].tobytes().decode()
    with pytest.raises(ContigNotFoundError):
        r.sequence("nope", 0, 1)
    with pytest.raises(FileNotFoundError):
        ReferenceWrapper(str(tmp_path / "none.2bit"))
    fa = tmp_path / "r.fa"
    fa.write_text(">chrZ desc\n" + "\n".join(seq.tobytes().decode()[i:i + 60] for i in range(0, 5003, 60)) + "\n")
    f = ReferenceWrapper(str(fa))
    assert f.chroms == {"chrZ": 5003} and f.sequence("chrZ", 90, 140) == r.sequence("chrZ", 90, 140)
    # device packing layout: base i at bits 2*(i%16) of word i//16, N bit i%32 of word i//32
    sw, nw = pack_twobit(codes, nm)
    i = np.arange(5003)
    assert np.array_equal((sw[i // 16] >> (2 * (i % 16))) & 3, codes) and np.array_equal((nw[i // 32] >> (i % 32)) & 1, nm.astype(np.uint32))


def test_bigwig_roundtrip_and_real_file_layout(tmp_path):
    from finaletoolkit_b200.io import bigwig
    p = str(tmp_path / "a.bw")
    rng = np.random.default_rng(1)
    v = rng.integers(-40, 40, 100_000).astype(np.float64)
    with bigwig.open(p, "w") as w:
        w.addHeader([("2", 5_000_000), ("10", 4_000_000)])
        w.addEntries("2", 123, values=v, span=1, step=1)
        w.addEntries("2", 2_000_000, values=v[:10], span=1, step=1)
        st = np.arange(50, 20_050)
        w.addEntries(["10"] * st.size, st, ends=st + 1, values=np.sin(st))
        with pytest.raises(RuntimeError):
            w.addEntries("2", 5, values=[1.0], span=1, step=1)       # out of order
        with pytest.raises(RuntimeError):
            w.addEntries("zz", 5, values=[1.0], span=1, step=1)      # unknown contig
    r = bigwig.open(p)
    assert r.chroms() == {"2": 5_000_000, "10": 4_000_000}
    s, e, x = r.intervals_arrays("2", 0, 5_000_000)
    assert np.array_equal(x[:100_000], v.astype(np.float32)) and s[0] == 123 and s[100_000] == 2_000_000
    assert r.intervals("2", 123 + 99_999, 2_000_001) == ((123 + 99_999, 123 + 100_000, float(np.float32(v[-1]))), (2_000_000, 2_000_001, float(np.float32(v[0]))))
    assert r.intervals("10", 0, 50) is None
    assert np.allclose(r.intervals_arrays("10", 0, 4_000_000)[2], np.sin(st).astype(np.float32))
    with pytest.raises(RuntimeError):
        r.intervals("2", 10, 5_000_001)   # pyBigWig: "Invalid interval bounds!"
    hd = r.header()
    assert hd["nBasesCovered"] == 100_000 + 10 + 20_000 and hd["minVal"] <= -39


def test_bigwig_sections_are_standard_zlib_and_prefetch(tmp_path):
    """The batched section codec (ftk_zlib_*_batch) writes plain zlib streams and reads them back."""
    import struct
    import zlib
    from finaletoolkit_b200.io import bigwig
    p = str(tmp_path / "b.bw")
    rng = np.random.default_rng(3)
    v = rng.integers(-60, 30, 70_000).astype(np.float64)
    with bigwig.open(p, "w") as w:
        w.addHeader([("1", 1_000_000)])
        for i in range(0, 70_000, 5000):                    # multi_wps-style: one call per interval
            w.addEntries("1", 1000 + i, values=v[i: i + 5000], span=1, step=1)
    r = bigwig.open(p)
    # every R-tree leaf points at an independent zlib stream python's zlib inflates
    got = []
    for doff, dsize in r._blocks(0, 0, 1_000_000):
        raw = zlib.decompress(r._buf[doff: doff + dsize])
        cid, s, e, step, span, typ, _, n = struct.unpack_from("<IIIIIBBH", raw, 0)
        assert (cid, step, span, typ) == (0, 1, 1, 3) and e - s == n and len(raw) == 24 + 4 * n
        got.append(np.frombuffer(raw, "<f4", n, 24))
    assert np.array_equal(np.concatenate(got), v.astype(np.float32))
    # prefetch == lazy reads; invalid queries are ignored by prefetch and raise when queried
    lazy = r.intervals_arrays("1", 3000, 60_000)
    r2 = bigwig.open(p)
    r2.prefetch([("1", 3000, 60_000), ("nope", 0, 5), ("1", 10, 2_000_000)])
    assert len(r2._cache) > 0
    pre = r2.intervals_arrays("1", 3000, 60_000)
    assert all(np.array_equal(a, b) for a, b in zip(lazy, pre))
    with pytest.raises(RuntimeError):
        r2.intervals_arrays("1", 10, 2_000_000)
    # the raw codec: bad slot -> invalid, corrupt stream -> io error
    from finaletoolkit_b200._lib import FtkLibraryError
    with pytest.raises(FtkLibraryError):
        bigwig._inflate_sections(b"not a zlib stream at all", [(0, 24)], 1024)


def test_savgol_tables_match_scipy():
    from scipy.signal import savgol_coeffs, savgol_filter
    from finaletoolkit_b200.device import savgol_tables
    x = np.random.default_rng(0).normal(size=300)
    for w, d in [(21, 2), (11, 3), (31, 4), (5, 2), (3, 1)]:
        c, ef, el = savgol_tables(w, d)
        y = savgol_filter(x, w, d)
        h = w // 2
        assert np.abs(c - savgol_coeffs(w, d)).max() < 1e-11
        assert np.abs(ef @ x[:w] - y[:h]).max() < 1e-10 and np.abs(el @ x[-w:] - y[-h:]).max() < 1e-10
    with pytest.raises(ValueError):
        savgol_tables(20, 2)


def test_lpt_packing():
    from finaletoolkit_b200.sharding import lpt_pack
    from finaletoolkit_b200.synth import B37_CONTIGS
    w = dict(B37_CONTIGS)
    tot = sum(w.values())
    # greedy LPT + exchange refinement: b37 lands within 1 % of perfect balance up to 8 ranks
    for n, bound in [(1, 0.0), (2, 0.001), (3, 0.001), (4, 0.002), (5, 0.002), (6, 0.003), (7, 0.01), (8, 0.01)]:
        bins = lpt_pack(w, n)
        assert sorted(c for b in bins for c in b) == sorted(w)
        loads = [sum(w[c] for c in b) for b in bins]
        assert max(loads) / (tot / n) - 1 <= bound, (n, loads)
        order = {c: i for i, c in enumerate(w)}
        assert all(b == sorted(b, key=order.get) for b in bins)
        assert bins == lpt_pack(dict(w), n)                      # deterministic: every rank computes the same shards
    # degenerate inputs: more ranks than contigs, zero weights, nothing at all
    assert sorted(map(tuple, lpt_pack({"a": 5, "b": 3}, 4))) == [(), (), ("a",), ("b",)]
    assert lpt_pack({"a": 0, "b": 0}, 2) in ([["a", "b"], []], [["a"], ["b"]])
    assert lpt_pack({}, 3) == [[], [], []]
    rng = __import__("numpy").random.default_rng(0)
    for _ in range(20):                                           # never worse than the greedy step it starts from
        ww = {f"c{i}": int(v) for i, v in enumerate(rng.integers(1, 10_000, int(rng.integers(1, 40))))}
        n = int(rng.integers(1, 12))
        bins = lpt_pack(ww, n)
        assert sorted(c for b in bins for c in b) == sorted(ww)
        greedy = [0] * n
        for c in sorted(ww, key=lambda c: -ww[c]):
            greedy[greedy.index(min(greedy))] += ww[c]
        assert max(sum(ww[c] for c in b) for b in bins) <= max(greedy)


_GLOO_WORKER = r'''
import os, sys, json
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["FTK_REPO"])
from finaletoolkit_b200.sharding import DistContext, genome_length_dict, lpt_pack, pack_partials, unpack_partials
from finaletoolkit_b200.synth import synth_fragments
from oracle import oracle as O
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["FTK_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
ctx = DistContext()
contigs = {"a": 50_000, "b": 30_000, "c": 80_000, "d": 10_000, "e": 45_000}
mine = lpt_pack(contigs, ctx.world)[ctx.rank]
order = {c: i for i, c in enumerate(contigs)}
n_bins = 601
parts, total, motif = [], 0, torch.zeros(256, dtype=torch.int64)
for c in mine:   # per-contig partials as the CUDA kernels would deliver them (here: from the oracle)
    st, sp, mq, sd = synth_fragments(contigs[c], contigs[c] // 5, order[c], seed_base=4000)
    fr = O.Frags(st, sp, mq, sd)
    d = O.length_dist(fr, None, None, 0, None, "midpoint", 30)
    hist = torch.zeros(n_bins, dtype=torch.int64); first = torch.full((n_bins,), 2**31 - 1, dtype=torch.int32)
    L = (sp - st); ok = (mq >= 30)
    for i in np.flatnonzero(ok):
        hist[L[i]] += 1
        first[L[i]] = min(int(first[L[i]]), int(i))
    assert {int(k): int(hist[k]) for k in torch.nonzero(hist).flatten()} == {k: v for k, v in sorted(d.items())}
    parts.append((order[c], hist, first)); total += int(hist.sum()); motif[order[c]] += 7
buf = pack_partials(total, torch.zeros(n_bins, dtype=torch.int64) if not parts else sum(p[1] for p in parts), motif)
ctx.all_reduce_sum(buf)
tot, hist, mot = unpack_partials(buf, n_bins, 256)
d = genome_length_dict(ctx, parts, n_bins)
if ctx.rank == 0:
    print(json.dumps({"total": tot, "hist_sum": int(hist.sum()), "motif": mot[:5].tolist(), "keys": list(d)[:40], "vals": list(d.values())[:40], "n": len(d)}))
dist.barrier(); dist.destroy_process_group()
'''


def test_gloo_world2_genome_histogram(tmp_path):
    """World-size-2 run of the N>1 host path on CPU (gloo): LPT sharding by contig, one packed
    SUM all-reduce + the first-seen MIN reduce; result must equal the single-process stream."""
    from finaletoolkit_b200.synth import synth_fragments
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", FTK_REPO=REPO, FTK_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=240) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    import json
    got = json.loads(outs[0][0].strip().splitlines()[-1])
    # single-process expectation: contigs streamed in file order a..e
    contigs = {"a": 50_000, "b": 30_000, "c": 80_000, "d": 10_000, "e": 45_000}
    dicts = []
    for i, (c, n) in enumerate(contigs.items()):
        st, sp, mq, sd = synth_fragments(n, n // 5, i, seed_base=4000)
        dicts.append(O.length_dist(O.Frags(st, sp, mq, sd), None, None, 0, None, "midpoint", 30))
    exp = O.merge_dists(dicts)
    assert got["total"] == sum(exp.values()) == got["hist_sum"] and got["n"] == len(exp)
    assert got["keys"] == list(exp)[:40] and got["vals"] == list(exp.values())[:40]
    assert got["motif"] == [7, 7, 7, 7, 7]


def test_native_decoder_bgzf_gzip_and_quirks(tmp_path, manifest):
    """C++ multi-threaded decoder (ftk_fragfile_*) == the tolerant Python row parser."""
    import gzip
    from helpers import write_bgzf
    from finaletoolkit_b200.io import fragments as FR
    from finaletoolkit_b200.synth import synth_fragments
    rows = []
    for ci, (c, n) in enumerate([("chr2", 40_000), ("chr10", 25_000), ("chrUn_gl000220", 3)]):
        st, sp, mq, sd = synth_fragments(3_000_000, n, ci, seed_base=123)
        rows += [f"{c}\t{a}\t{b}\t{q}\t{'+' if s else '-'}" for a, b, q, s in zip(st.tolist(), sp.tolist(), mq.tolist(), sd.tolist())]
    rows.insert(10, "chr2\tx\t5\t60\t+"); rows.insert(500, "chr2\t7"); rows.insert(900, "# a comment"); rows.insert(901, "")
    rows.insert(20_000, "chr2\t100\t260\t300\t+-")      # mapq > 255 clamps, '+' anywhere in the strand field
    text = "\n".join(rows) + "\n"
    exp = FR._parse_text_rows(text.splitlines(keepends=True))
    p1 = write_bgzf(tmp_path / "a.frag.gz", text)
    with gzip.open(tmp_path / "b.frag.gz", "wt") as fh:
        fh.write(text)
    open(str(tmp_path / "b.frag.gz") + ".tbi", "wb").close()
    for path, threads in [(p1, 0), (p1, 1), (p1, 5), (str(tmp_path / "b.frag.gz"), 3)]:
        got = FR._decode_native(path, threads)
        assert got is not None and list(got) == list(exp)
        for c in exp:
            for a, b in zip(got[c], exp[c]):
                assert np.array_equal(a, b), (path, c)
    # python's gzip reads the BGZF we wrote (it is plain multi-member gzip)
    assert gzip.open(p1, "rt").read() == text
    # BED6 detection + warning, through the public loader
    m = manifest["fixture17"]
    p6 = write_bgzf(tmp_path / "c.bed.gz", m["frag_bed_gz_text"])
    with pytest.warns(UserWarning):
        t = FR.load_fragments(p6)
    assert t.n_fragments() == 17 and t.host("12")[2][4] == 54
    # corrupt file -> the native decoder declines, the loader falls back and raises
    bad = tmp_path / "bad.frag.gz"; bad.write_bytes(b"\x1f\x8b\x08\x00garbage"); open(str(bad) + ".tbi", "wb").close()
    assert FR._decode_native(str(bad)) is None


def test_c_abi_argument_validation_needs_no_gpu():
    """Every entry point validates its arguments before touching CUDA: zero work is FTK_OK, nonsense is
    a negative code with a message (include/ftk_b200.h: FTK_E_INVALID -1, FTK_E_RANGE -3)."""
    import ctypes
    from finaletoolkit_b200._lib import FtkLibraryError, check, lib
    L = lib()
    assert L.ftk_abi_version() >= 1
    assert b"invalid" in L.ftk_error_string(-1).lower() and L.ftk_error_string(-3) and L.ftk_error_string(-4)
    i64 = (ctypes.c_int64 * 4)(0, 10, 0, 0)
    i32 = (ctypes.c_int32 * 4)()
    # zero work -> FTK_OK without any pointer
    assert L.ftk_wps_tiles_i32(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 120, 120, 180, 30, 0, 0, 0, 0) == 0
    assert L.ftk_interval_hist_u64(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0) == 0
    assert L.ftk_end_motif_hist_u64(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 4, 0, 30, 0, 1, 0, 0, 0, 0) == 0
    assert L.ftk_breakpoint_motif_hist_u64(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 6, 0, 30, 0, 1, 0, 0, 0) == 0
    assert L.ftk_delfi_windows_u64(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, None, 30, 1, 0, 0, 0) == 0
    assert L.ftk_agg_signal_f64(0, 0, 0, 0, 0, 0, 0, 0) == 0
    assert L.ftk_savgol_f64(0, 0, 0, 0, 21, 0, 0, 0, 0, 0) == 0
    assert L.ftk_cleavage_tiles_f64(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0) == 0
    # nonsense -> negative code, never a launch
    assert L.ftk_wps_tiles_i32(0, 0, 0, 5, 0, 0, 0, 0, 0, 3, 120, 120, 180, 30, 0, 0, 0, 0) == -1     # tiles, no tables
    assert L.ftk_wps_tiles_i16(0, 0, 0, 0, 0, 0, 0, 0, 0, 3, 120, 120, 180, 30, 0, 0, 0, 0, 0) == -1  # no overflow flag
    assert L.ftk_end_motif_hist_u64(0, 0, 0, 0, 0, 0, 1, 1, 9, 1, 1, 2, 13, 0, 30, 0, 1, 1, 1, 1, 0) == -1    # k > 12
    assert L.ftk_end_motif_hist_u64(0, 0, 0, 0, 0, 0, 1, 1, 9, 1, 1, 2, 4, 7, 30, 0, 1, 1, 1, 1, 0) == -1     # strand mode
    assert L.ftk_breakpoint_motif_hist_u64(0, 0, 0, 0, 0, 0, 0, 0, 9, 1, 1, 2, 6, 0, 30, 0, 1, 1, 1, 0) == -1  # no contig
    assert L.ftk_delfi_windows_u64(0, 0, 0, 5, 0, 0, 0, 0, 1, 1, 2, 0, 0, 0, None, 30, 1, 1, 1, 0) == -1      # fragments, no columns
    assert L.ftk_delfi_windows_u64(0, 0, 0, 0, 0, 1, 0, 9, 1, 1, 2, 0, 0, 0, None, 30, 1, 1, 1, 0) == -1      # seq without N mask
    assert L.ftk_agg_signal_f64(1, 2, 10, 6, 6, 1, 1, 0) == -1                                                  # trim + out > row
    assert L.ftk_savgol_f64(1, 1, 1, 10, 20, 1, 1, 1, 2, 0) == -1                                               # even window
    assert L.ftk_adjust_wps_f64(1, 1, 1, 1, 0, 1, 1, 999, 0, 100, 1, 1, 0) == -1                                # odd median window
    n_tiles = L.ftk_wps_plan_tiles(i64, ctypes.cast(ctypes.byref(i64, 8), ctypes.POINTER(ctypes.c_int64)), i64, 1,
                                   2 ** 40, 180, None, None, None, None, None)
    assert n_tiles == -3                                                                                         # chrom_size > int32
    with pytest.raises(FtkLibraryError, match="ftk_wps_plan_tiles"):
        check(n_tiles, "ftk_wps_plan_tiles")
    err = ctypes.c_int32(0)
    assert L.ftk_fragfile_open(b"/nonexistent/x.frag.gz", 1, ctypes.byref(err)) is None and err.value == -4
    o = (ctypes.c_int64 * 2)(0, 4); sz = (ctypes.c_int64 * 1)()
    buf = (ctypes.c_uint8 * 8)(); out = (ctypes.c_uint8 * 8)()
    assert L.ftk_zlib_compress_batch(buf, o, 1, 6, 1, out, o, sz) == -1                                         # slot < compressBound
    assert L.ftk_zlib_uncompress_batch(buf, o, sz, -1, 1, out, o, sz) == -1
    del i32


def test_delfi_host_logic_against_reference_tables(tmp_path, manifest):
    """Host side of the DELFI path (no GPU): gap track -> arms, blacklist CSR, gap-overlap bin filter
    and the 50-bin merge, against what the reference produced (tests/golden, frag/_delfi.py,
    frag/_delfi_merge_bins.py, genome/gaps.py)."""
    import io
    import pandas
    from helpers import delfi_tracks
    from finaletoolkit_b200.device import blacklist_in_windows
    from finaletoolkit_b200.frag._delfi import _bins_overlapping_gaps, _load_blacklist_indexed, delfi_merge_bins
    from finaletoolkit_b200.genome import GenomeGaps
    m = manifest["delfi"]
    gap_path = tmp_path / "gaps.bed"; gap_path.write_text(m["gaps"])
    bl_path = tmp_path / "bl.bed"; bl_path.write_text(m["blacklist"])
    gaps = GenomeGaps(str(gap_path))
    bins = [tuple(b) for b in m["bins_list"]]
    # arms exactly as _delfi_single_window derives them (in_tcmere first, then get_arm)
    case = next(c for c in m["single_window"] if c["use_gaps"])
    for (c, a, b), arm in zip(bins, case["arms"]):
        cg = gaps.get_contig_gaps(c)
        got = c if cg is None else ("NOARM" if cg.in_tcmere(a, b) else cg.get_arm(a, b))
        assert got == arm, (c, a, b)
    assert gaps.get_contig_gaps("chrX9") is None and gaps.in_tcmere("chrX9", 0, 10) is None
    assert gaps.in_tcmere("chr7", 5_000, 20_000) is True and gaps.overlaps_gap("chr21", 45_000, 49_000) is False
    assert gaps.get_arm("chr21", 10, 20) == "NOARM" and gaps.get_arm("chr7", 700_000, 800_000) == "7q"
    out = tmp_path / "gaps_out.bed"; gaps.to_bed(str(out))
    assert sorted(out.read_text().splitlines()) == sorted("\t".join(ln.split()) for ln in m["gaps"].splitlines())
    # blacklist: same parse as the reference, CSR == brute force containment
    bl = _load_blacklist_indexed(str(bl_path)); bl_ref, _ = delfi_tracks(m)
    assert set(bl) == set(bl_ref) and all(np.array_equal(bl[c][0], bl_ref[c][0]) and np.array_equal(bl[c][1], bl_ref[c][1]) for c in bl)
    ws = np.array([b[1] for b in bins if b[0] == "chr7"]); we = np.array([b[2] for b in bins if b[0] == "chr7"])
    off, rs, re = blacklist_in_windows(bl["chr7"][0], bl["chr7"][1], ws, we)
    for j in range(len(ws)):
        exp = [(a, b) for a, b in zip(bl["chr7"][0].tolist(), bl["chr7"][1].tolist()) if a >= ws[j] and b <= we[j]]
        assert list(zip(rs[off[j]: off[j + 1]].tolist(), re[off[j]: off[j + 1]].tolist())) == exp
    assert off[-1] >= 4
    # bins overlapping any gap are dropped before counting (utils.overlaps)
    df = pandas.DataFrame(bins, columns=["contig", "start", "stop"])
    hit = _bins_overlapping_gaps(df, gaps)
    g = gaps.gaps
    brute = [bool(np.any((g["contig"] == c) & (a < g["stop"]) & (b > g["start"]))) for c, a, b in bins]
    assert hit.tolist() == brute and 0 < hit.sum() < len(bins)
    # merge: the reference's per-bin table -> its merged table (p arms from the first bin, q arms from the last)
    per_bin = pandas.read_csv(io.StringIO(m["delfi"][0]["tsv"]), sep="\t", float_precision="round_trip").rename(columns={"#contig": "contig"})
    merged = delfi_merge_bins(per_bin, gc_corrected=False)
    buf = io.StringIO(); merged.rename(columns={"contig": "#contig"}).to_csv(buf, sep="\t", index=False)
    assert buf.getvalue() == m["delfi"][1]["tsv"]
    with pytest.raises(ImportError):
        from finaletoolkit_b200.frag._delfi import delfi_gc_correct
        delfi_gc_correct(per_bin)


def test_native_text_outputs(tmp_path):
    """ftk_format_bedgraph_i64 writes the reference's bedGraph lines (frag/_multi_wps.py:328-341) and
    ftk_gzip_compress_batch members concatenate into a .gz every gzip reader accepts."""
    import gzip
    import subprocess
    from finaletoolkit_b200.io.textout import GzipTextWriter, bedgraph_bytes, bedgraph_text
    rng = np.random.default_rng(0)
    for contig, start, n in [("1", 0, 5000), ("chrUn_KI270742v1", 2_147_480_000, 33), ("12", 9, 1), ("X", 99, 200_000)]:
        sc = rng.integers(-3000, 3000, n)
        exp = "".join(f"{contig}\t{p}\t{p + 1}\t{v}\n" for p, v in zip(range(start, start + n), sc.tolist()))
        assert bedgraph_bytes(contig, start, sc).decode() == exp
    assert bedgraph_bytes("1", 5, []) == b"" and bedgraph_bytes("1", 7, [np.iinfo(np.int64).min]) == f"1\t7\t8\t{np.iinfo(np.int64).min}\n".encode()
    path = str(tmp_path / "out.bedgraph.gz")
    chunks = [bedgraph_text("7", 1_000_000 * k, rng.integers(-50, 20, 300_000)) for k in range(8)]
    with GzipTextWriter(path) as w:
        w.write("# header as str\n")
        for c in chunks:
            w.write(c)
        w.write(b"tail as bytes\n")
    exp = b"# header as str\n" + b"".join(c.tobytes() for c in chunks) + b"tail as bytes\n"
    assert gzip.open(path, "rb").read() == exp
    assert len(exp) > (4 << 20)                                       # several 1 MiB members
    assert subprocess.run(["gzip", "-t", path]).returncode == 0
    empty = str(tmp_path / "empty.gz")
    with GzipTextWriter(empty):
        pass
    assert gzip.open(empty, "rb").read() == b""


def test_tabix_index_and_lazy_contig_decode(tmp_path, golden, monkeypatch):
    """.tbi reader + per-contig decode through the index (io/tabix.py, ftk_fragfile_open_slice):
    the htslib-made fixture index, and synthetic multi-contig BGZF files indexed by the test helper
    (which reproduces htslib's index bytes on the fixture) - lazy columns == whole-file decode."""
    import struct
    from helpers import write_bgzf_indexed
    from finaletoolkit_b200.io import fragments
    from finaletoolkit_b200.io.tabix import read_tbi
    g = golden("fixture17")
    # 1. the reference's own files, byte for byte
    for stem, key in (("fx.frag.gz", "frag_gz"), ("fx.bed.gz", "bed_gz")):
        p = tmp_path / stem
        p.write_bytes(g[key + "_file"].tobytes()); (tmp_path / (stem + ".tbi")).write_bytes(g[key + "_tbi_file"].tobytes())
        idx = read_tbi(str(p) + ".tbi")
        assert idx.names == ["12"] and (idx.col_seq, idx.col_beg, idx.col_end, idx.meta) == (1, 2, 3, "#")
        cb, ub, ce, ue = idx.ranges["12"]
        assert (cb, ub, ue) == (0, 0, 0) and ce == p.stat().st_size - 28          # up to the BGZF EOF block
        monkeypatch.setenv("FTK_LAZY_MIN_BYTES", "0")
        fragments._CACHE.clear()
        import warnings as w
        with w.catch_warnings():
            w.simplefilter("ignore")
            lazy = fragments.load_fragments(str(p))
        assert lazy._loader is not None and lazy.contigs == ["12"] and lazy.columns == {}
        st, sp, mq, sd = lazy.host("12")
        assert np.array_equal(st, g["start"]) and np.array_equal(sp, g["stop"]) and np.array_equal(mq, g["mapq"]) \
            and np.array_equal(sd, g["strand"])
        assert lazy.n_fragments("nope") == 0 and lazy.n_fragments() == 17
        # the test indexer writes the same index htslib wrote (modulo its own compressed block size)
        import gzip
        mine = write_bgzf_indexed(tmp_path / ("re_" + stem), gzip.open(p, "rt").read(), block=65280)
        a = gzip.open(mine + ".tbi", "rb").read(); b = gzip.open(str(p) + ".tbi", "rb").read()
        own_end = (tmp_path / ("re_" + stem)).stat().st_size - 28
        assert a.replace(struct.pack("<Q", own_end << 16), struct.pack("<Q", ce << 16)) == b
    assert read_tbi(str(tmp_path / "fx.frag.gz")) is None                            # not an index
    # 2. three contigs, lines straddling 4 KiB blocks, a one-row contig in the middle, comment lines
    rng = np.random.default_rng(5)
    rows, cols = ["#made by the test"], {}
    for contig, n in (("chr1", 30_000), ("chrTiny", 1), ("chrX_random", 12_345)):
        st = np.sort(rng.integers(0, 50_000_000, n)); sp = st + rng.integers(30, 600, n)
        mq = rng.integers(0, 61, n); sd = rng.integers(0, 2, n)
        cols[contig] = (st.astype(np.int32), sp.astype(np.int32), mq.astype(np.uint8), sd.astype(np.uint8))
        rows += [f"{contig}\t{a}\t{b}\t{q}\t{'+' if s else '-'}" for a, b, q, s in zip(st.tolist(), sp.tolist(), mq.tolist(), sd.tolist())]
    path = write_bgzf_indexed(tmp_path / "multi.frag.gz", "\n".join(rows) + "\n", block=4096)
    monkeypatch.setenv("FTK_LAZY_MIN_BYTES", str(10 ** 12))
    fragments._CACHE.clear()
    whole = fragments.load_fragments(path)
    assert whole._loader is None and whole.contigs == list(cols)
    monkeypatch.setenv("FTK_LAZY_MIN_BYTES", "0")
    fragments._CACHE.clear()
    lazy = fragments.load_fragments(path)
    assert lazy._loader is not None and lazy.contigs == list(cols) and lazy.columns == {}
    assert lazy.n_fragments("chrTiny") == 1 and list(lazy.columns) == ["chrTiny"]    # only what was asked for
    for contig in ("chrX_random", "chr1", "chrTiny"):
        for x, y, z in zip(lazy.host(contig), whole.host(contig), cols[contig]):
            assert np.array_equal(x, y) and np.array_equal(x, z), contig
    assert lazy.n_fragments() == sum(len(c[0]) for c in cols.values())
    # 3. BED6 layout through the lazy path (mapq = column 5, strand = column 6) + its UserWarning
    bed_rows = [f"c\t{a}\t{a + 100}\tname\t{q}\t{'+-'[a & 1]}" for a, q in zip(range(0, 90_000, 3), rng.integers(0, 61, 30_000).tolist())]
    bed = write_bgzf_indexed(tmp_path / "multi.bed.gz", "\n".join(bed_rows) + "\n", block=8192)
    fragments._CACHE.clear()
    with pytest.warns(UserWarning, match="BED6"):
        t6 = fragments.load_fragments(bed)
    st, sp, mq, sd = t6.host("c")
    assert st.size == 30_000 and np.array_equal(st, np.arange(0, 90_000, 3)) and np.array_equal(sd, 1 - (st & 1))
    # a placeholder .tbi (what the other tests write) falls back to the whole-file decode
    fragments._CACHE.clear()
    open(path + ".tbi", "wb").close()
    assert fragments.load_fragments(path)._loader is None
    fragments._CACHE.clear()


def test_native_bam_decoder(tmp_path, manifest, golden):
    """ftk_bamfile_open == the reference's _fetch_sam on its own BAM fixture, and == the oracle's record
    walk on synthetic BAMs covering every filtered flag, tlen sign, CIGAR op and block-straddling records."""
    from helpers import write_bam
    from finaletoolkit_b200.io import fragments
    g = golden("fixture17"); m = manifest["fixture17"]
    # the oracle restatement is pinned on what the reference yields from tests/data/12.3444.b37.bam
    refs, rows = O.bam_fragments(g["bam_file"].tobytes())
    assert len(refs) == m["bam_n_refs"] and dict(refs)["12"] == m["bam_ref_12"]
    assert [r[1] for r in rows] == g["bam_start"].tolist() and [r[2] for r in rows] == g["bam_stop"].tolist()
    assert [r[3] for r in rows] == g["bam_mapq"].tolist() and [int(r[4]) for r in rows] == g["bam_strand"].tolist()
    bam = tmp_path / "fx.bam"; bam.write_bytes(g["bam_file"].tobytes()); (tmp_path / "fx.bam.bai").write_bytes(b"")
    fragments._CACHE.clear()
    tab = fragments.load_fragments(str(bam))
    assert tab.is_sam and tab.contigs == m["bam_contigs"] and len(tab.contig_lengths) == m["bam_n_refs"]
    assert tab.contig_lengths["12"] == m["bam_ref_12"]
    st, sp, mq, sd = tab.host("12")
    order = np.argsort(g["bam_start"], kind="stable")          # the table is start-sorted, file order kept among ties
    assert np.array_equal(st, g["bam_start"][order]) and np.array_equal(sp, g["bam_stop"][order])
    assert np.array_equal(mq, g["bam_mapq"][order]) and np.array_equal(sd, g["bam_strand"][order])
    # same coordinates and strands as the fragment file made from this BAM (its mapq column is the pair's)
    assert np.array_equal(st, g["start"]) and np.array_equal(sp, g["stop"]) and np.array_equal(sd, g["strand"])
    # synthetic: 3 references, ~6000 reads, every flag bit of the filter, both tlen signs, all CIGAR ops
    rng = np.random.default_rng(3)
    refs = [("chrA", 5_000_000), ("chrB", 900_000), ("chrEmpty", 1000)]
    good = 0x1 | 0x2 | 0x40
    recs = []
    for ref, n in ((0, 4000), (1, 2000)):
        pos = np.sort(rng.integers(0, refs[ref][1] - 1000, n))
        for p in pos.tolist():
            flag = good | (0x10 if rng.random() < 0.5 else 0)
            u = rng.random()
            if u < 0.30:
                flag ^= int(rng.choice([0x1, 0x2, 0x4, 0x8, 0x100, 0x200, 0x400, 0x800]))   # one filter bit flipped
            elif u < 0.40:
                flag = (flag & ~0x40) | 0x80                                                 # read 2
            tlen = int(rng.choice([0, 1, -1])) * int(rng.integers(30, 600))
            ops = [(4, 5)] if rng.random() < 0.3 else []
            ops += [(0, int(rng.integers(20, 80)))]
            if rng.random() < 0.5:
                ops += [(int(rng.choice([1, 2, 3, 7, 8])), int(rng.integers(1, 30))), (0, int(rng.integers(5, 40)))]
            if rng.random() < 0.2:
                ops += [(5, 3)]
            recs.append(dict(ref=ref, pos=p, mapq=int(rng.integers(0, 61)), flag=flag, tlen=tlen, cigar=ops))
    recs.append(dict(ref=-1, pos=-1, mapq=0, flag=0x4 | 0x1, tlen=0, cigar=[]))              # unplaced read at the end
    path = write_bam(tmp_path / "syn.bam", refs, recs, block=3000)
    _, exp = O.bam_fragments(open(path, "rb").read())
    assert 1500 < len(exp) < len(recs)
    fragments._CACHE.clear()
    tab = fragments.load_fragments(path)
    assert tab.contigs == ["chrA", "chrB"] and tab.contig_lengths == dict(refs)
    for contig in tab.contigs:
        rows = [r for r in exp if r[0] == contig]
        order = np.argsort(np.array([r[1] for r in rows]), kind="stable")
        st, sp, mq, sd = tab.host(contig)
        assert st.tolist() == [rows[i][1] for i in order] and sp.tolist() == [rows[i][2] for i in order]
        assert mq.tolist() == [rows[i][3] for i in order] and sd.tolist() == [int(rows[i][4]) for i in order]
    # a truncated file is an I/O error for the native decoder; the loader then needs pysam and says so
    cut = tmp_path / "cut.bam"; cut.write_bytes(open(path, "rb").read()[:5000]); (tmp_path / "cut.bam.bai").write_bytes(b"")
    from finaletoolkit_b200.exceptions import UnsupportedFormatError
    fragments._CACHE.clear()
    with pytest.raises(UnsupportedFormatError):
        fragments.load_fragments(str(cut))
    fragments._CACHE.clear()


def test_savgol_rational_coefficients():
    """The exact rational form of the interior Savitzky-Golay coefficients the sliding-moment smoothing uses
    (device.savgol_rational: c_i = (a + b i^2) / den) against scipy's own coefficients and exact fractions."""
    from fractions import Fraction
    from scipy.signal import savgol_coeffs
    from finaletoolkit_b200.device import savgol_rational
    assert savgol_rational(21, 2) == (329, -5, 3059)            # the textbook 21-point quadratic smoother
    for m in range(3, 61, 2):
        h = m // 2
        for deg in range(0, min(m, 6)):
            a, b, den = savgol_rational(m, deg)
            if deg >= 4:
                assert (a, b, den) == (0, 0, 0)
                continue
            assert den > 0
            c = np.array([(a + b * i * i) / den for i in range(-h, h + 1)])
            assert np.abs(c - savgol_coeffs(m, deg)).max() < 1e-12, (m, deg)
            assert sum(Fraction(a + b * i * i, den) for i in range(-h, h + 1)) == 1      # a smoother preserves constants
            if deg >= 2:                                                                   # ... and quadratics
                assert sum(Fraction(a + b * i * i, den) * i * i for i in range(-h, h + 1)) == 0


def test_flat_namespace_and_overlaps():
    """The reference's flat namespace (finaletoolkit/__init__.py:30-128) for everything on the path: features,
    containers, exceptions, aliases; ``overlaps`` (utils/utils.py:346-383) against the all-pairs definition."""
    import finaletoolkit_b200 as F
    for name in ("wps", "multi_wps", "adjust_wps", "coverage", "single_coverage", "frag_length", "frag_length_bins",
                 "frag_length_intervals", "end_motifs", "region_end_motifs", "interval_end_motifs", "EndMotifFreqs",
                 "EndMotifsIntervals", "breakpoint_motifs", "region_breakpoint_motifs", "interval_breakpoint_motifs",
                 "BreakpointMotifFreqs", "BreakpointMotifsIntervals", "cleavage_profile", "multi_cleavage_profile", "delfi",
                 "delfi_gc_correct", "delfi_merge_bins", "agg_bw", "frag_generator", "frag_array", "frags_in_region",
                 "get_intervals", "overlaps", "gen_kmers", "reverse_complement", "chrom_sizes_to_dict",
                 "chrom_sizes_to_list", "GenomeGaps", "ContigGaps", "ReferenceWrapper", "FinaleToolkitError",
                 "InvalidInputError", "UnsupportedFormatError", "MissingReferenceError", "MissingIndexError",
                 "ContigNotFoundError", "ContigMismatchError", "OutOfBoundsError"):
        assert getattr(F, name) is not None and name in dir(F), name
    assert F.end_motif is F.end_motifs and F.breakpoint_motif is F.breakpoint_motifs
    assert issubclass(F.InvalidInputError, F.FinaleToolkitError) and issubclass(F.InvalidInputError, ValueError)
    assert issubclass(F.MissingIndexError, FileNotFoundError) and issubclass(F.OutOfBoundsError, IndexError)
    with pytest.raises(AttributeError):
        F.no_such_feature
    rng = np.random.default_rng(5)
    for _ in range(100):
        n1, n2 = int(rng.integers(0, 30)), int(rng.integers(0, 30))
        c1, c2 = rng.choice(["a", "b", "c"], n1), rng.choice(["a", "b", "d"], n2)
        s1 = rng.integers(0, 100, n1); e1 = s1 + rng.integers(0, 20, n1)
        s2 = rng.integers(0, 100, n2); e2 = s2 + rng.integers(0, 20, n2)
        exp = (np.any((s1[:, None] < e2[None]) & (e1[:, None] > s2[None]) & (c1[:, None] == c2[None]), axis=1)
               if n1 and n2 else np.zeros(n1, bool))
        assert np.array_equal(F.overlaps(c1, s1, e1, c2, s2, e2), exp)
