"""Packed fragment columns: what the host decoder hands to the GPU (3.06 or 4.06 B per fragment).

Layout and rationale: ``csrc/ftk_pack.cu`` / ``include/ftk_b200.h``.  The host side packs once per
contig (``ftk_pack_fragments_host``, multi-threaded, at decode time); the device side unpacks a
whole contig or any 64-fragment-aligned slice into the int32 / uint8 columns the kernels read
(``ftk_unpack_fragments``).  Replaces the reference's per-interval text stream
(io/alignment.py:270-302) as the host -> device seam.
"""
from __future__ import annotations

from ctypes import POINTER, c_int32, c_uint8, c_uint32

import numpy as np

from ._lib import check, lib
from .device import ContigFragments, _launch, require_cuda, torch

__all__ = ["PackedFragments", "PACK_BLOCK"]

PACK_BLOCK = 64


def _p(a, ctype):
    return None if a is None else a.ctypes.data_as(POINTER(ctype))


class PackedFragments:
    """Start-sorted fragments of one contig in the packed wire format, in (pinned) host memory."""

    def __init__(self, start, stop, mapq=None, strand=None, pinned=True, threads=0, max_len=None,
                 record_bytes=None):
        t = torch()
        start = np.ascontiguousarray(start, dtype=np.int32)
        stop = np.ascontiguousarray(stop, dtype=np.int32)
        mapq = None if mapq is None else np.ascontiguousarray(mapq, dtype=np.uint8)
        strand = None if strand is None else np.ascontiguousarray(strand, dtype=np.uint8)
        if start.size and not np.all(start[1:] >= start[:-1]):
            order = np.argsort(start, kind="stable")
            start, stop = start[order], stop[order]
            mapq = None if mapq is None else mapq[order]
            strand = None if strand is None else strand[order]
        self.n = int(start.size)
        self.has_mapq, self.has_strand = mapq is not None, strand is not None
        if max_len is None:
            max_len = int((stop.astype(np.int64) - start).max()) if self.n else 0
        self.max_len = max(int(max_len), 0)
        self.n_blocks = (self.n + PACK_BLOCK - 1) // PACK_BLOCK
        L = lib()
        args = (_p(start, c_int32), _p(stop, c_int32), _p(mapq, c_uint8), _p(strand, c_uint8), self.n, int(threads))
        # record width: the narrow 24-bit records unless their escapes (gaps >= 64 bp, fragments >= 512 bp)
        # would put more bytes on the wire than the 32-bit records (sparse or long-fragment data)
        widths = (3, 4) if record_bytes is None else (int(record_bytes),)
        best = None
        for rb in widths:
            n_raw = L.ftk_pack_fragments_host(*args, None, None, None, None, None, None, 0, rb)
            check(n_raw, "ftk_pack_fragments_host")
            cost = self.n_blocks * (PACK_BLOCK * rb + 4) + int(n_raw) * PACK_BLOCK * 10
            if best is None or cost < best[0]:
                best = (cost, rb, int(n_raw))
        _, self.record_bytes, self.n_raw = best
        self.words_per_block = PACK_BLOCK * self.record_bytes // 4

        def host(shape, dtype):
            x = t.empty(shape, dtype=dtype)
            return x.pin_memory() if (pinned and t.cuda.is_available() and x.numel()) else x

        self.words = host(max(self.n_blocks * self.words_per_block, 2), t.int32)       # record bit patterns
        self.anchors = host(max(self.n_blocks, 1), t.int32)
        r = max(self.n_raw, 1) * PACK_BLOCK
        self.raw_start, self.raw_stop = host(r, t.int32), host(r, t.int32)
        self.raw_mapq, self.raw_strand = host(r, t.uint8), host(r, t.uint8)
        if self.n:
            got = L.ftk_pack_fragments_host(
                *args, _p(self.words.numpy().view(np.uint32), c_uint32), _p(self.anchors.numpy(), c_int32),
                _p(self.raw_start.numpy(), c_int32), _p(self.raw_stop.numpy(), c_int32),
                _p(self.raw_mapq.numpy(), c_uint8), _p(self.raw_strand.numpy(), c_uint8), self.n_raw, self.record_bytes)
            check(got, "ftk_pack_fragments_host")
        self.first_start = start[::PACK_BLOCK].copy()    # block -> first start (host-side slicing by position)

    # bytes that cross PCIe for fragments [f0, f1) (f0 a multiple of PACK_BLOCK)
    def wire_bytes(self, f0=0, f1=None) -> int:
        f1 = self.n if f1 is None else f1
        nb = (f1 - f0 + PACK_BLOCK - 1) // PACK_BLOCK
        return nb * PACK_BLOCK * self.record_bytes + nb * 4

    def raw_bytes(self) -> int:
        return self.n_raw * PACK_BLOCK * 10

    def raw_to_device(self, device):
        """The (tiny) raw side columns, resident on the device."""
        dev = require_cuda(device)
        return tuple(x.to(dev, non_blocking=True) for x in (self.raw_start, self.raw_stop, self.raw_mapq, self.raw_strand))

    def unpack_into(self, d_words, d_anchors, d_raw, n, d_start, d_stop, d_mapq, d_strand, device):
        """Launch the unpack kernel on the current stream: device words/anchors (of the slice's first
        block) -> columns of ``n`` fragments."""
        _launch(device, "ftk_unpack_fragments",
                d_words.data_ptr(), d_anchors.data_ptr(), d_raw[0].data_ptr(), d_raw[1].data_ptr(), d_raw[2].data_ptr(),
                d_raw[3].data_ptr() if self.has_strand else 0, self.n_raw, int(n), d_start.data_ptr(), d_stop.data_ptr(),
                0 if d_mapq is None else d_mapq.data_ptr(), 0 if d_strand is None else d_strand.data_ptr(),
                self.record_bytes)

    def to_device(self, device=None, contig=None) -> ContigFragments:
        """H2D of the packed columns + on-device unpack -> resident ``ContigFragments``."""
        t = torch()
        dev = require_cuda(device)
        n = self.n
        npad = max(self.n_blocks * PACK_BLOCK, 2)
        d_start = t.empty(npad, dtype=t.int32, device=dev)
        d_stop = t.empty(npad, dtype=t.int32, device=dev)
        d_mapq = t.empty(npad, dtype=t.uint8, device=dev) if self.has_mapq else None
        d_strand = t.empty(npad, dtype=t.uint8, device=dev) if self.has_strand else None
        if n:
            d_words = self.words.to(dev, non_blocking=True)
            d_anch = self.anchors.to(dev, non_blocking=True)
            raw = self.raw_to_device(dev)
            self.unpack_into(d_words, d_anch, raw, n, d_start, d_stop, d_mapq, d_strand, dev)
        return ContigFragments(d_start[:n], d_stop[:n], None if d_mapq is None else d_mapq[:n],
                               None if d_strand is None else d_strand[:n], device=dev, contig=contig,
                               max_len=self.max_len)
