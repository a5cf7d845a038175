"""Host-side packing of genotype calls into the 2-bit-per-call matrix the GPU consumes (K0, DESIGN.md).

Per SNP: the 2-bit codes of 32 samples are stored as two bit-plane words, (lo bits, hi bits), bit b = sample 32g + b of
group g; population-1 pairs then population-2 pairs, each population padded with zeros to a whole pair.  Codes:
0 = 0/0, 1 = 0/1, 3 = 1/1, 2 = missing, so that #missing = popcount(hi & ~lo), alt = popcount(all words) - #missing
and ref = 2*(samples - #missing) - alt: the count kernel needs one logic op per 32 samples to find the missing calls.
Memory layout "B32" (block-transposed): SNPs are grouped in blocks of 32; word w of SNP s is stored at uint32 index
((s // 32) * RW + w) * 32 + s % 32, RW = W1 + W2.  A warp therefore reads word w of 32 consecutive SNPs as one
128-byte line, and in shared memory as one conflict-free access.  The last block is zero padded.
Replaces the per-sample character counting of make_data_dict_vcf (scripts/src/twoDSFS_class.py:118-130)."""
from __future__ import annotations

import numpy as np

CODE_HOMREF, CODE_HET, CODE_MISSING, CODE_HOMALT = 0, 1, 2, 3


def words_for(n_samples: int) -> int:
    """uint32 words per SNP of one population: a (lo plane, hi plane) pair per 32 samples."""
    return 2 * max(1, (n_samples + 31) // 32)


def _pack_block(codes: np.ndarray) -> np.ndarray:
    """codes[S, ns] -> words[S, W]: word 2g = lo bits, word 2g+1 = hi bits of samples 32g .. 32g+31."""
    S, ns = codes.shape
    W = words_for(ns)
    padded = np.zeros((S, W * 16), dtype=np.uint32)
    padded[:, :ns] = codes
    g = padded.reshape(S, W // 2, 32)
    shifts = np.arange(32, dtype=np.uint32)[None, None, :]
    out = np.empty((S, W), dtype=np.uint32)
    out[:, 0::2] = ((g & 1) << shifts).sum(axis=2, dtype=np.uint32)
    out[:, 1::2] = ((g >> 1) << shifts).sum(axis=2, dtype=np.uint32)
    return out


def unpack_block(words: np.ndarray, ns: int) -> np.ndarray:
    """words[S, W] of one population -> codes[S, ns] (inverse of _pack_block)."""
    words = np.asarray(words, dtype=np.uint32)
    S, W = words.shape
    shifts = np.arange(32, dtype=np.uint32)[None, None, :]
    lo = (words[:, 0::2, None] >> shifts) & np.uint32(1)
    hi = (words[:, 1::2, None] >> shifts) & np.uint32(1)
    return (lo | (hi << np.uint32(1))).reshape(S, -1)[:, :ns].astype(np.uint8)


def to_b32(rows: np.ndarray) -> np.ndarray:
    """row-major words [S, RW] -> B32 buffer (flat uint32, ceil(S/32)*RW*32 words)."""
    S, RW = rows.shape
    nb = (S + 31) // 32
    pad = np.zeros((nb * 32, RW), dtype=np.uint32)
    pad[:S] = rows
    return np.ascontiguousarray(pad.reshape(nb, 32, RW).transpose(0, 2, 1)).reshape(-1)


def from_b32(buf: np.ndarray, S: int, RW: int) -> np.ndarray:
    """B32 buffer -> row-major words [S, RW]."""
    nb = (S + 31) // 32
    return np.ascontiguousarray(np.asarray(buf, dtype=np.uint32).reshape(nb, RW, 32).transpose(0, 2, 1)).reshape(nb * 32, RW)[:S]


def pack_codes(codes1: np.ndarray, codes2: np.ndarray):
    """codes[S, ns] of 2-bit codes -> (G in B32 layout (flat uint32), W1, W2)."""
    b1, b2 = _pack_block(np.asarray(codes1)), _pack_block(np.asarray(codes2))
    return to_b32(np.concatenate([b1, b2], axis=1)), b1.shape[1], b2.shape[1]


# ----------------------------------------------------------------------------------------------- VCF packer (K0, C++)
import ctypes as _C
import os as _os

_PACK_LIB = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "lib", "libtdsfs_pack.so")
_plib = None


def _packer():
    global _plib
    if _plib is None:
        if not _os.path.exists(_PACK_LIB):
            raise RuntimeError(f"{_PACK_LIB} not found: build it with `python 2dsfs-scan_b200/build.py`")
        L = _C.CDLL(_PACK_LIB)
        L.tdsfs_pack_vcf.restype = _C.c_void_p
        L.tdsfs_pack_vcf.argtypes = [_C.c_char_p, _C.c_char_p, _C.c_char_p, _C.c_char_p, _C.c_int]
        L.tdsfs_pack_last_error.restype = _C.c_char_p
        for f in ("tdsfs_pack_genotypes", "tdsfs_pack_positions", "tdsfs_pack_chrom_off", "tdsfs_pack_ann_codes", "tdsfs_pack_fixups"):
            getattr(L, f).restype = _C.c_void_p
            getattr(L, f).argtypes = [_C.c_void_p]
        for f in ("tdsfs_pack_chrom_names", "tdsfs_pack_ann_vocab"):
            getattr(L, f).restype = _C.c_char_p
            getattr(L, f).argtypes = [_C.c_void_p]
        L.tdsfs_pack_dims.argtypes = [_C.c_void_p, _C.c_void_p, _C.c_void_p]
        L.tdsfs_pack_free.argtypes = [_C.c_void_p]
        L.tdsfs_vcf_counts.restype = _C.c_void_p
        L.tdsfs_vcf_counts.argtypes = [_C.c_char_p, _C.c_char_p, _C.c_int]
        L.tdsfs_vcf_counts_free.argtypes = [_C.c_void_p]
        L.tdsfs_vcf_counts_dims.argtypes = [_C.c_void_p, _C.c_void_p]
        for f in ("keys", "key_off", "refalt", "ann_codes", "cnt", "ncols", "first_col"):
            getattr(L, "tdsfs_vcf_counts_" + f).restype = _C.c_void_p
            getattr(L, "tdsfs_vcf_counts_" + f).argtypes = [_C.c_void_p]
        for f in ("pops", "vocab"):
            getattr(L, "tdsfs_vcf_counts_" + f).restype = _C.c_char_p
            getattr(L, "tdsfs_vcf_counts_" + f).argtypes = [_C.c_void_p]
        _plib = L
    return _plib


class _PackOwner:
    """Owns the C++ result of tdsfs_pack_vcf; the numpy views of its arrays keep it alive."""

    def __init__(self, lib, handle):
        self._lib, self._h = lib, handle

    def __del__(self):
        if self._h:
            self._lib.tdsfs_pack_free(self._h)
            self._h = None


class PackedPanel:
    """A VCF packed for the GPU: the array form of a data_dict restricted to two populations, at genotype level.
    Accepted by the scanners of LikelihoodInference_jointSFS in place of a data_dict (fast path: no Python dict)."""

    def __init__(self):
        self.G = None            # uint32, B32 layout
        self.W1 = self.W2 = self.ns1 = self.ns2 = 0
        self.pos = None          # int64 (int32 range), sorted by (chromosome string, position)
        self.off = None
        self.chroms = []
        self.ann = None          # object array of annotation strings
        self.fixups = None
        self.pops = (None, None)
        self.n = 0
        self.last_key_row = -1
        self.n_records = self.n_skipped = 0
        self.cache_sources = []
        self.ld_prune = None     # (size, step, threshold) of the LD pruning that produced this panel (subset_panel)

    def __len__(self):
        return self.n

    def save(self, path, sources=()):
        """Write the packed panel to disk (save_panel); PackedPanel.load(path) maps it back without re-parsing the VCF."""
        return save_panel(self, path, sources)

    @staticmethod
    def load(path, mmap=True):
        return load_panel(path, mmap)

    def check_ranges(self):
        pass

    def counts(self):
        """(ref1, alt1, ref2, alt2) per SNP decoded on the host (debug / tests only)."""
        rows = from_b32(self.G, self.n, self.W1 + self.W2)
        out = np.zeros((self.n, 4), dtype=np.int64)
        for p, (w0, w1, ns) in enumerate(((0, self.W1, self.ns1), (self.W1, self.W1 + self.W2, self.ns2))):
            codes = unpack_block(rows[:, w0:w1], ns)
            alt = (codes == CODE_HET).sum(1) + 2 * (codes == CODE_HOMALT).sum(1)
            out[:, 2 * p + 1] = alt
            out[:, 2 * p] = (codes == CODE_HET).sum(1) + 2 * (codes == CODE_HOMREF).sum(1)
        if self.fixups is not None:
            for f in self.fixups:
                out[f["snp"], 2 * f["pop"]] += f["dref"]
                out[f["snp"], 2 * f["pop"] + 1] += f["dalt"]
        return out


# ----------------------------------------------------------------------------------------------- packed-panel cache
# On-disk form of a PackedPanel: replaces the reference's pickle + bz2 cache of the parsed dict (scripts/twoDSFS.py:505-510,
# scripts/src/twoDSFS_class.py:1918-1919).  One file: magic, a JSON header, then the raw arrays at 4096-byte aligned offsets,
# so that a 13 GB matrix is memory-mapped (np.memmap) instead of re-parsed or copied, and can be uploaded straight from the
# page cache.
_CACHE_MAGIC = b"TDSFSPK1"
_CACHE_ALIGN = 4096
_FIX_DT = np.dtype([("snp", "<i8"), ("pop", "<i4"), ("dref", "<i4"), ("dalt", "<i4")], align=True)


def _source_stamp(paths):
    out = []
    for p in paths:
        st = _os.stat(p)
        out.append([_os.path.abspath(str(p)), int(st.st_size), int(st.st_mtime_ns)])
    return out


def save_panel(panel, path, sources=()):
    """Write `panel` to `path` (atomically).  sources: files the panel was built from; their size and mtime are recorded
    so that cached_pack_vcf can tell a stale cache."""
    import json
    vocab, codes = np.unique(np.asarray(panel.ann, dtype=object).astype(str), return_inverse=True) if panel.n else (np.array([], dtype=str), np.zeros(0, np.int64))
    arrays = {"G": np.ascontiguousarray(panel.G, dtype=np.uint32), "pos": np.ascontiguousarray(panel.pos, dtype=np.int64),
              "off": np.ascontiguousarray(panel.off, dtype=np.int64), "ann_codes": np.ascontiguousarray(codes, dtype=np.int32),
              "fixups": np.ascontiguousarray(panel.fixups if panel.fixups is not None else np.zeros(0, _FIX_DT), dtype=_FIX_DT)}
    header = {"version": 1, "n": int(panel.n), "W1": int(panel.W1), "W2": int(panel.W2), "ns1": int(panel.ns1), "ns2": int(panel.ns2),
              "chroms": list(panel.chroms), "pops": list(panel.pops), "last_key_row": int(panel.last_key_row),
              "n_records": int(panel.n_records), "n_skipped": int(panel.n_skipped), "ann_vocab": [str(v) for v in vocab],
              "sources": _source_stamp(sources), "arrays": {}}
    if panel.ld_prune is not None:
        header["ld_prune"] = [int(panel.ld_prune[0]), int(panel.ld_prune[1]), float(panel.ld_prune[2])]
    # two passes: the header's length decides the first offset
    offset = 0
    for _ in range(2):
        blob = json.dumps(header).encode()
        offset = (16 + len(blob) + _CACHE_ALIGN - 1) // _CACHE_ALIGN * _CACHE_ALIGN + _CACHE_ALIGN  # slack for the offsets' digits
        for name, a in arrays.items():
            header["arrays"][name] = {"offset": offset, "nbytes": int(a.nbytes), "count": int(a.shape[0])}
            offset = (offset + a.nbytes + _CACHE_ALIGN - 1) // _CACHE_ALIGN * _CACHE_ALIGN
    blob = json.dumps(header).encode()
    tmp = str(path) + ".tmp%d" % _os.getpid()
    with open(tmp, "wb") as f:
        f.write(_CACHE_MAGIC)
        f.write(len(blob).to_bytes(8, "little"))
        f.write(blob)
        for name, a in arrays.items():
            f.seek(header["arrays"][name]["offset"])
            f.write(memoryview(a).cast("B"))
        f.truncate(max(offset, f.tell()))
    _os.replace(tmp, str(path))
    return str(path)


def load_panel(path, mmap=True):
    """Read a PackedPanel written by save_panel.  mmap=True maps the arrays read-only (no copy of the genotype matrix)."""
    import json
    with open(path, "rb") as f:
        if f.read(8) != _CACHE_MAGIC:
            raise ValueError(f"{path}: not a packed-panel cache")
        hlen = int.from_bytes(f.read(8), "little")
        header = json.loads(f.read(hlen).decode())
    if header.get("version") != 1:
        raise ValueError(f"{path}: unsupported packed-panel cache version {header.get('version')}")

    def arr(name, dt):
        meta = header["arrays"][name]
        if meta["count"] == 0:
            return np.zeros(0, dtype=dt)
        if mmap:
            return np.memmap(path, dtype=dt, mode="r", offset=meta["offset"], shape=(meta["count"],))
        with open(path, "rb") as f:
            f.seek(meta["offset"])
            return np.frombuffer(f.read(meta["nbytes"]), dtype=dt).copy()

    P = PackedPanel()
    P.n, P.W1, P.W2, P.ns1, P.ns2 = header["n"], header["W1"], header["W2"], header["ns1"], header["ns2"]
    P.chroms, P.pops, P.last_key_row = list(header["chroms"]), tuple(header["pops"]), header["last_key_row"]
    P.n_records, P.n_skipped = header["n_records"], header["n_skipped"]
    P.G = arr("G", np.uint32)
    P.pos = np.asarray(arr("pos", np.int64))
    P.off = np.array(arr("off", np.int64))
    vocab = np.array(header["ann_vocab"], dtype=object)
    P.ann = vocab[np.asarray(arr("ann_codes", np.int32))] if P.n else np.array([], dtype=object)
    fx = arr("fixups", _FIX_DT)
    P.fixups = np.array(fx) if len(fx) else None
    P.cache_sources = header["sources"]
    lp = header.get("ld_prune")  # absent: not a pruned panel (every file written before the key existed)
    P.ld_prune = None if lp is None else (int(lp[0]), int(lp[1]), float(lp[2]))
    return P


def subset_panel(panel, keep, ld_prune=None):
    """The rows of `panel` where keep[S] is True, as a new PackedPanel that looks like one the packer could have produced
    from the VCF with only those records: G rebuilt in the B32 layout, positions, annotations and fix-ups (renumbered) of
    the kept rows, `off` recomputed and chromosomes left without rows dropped.  last_key_row (the row of the VCF's last
    record) maps to its kept row; when that row is dropped, to the nearest kept row before it on its chromosome (the last
    record of a position-sorted VCF filtered the same way), else to the panel's last kept row.  n_records / n_skipped stay
    those of the VCF the panel was packed from.  cache_sources is empty, so that cached_pack_vcf never takes the subset for
    the VCF's own cache; ld_prune records the (size, step, threshold) that chose the rows, if any.  The matrix goes through
    row-major form on the host (from_b32 / to_b32): about 3x the panel's genotype bytes of host RAM at the peak."""
    keep = np.asarray(keep, dtype=bool)
    if keep.shape != (panel.n,):
        raise ValueError(f"keep has shape {keep.shape}; the panel has {panel.n} rows")
    idx = np.flatnonzero(keep)
    new_row = np.cumsum(keep) - 1  # new index of every kept row
    off = np.asarray(panel.off, dtype=np.int64)
    per_chrom = np.array([int(keep[off[c]:off[c + 1]].sum()) for c in range(len(panel.chroms))], dtype=np.int64)
    P = PackedPanel()
    P.W1, P.W2, P.ns1, P.ns2, P.pops = panel.W1, panel.W2, panel.ns1, panel.ns2, tuple(panel.pops)
    P.n = len(idx)
    P.G = to_b32(from_b32(panel.G, panel.n, panel.W1 + panel.W2)[idx]) if P.n else np.zeros(0, dtype=np.uint32)
    P.pos = np.asarray(panel.pos, dtype=np.int64)[idx]
    P.chroms = [c for c, k in zip(panel.chroms, per_chrom) if k > 0]
    P.off = np.concatenate([[0], np.cumsum(per_chrom[per_chrom > 0])]).astype(np.int64)
    P.ann = np.asarray(panel.ann, dtype=object)[idx] if P.n else np.array([], dtype=object)
    P.fixups = None
    if panel.fixups is not None and len(panel.fixups):
        fx = np.asarray(panel.fixups)
        fx = fx[keep[fx["snp"]]].copy()
        if len(fx):
            fx["snp"] = new_row[fx["snp"]]
            P.fixups = fx
    last = int(panel.last_key_row)
    P.last_key_row = -1
    if 0 <= last < panel.n and P.n:
        c = int(np.searchsorted(off, last, side="right")) - 1
        before = np.flatnonzero(keep[off[c]:last + 1])
        P.last_key_row = int(new_row[off[c] + before[-1]]) if len(before) else P.n - 1
    P.n_records, P.n_skipped = panel.n_records, panel.n_skipped
    P.cache_sources = []
    P.ld_prune = None if ld_prune is None else (int(ld_prune[0]), int(ld_prune[1]), float(ld_prune[2]))
    return P


def cached_pack_vcf(vcf_filename, popinfo_filename, pop1, pop2, cache_path=None, nthreads=0):
    """pack_vcf with an on-disk cache next to the VCF (`<vcf>.<pop1>.<pop2>.tdsfspk`): reused while the VCF and the popmap
    are unchanged (size + mtime), rebuilt otherwise.  The drop-in for `pickle.load(bz2.open(...))` of the reference."""
    cache_path = cache_path or f"{vcf_filename}.{pop1}.{pop2}.tdsfspk"
    srcs = (vcf_filename, popinfo_filename)
    if _os.path.exists(cache_path):
        try:
            P = load_panel(cache_path)
            if P.cache_sources == _source_stamp(srcs) and tuple(P.pops) == (pop1, pop2) and P.ld_prune is None:
                return P
        except (ValueError, KeyError, OSError):
            pass
    P = pack_vcf(vcf_filename, popinfo_filename, pop1, pop2, nthreads)
    save_panel(P, cache_path, srcs)
    return P


def pack_vcf(vcf_filename, popinfo_filename, pop1, pop2, nthreads=0):
    """gzip VCF + popmap -> PackedPanel with the reference's ingest rules (make_data_dict_vcf, reference :36-138)."""
    L = _packer()
    h = L.tdsfs_pack_vcf(str(vcf_filename).encode(), str(popinfo_filename).encode(), str(pop1).encode(), str(pop2).encode(), int(nthreads))
    if not h:
        msg = L.tdsfs_pack_last_error().decode()
        if "cannot open" in msg:
            raise FileNotFoundError(msg)
        if "not in list" in msg or "invalid literal" in msg:
            raise ValueError(msg)
        if "index out of range" in msg:
            raise IndexError(msg)
        raise RuntimeError(msg)
    owner = _PackOwner(L, h)   # frees the C++ object when the last array that views its memory is gone
    dims = (_C.c_int64 * 8)()
    dims2 = (_C.c_int64 * 4)()
    L.tdsfs_pack_dims(h, dims, dims2)
    S, W1, W2, ns1, ns2, C, nfix, last = [int(v) for v in dims]
    P = PackedPanel()
    P.n, P.W1, P.W2, P.ns1, P.ns2, P.last_key_row = S, W1, W2, ns1, ns2, last
    P.n_records, P.n_skipped = int(dims2[0]), int(dims2[1])
    gw = int(dims2[3])

    def view(ptr, n, dt):
        """zero-copy numpy view of the packer's memory (the 2-bit matrix of a large VCF is the size of host RAM budgets)"""
        if n == 0:
            return np.zeros(0, dtype=dt)
        buf = (_C.c_uint8 * (n * np.dtype(dt).itemsize)).from_address(ptr)
        buf._owner = owner
        return np.frombuffer(buf, dtype=dt)

    P.G = view(L.tdsfs_pack_genotypes(h), gw, np.uint32)
    P.pos = view(L.tdsfs_pack_positions(h), S, np.int32).astype(np.int64)
    P.off = view(L.tdsfs_pack_chrom_off(h), C + 1, np.int64).copy()
    names = L.tdsfs_pack_chrom_names(h).decode()
    P.chroms = names.split("\n")[:-1] if names else []
    vocab = L.tdsfs_pack_ann_vocab(h).decode().split("\n")[:-1]
    codes = view(L.tdsfs_pack_ann_codes(h), S, np.int32)
    P.ann = np.array(vocab, dtype=object)[codes] if S else np.array([], dtype=object)
    fix_dt = np.dtype([("snp", "<i8"), ("pop", "<i4"), ("dref", "<i4"), ("dalt", "<i4")], align=True)
    P.fixups = view(L.tdsfs_pack_fixups(h), nfix, fix_dt).copy() if nfix else None
    P.pops = (pop1, pop2)
    return P


def _raise_pack_error(msg):
    if "cannot open" in msg:
        raise FileNotFoundError(msg)
    if "not in list" in msg or "invalid literal" in msg:
        raise ValueError(msg)
    if "index out of range" in msg:
        raise IndexError(msg)
    raise RuntimeError(msg)


def vcf_to_data_dict(vcf_filename, popinfo_filename, nthreads=0):
    """make_data_dict_vcf (reference :36-138) with the text work in C++ (csrc/vcf_pack.cpp, counts mode: gzip or BGZF, parsed
    in parallel); only the construction of the dict itself stays in Python.  Same dict, same exception types."""
    L = _packer()
    h = L.tdsfs_vcf_counts(str(vcf_filename).encode(), str(popinfo_filename).encode(), int(nthreads))
    if not h:
        _raise_pack_error(L.tdsfs_pack_last_error().decode())
    try:
        dims = (_C.c_int64 * 4)()
        L.tdsfs_vcf_counts_dims(h, dims)
        n, npop, key_bytes = int(dims[0]), int(dims[1]), int(dims[2])

        def arr(ptr, count, dt):
            if count == 0:
                return np.zeros(0, dtype=dt)
            return np.frombuffer((_C.c_uint8 * (count * np.dtype(dt).itemsize)).from_address(ptr), dtype=dt)

        pops = L.tdsfs_vcf_counts_pops(h).decode().split("\n")[:-1]
        vocab = L.tdsfs_vcf_counts_vocab(h).decode().split("\n")[:-1]
        raw = _C.string_at(L.tdsfs_vcf_counts_keys(h), key_bytes) if key_bytes else b""
        # key_off holds BYTE offsets: a str can be sliced with them only when every character is one byte
        blob = raw.decode() if raw.isascii() else None
        off = arr(L.tdsfs_vcf_counts_key_off(h), n + 1, np.int64).tolist()
        refalt = _C.string_at(L.tdsfs_vcf_counts_refalt(h), 2 * n).decode() if n else ""
        ann = arr(L.tdsfs_vcf_counts_ann_codes(h), n, np.int32).tolist()
        ncols = arr(L.tdsfs_vcf_counts_ncols(h), n, np.int32).tolist()
        first = arr(L.tdsfs_vcf_counts_first_col(h), npop, np.int32).tolist()
        cnt = arr(L.tdsfs_vcf_counts_cnt(h), n * npop * 2, np.int32).reshape(n, npop, 2).tolist() if n and npop else [[] for _ in range(n)]
        # a population enters calls_dict when its first zipped column is reached (:118-130); insertion order = first appearance
        order = sorted(range(npop), key=lambda p: first[p])
        full = max(first) + 1 if first else 0
        data_dict = {}
        for i in range(n):
            ref, alt = refalt[2 * i], refalt[2 * i + 1]
            c, nc = cnt[i], ncols[i]
            if nc >= full:
                calls = {pops[p]: (c[p][0], c[p][1]) for p in order}
            else:
                calls = {pops[p]: (c[p][0], c[p][1]) for p in order if first[p] < nc}
            key = blob[off[i]:off[i + 1]] if blob is not None else raw[off[i]:off[i + 1]].decode()
            data_dict[key] = {"segregating": (ref, alt), "context": "-" + ref + "-", "calls": calls,
                                                  "annotation": vocab[ann[i]]}
        return data_dict
    finally:
        L.tdsfs_vcf_counts_free(h)
