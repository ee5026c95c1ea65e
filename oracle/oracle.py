"""ctypes front-end of oracle/oligo_oracle.c — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product (kmertools_b200, pykmertools, the C-ABI library) never does.

Also holds a minimal FASTA/FASTQ(.gz) reader restating what the reference's own tests pin for
ktio/src/seq.rs:97-155 (multi-line FASTA concatenated, id = first token, 4-line FASTQ, gzip), used to
feed the oracle from the golden fixture files.
"""
from __future__ import annotations

import ctypes as C
import gzip
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SO = _HERE / "_build" / "liboligo_oracle.so"
_lib = None


def build(force: bool = False) -> Path:
    """Compile the oracle with the Makefile next to this file (gcc, OpenMP)."""
    src = _HERE / "oligo_oracle.c"
    if force or not _SO.exists() or _SO.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(_HERE), "-s"], check=True)
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(_SO))
        u8p, u64p, f64p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint64), C.POINTER(C.c_double)
        L.ktb_oracle_nt4.restype = C.c_uint8
        L.ktb_oracle_nt4.argtypes = [C.c_uint8]
        L.ktb_oracle_rev_comp.restype = C.c_uint64
        L.ktb_oracle_rev_comp.argtypes = [C.c_uint64, C.c_int]
        L.ktb_oracle_kmers.restype = C.c_uint64
        L.ktb_oracle_kmers.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
        L.ktb_oracle_kmer_pos_maps.restype = C.c_uint64
        L.ktb_oracle_kmer_pos_maps.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.ktb_oracle_dim.restype = C.c_uint64
        L.ktb_oracle_dim.argtypes = [C.c_int, C.c_int]
        L.ktb_oracle_numeric_to_kmer.restype = None
        L.ktb_oracle_numeric_to_kmer.argtypes = [C.c_uint64, C.c_int, C.c_char_p]
        L.ktb_oracle_kmer_to_numeric.restype = None
        L.ktb_oracle_kmer_to_numeric.argtypes = [C.c_char_p, u64p, u64p]
        L.ktb_oracle_vectorise_one.restype = C.c_uint64
        L.ktb_oracle_vectorise_one.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int,
                                               C.c_int, C.c_void_p, C.c_uint64]
        L.ktb_oracle_vectorise_batch.restype = C.c_int
        L.ktb_oracle_vectorise_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                                                 C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.ktb_oracle_baseline_batch.restype = C.c_double
        L.ktb_oracle_baseline_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                                                C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.ktb_oracle_max_threads.restype = C.c_int
        L.ktb_oracle_header.restype = C.c_int
        L.ktb_oracle_baseline_text.restype = C.c_uint64
        L.ktb_oracle_baseline_text.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                               C.c_char_p, C.c_int, C.POINTER(C.c_int)]
        L.ktb_oracle_header.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint64]
        L.ktb_oracle_format_row.restype = C.c_int64
        L.ktb_oracle_format_row.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_char_p, C.c_char_p,
                                            C.c_uint64]
        L.ktb_oracle_check_quot_f32.restype = C.c_uint64
        L.ktb_oracle_check_quot_f32.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
        _ = (u8p, f64p)
        _lib = L
    return _lib


# ----------------------------------------------------------------------------- primitives

def nt4(b: int) -> int:
    return int(lib().ktb_oracle_nt4(b))


def rev_comp(kmer: int, k: int) -> int:
    return int(lib().ktb_oracle_rev_comp(kmer, k))


def kmers(seq: bytes, k: int) -> list[tuple[int, int]]:
    """All (forward, reverse-complement) pairs KmerGenerator would yield (kmer/src/kmer.rs:80-106)."""
    n = len(seq)
    f = np.zeros(max(n, 1), dtype=np.uint64)
    r = np.zeros(max(n, 1), dtype=np.uint64)
    buf = np.frombuffer(seq, dtype=np.uint8) if n else np.zeros(1, dtype=np.uint8)
    m = lib().ktb_oracle_kmers(buf.ctypes.data, n, k, f.ctypes.data, r.ctypes.data)
    return [(int(f[i]), int(r[i])) for i in range(m)]


def kmer_arrays(buf, k: int, want_pairs: bool = True):
    """kmers() as two uint64 arrays and the count, without building tuples: (f, r, count).  `buf` is bytes or a uint8
    array (copied only when not contiguous).  With want_pairs=False only the count is computed and returned."""
    if isinstance(buf, (bytes, bytearray, memoryview)):
        buf = np.frombuffer(buf, dtype=np.uint8)
    buf = np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)
    n = buf.size
    src = buf if n else np.zeros(1, dtype=np.uint8)
    if not want_pairs:
        return int(lib().ktb_oracle_kmers(src.ctypes.data, n, k, None, None))
    cap = max(n - k + 1, 0)
    f = np.empty(max(cap, 1), dtype=np.uint64)
    r = np.empty(max(cap, 1), dtype=np.uint64)
    m = int(lib().ktb_oracle_kmers(src.ctypes.data, n, k, f.ctypes.data, r.ctypes.data))
    assert m <= cap
    return f[:m], r[:m], m


def kmer_pos_maps(k: int) -> tuple[np.ndarray, np.ndarray, int]:
    """(pos_map[4^k], pos_to_kmer[count], count) — kmer/src/kmer.rs:54-73."""
    n = 4 ** k
    pos_map = np.zeros(n, dtype=np.uint64)
    p2k = np.zeros(n, dtype=np.uint64)
    cnt = int(lib().ktb_oracle_kmer_pos_maps(k, pos_map.ctypes.data, p2k.ctypes.data))
    return pos_map, p2k[:cnt].copy(), cnt


def dim(k: int, canonical: bool = True) -> int:
    return int(lib().ktb_oracle_dim(k, int(canonical)))


def numeric_to_kmer(kmer: int, k: int) -> str:
    buf = C.create_string_buffer(k + 1)
    lib().ktb_oracle_numeric_to_kmer(kmer, k, buf)
    return buf.value.decode()


def kmer_to_numeric(kmer: str) -> tuple[int, int]:
    f, r = C.c_uint64(), C.c_uint64()
    lib().ktb_oracle_kmer_to_numeric(kmer.encode(), C.byref(f), C.byref(r))
    return int(f.value), int(r.value)


def header(k: int, canonical: bool = True) -> list[str]:
    d = dim(k, canonical)
    buf = C.create_string_buffer(d * k + 1)
    rc = lib().ktb_oracle_header(k, int(canonical), buf, d * k)
    assert rc == 0
    raw = buf.raw[: d * k].decode()
    return [raw[i * k:(i + 1) * k] for i in range(d)]


# ----------------------------------------------------------------------------- vectors

def pack(seqs: list[bytes]) -> tuple[np.ndarray, np.ndarray]:
    """Concatenate sequences into (bases u8[total], offsets u64[n+1])."""
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    if seqs:
        offsets[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy() if seqs else np.zeros(0, np.uint8)
    return bases, offsets


def vectorise_batch(bases: np.ndarray, offsets: np.ndarray, k: int, canonical: bool = True,
                    norm_mode: int = 1, threads: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """Oracle rows (n x dim f64) and valid-window totals (u64[n]).

    norm_mode 0 counts, 1 CLI normalisation, 2 pybindings normalisation (raw mode halves)."""
    n = len(offsets) - 1
    d = dim(k, canonical)
    out = np.zeros((n, d), dtype=np.float64)
    totals = np.zeros(n, dtype=np.uint64)
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    bptr = bases.ctypes.data if bases.size else np.zeros(1, np.uint8).ctypes.data
    lib().ktb_oracle_vectorise_batch(bptr, offsets.ctypes.data, n, k, int(canonical), norm_mode,
                                     out.ctypes.data, totals.ctypes.data, threads)
    return out, totals


def vectorise_one(seq: bytes, k: int, canonical: bool = True, norm_mode: int = 1) -> np.ndarray:
    bases, offsets = pack([seq])
    return vectorise_batch(bases, offsets, k, canonical, norm_mode, threads=1)[0][0]


def baseline_batch(bases: np.ndarray, offsets: np.ndarray, k: int, canonical: bool = True,
                   norm_mode: int = 1, threads: int = 0) -> tuple[float, int]:
    """Run the timed CPU stand-in once; returns (checksum, threads used)."""
    used = C.c_int(0)
    n = len(offsets) - 1
    cs = lib().ktb_oracle_baseline_batch(bases.ctypes.data, offsets.ctypes.data, n, k, int(canonical),
                                         norm_mode, threads, C.byref(used))
    return float(cs), int(used.value)


def baseline_text(bases: np.ndarray, offsets: np.ndarray, k: int, canonical: bool = True, norm: bool = True,
                  delim: str = " ", path: str | None = None, threads: int = 0) -> tuple[int, int]:
    """CPU baseline of the file-level path (vectorise + format every value + ordered write), composition/src/oligo.rs:
    126-144.  Returns (text bytes, threads used)."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    used = C.c_int(0)
    nbytes = lib().ktb_oracle_baseline_text(bases.ctypes.data if bases.size else np.zeros(1, np.uint8).ctypes.data,
                                            offsets.ctypes.data, len(offsets) - 1, k, int(canonical), int(norm),
                                            delim.encode(), os.fsencode(path) if path else None, threads, C.byref(used))
    return int(nbytes), int(used.value)


def check_quot_f32(dlo: int, dhi: int, cstep: int = 1) -> int:
    """Mismatches of the GPU's f32 division sequence vs (float)(f64 quotient) over a divisor range."""
    return int(lib().ktb_oracle_check_quot_f32(dlo, dhi, cstep))


def max_threads() -> int:
    return int(lib().ktb_oracle_max_threads())


def format_rows(rows: np.ndarray, norm: bool, delim: str = " ") -> bytes:
    """Text body exactly as composition/src/oligo.rs:130-143 writes it."""
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    n, d = rows.shape
    cap = d * 32 + 16
    buf = C.create_string_buffer(cap)
    out = []
    for i in range(n):
        w = lib().ktb_oracle_format_row(rows[i].ctypes.data, d, int(norm), delim.encode(), buf, cap)
        assert w > 0
        out.append(buf.raw[:w])
    return b"".join(out)


def comp_oligo_text(path: str | os.PathLike, k: int, canonical: bool = True, norm: bool = True,
                    delim: str = " ", with_header: bool = False) -> bytes:
    """What `kmertools comp oligo -i path -k k [...]` writes (composition/src/oligo.rs:88-229)."""
    seqs = [s for _, s in read_fastx(path)]
    bases, offsets = pack(seqs)
    rows, _ = vectorise_batch(bases, offsets, k, canonical, 1 if norm else 0)
    body = format_rows(rows, norm, delim)
    if with_header:
        body = (delim.join(header(k, canonical)) + "\n").encode() + body
    return body


def _rust_f64(v: float) -> str:
    """Rust's `{}` of an f64: the shortest digits that round-trip, never an exponent, no trailing ".0"."""
    return np.format_float_positional(v, unique=True, trim="-")


def cgr_points(k: int, vecsize: int) -> list[tuple[float, float]]:
    """The fixed point of every canonical k-mer, in header(k, True) order (composition/src/oligocgr.rs:123-143,165-190):
    the midpoint recurrence from (v/2, v/2) towards the corner of each base, A (0,0), T (v,0), G (v,v), C (0,v)."""
    v = float(vecsize)
    corner = {"A": (0.0, 0.0), "T": (v, 0.0), "G": (v, v), "C": (0.0, v)}
    pts = []
    for kmer in header(k, True):
        x = y = v / 2.0
        for b in kmer:
            cx, cy = corner[b]
            x, y = (cx + x) / 2.0, (cy + y) / 2.0
        pts.append((x, y))
    return pts


def comp_cgr_text(path: str | os.PathLike, k: int, vecsize: int, norm: bool = True) -> bytes:
    """What `kmertools comp cgr -i path -k k -v vecsize [-c]` writes (composition/src/oligocgr.rs:88-101,123-190):
    one line per record, "(x,y,value)" per canonical k-mer joined by spaces; a frequency is `{}` of the f64 quotient,
    a count `{}` of an integral f64."""
    seqs = [s for _, s in read_fastx(path)]
    rows, _ = vectorise_batch(*pack(seqs), k, True, 1 if norm else 0)
    pref = ["(%s,%s," % (_rust_f64(x), _rust_f64(y)) for x, y in cgr_points(k, vecsize)]
    d = len(pref)
    zero = [p + "0) " for p in pref]
    zero[-1] = zero[-1][:-1] + "\n"
    lines = []
    for row in rows:   # most cells of short records are 0: rebuild only the others
        cells = list(zero)
        for j in np.flatnonzero(row):
            v = row[j]
            cells[j] = pref[j] + (_rust_f64(v) if norm else str(int(v))) + (")\n" if j == d - 1 else ") ")
        lines.append("".join(cells))
    return "".join(lines).encode()


# ----------------------------------------------------------------------------- feeder

def read_fastx(path: str | os.PathLike) -> list[tuple[str, bytes]]:
    """(id, sequence) records of a FASTA/FASTQ file, optionally .gz (ktio/src/seq.rs:29-42,141-155)."""
    p = str(path)
    opener = gzip.open if p.endswith(".gz") else open
    with opener(p, "rb") as fh:
        data = fh.read()
    recs: list[tuple[str, bytes]] = []
    lines = data.split(b"\n")
    if not data:
        return recs
    if data[:1] == b">":
        name, parts = None, []
        for ln in lines:
            ln = ln.rstrip(b"\r")
            if ln.startswith(b">"):
                if name is not None:
                    recs.append((name, b"".join(parts)))
                toks = ln[1:].split()
                name, parts = (toks[0].decode() if toks else ""), []
            elif name is not None:
                parts.append(ln)
        if name is not None:
            recs.append((name, b"".join(parts)))
    else:
        i = 0
        while i + 1 < len(lines):
            if not lines[i].startswith(b"@"):
                i += 1
                continue
            toks = lines[i][1:].split()
            recs.append((toks[0].decode() if toks else "", lines[i + 1].rstrip(b"\r")))
            i += 4
    return recs
