"""On-disk compatibility with the reference's index directories (SURVEY §8f-1).

`FaissVS.index` writes `{index_dir}/index` with faiss.write_index and `{index_dir}/vecs` as a pickle of the
ndarray it was given (lotus/vector_store/faiss_vs.py:27-30); `load_index` reads both (:32-36).
The faiss file of an IndexFlat is (faiss/impl/index_write.cpp, write_index + write_index_header):
    fourcc "IxFI" (inner product) | "IxF2" (L2)                      4 bytes
    d            int32          ntotal       int64
    dummy, dummy int64 (1<<20)  is_trained   uint8      metric_type int32   [metric_arg float32 if metric_type > 1]
    size         uint64 = number of float32 values (WRITEXBVECTOR writes codes.size()/4)
    data         float32[ntotal*d]
The file of an IndexScalarQuantizer(d, QT_fp16) — factory string "SQfp16" — is (index_write.cpp, write_ScalarQuantizer):
    fourcc "IxSQ"                                                    4 bytes
    the same index header as above
    qtype int32 = 4 (QT_fp16)   rangestat int32 = 0   rangestat_arg float32 = 0
    d uint64                    code_size uint64 = 2 * d
    trained      uint64 count = 0 (no float32 values follow)
    codes        uint64 byte count = ntotal * 2 * d, then the fp16 rows (IEEE binary16, little endian)
This module reads and writes those layouts with numpy only, so directories produced by either backend load in both.
The IxSQ layout is restated from upstream faiss; it has not been checked against a file written by a running faiss here.
"""
from __future__ import annotations

import os
import pickle
import struct

import numpy as np

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1


FLAT, SQFP16 = "Flat", "SQfp16"  # the index kinds (factory strings) this module reads and writes
QT_FP16 = 4  # faiss ScalarQuantizer::QT_fp16


def _header(d: int, n: int, metric: int) -> bytes:
    return struct.pack("<iqqqBi", d, n, 1 << 20, 1 << 20, 1, metric)


def write_flat_index(path: str, x: np.ndarray, metric: int) -> None:
    x = np.ascontiguousarray(x, dtype=np.float32)
    n, d = x.shape
    fourcc = b"IxFI" if metric == METRIC_INNER_PRODUCT else b"IxF2"
    with open(path, "wb") as f:
        f.write(fourcc)
        f.write(_header(d, n, metric))
        f.write(struct.pack("<Q", n * d))
        x.tofile(f)


def write_sq_fp16_index(path: str, x16: np.ndarray, metric: int) -> None:
    """faiss IndexScalarQuantizer(d, QT_fp16, metric) holding the rows `x16` (np.float16 [n, d])."""
    x16 = np.ascontiguousarray(x16, dtype=np.float16)
    n, d = x16.shape
    with open(path, "wb") as f:
        f.write(b"IxSQ")
        f.write(_header(d, n, metric))
        f.write(struct.pack("<iif", QT_FP16, 0, 0.0))
        f.write(struct.pack("<QQ", d, 2 * d))
        f.write(struct.pack("<Q", 0))
        f.write(struct.pack("<Q", n * 2 * d))
        x16.astype("<f2", copy=False).tofile(f)


def read_index(path: str):
    """-> (x, metric, kind): kind FLAT gives x float32 [n,d]; kind SQFP16 gives x np.float16 [n,d] (the stored rows)."""
    with open(path, "rb") as f:
        fourcc = f.read(4)
    if fourcc != b"IxSQ":
        x, metric = read_flat_index(path)
        return x, metric, FLAT
    with open(path, "rb") as f:
        f.read(4)
        d, n, _d1, _d2, _trained, metric = struct.unpack("<iqqqBi", f.read(4 + 8 * 3 + 1 + 4))
        if metric > 1:
            f.read(4)
        qtype, _rangestat, _rangestat_arg = struct.unpack("<iif", f.read(12))
        if qtype != QT_FP16:
            raise ValueError(f"{path}: IndexScalarQuantizer with qtype {qtype}; only QT_fp16 ({QT_FP16}, factory string 'SQfp16') "
                             "is supported")
        sq_d, code_size = struct.unpack("<QQ", f.read(16))
        (n_trained,) = struct.unpack("<Q", f.read(8))
        f.read(4 * n_trained)
        (nbytes,) = struct.unpack("<Q", f.read(8))
        if sq_d != d or code_size != 2 * d or nbytes != n * 2 * d:
            raise ValueError(f"{path}: corrupt IndexScalarQuantizer payload (d {sq_d}, code size {code_size}, {nbytes} bytes for {n}x{d})")
        x = np.fromfile(f, dtype="<f2", count=n * d).astype(np.float16, copy=False).reshape(n, d)
    return x, metric, SQFP16


def read_flat_index(path: str, mmap: bool = False):
    """-> (x float32 [n,d], metric)."""
    with open(path, "rb") as f:
        fourcc = f.read(4)
        if fourcc not in (b"IxFI", b"IxF2", b"IxFl"):
            raise ValueError(f"{path}: not a faiss IndexFlat file (fourcc {fourcc!r}); only factory strings 'Flat' and 'SQfp16' "
                             "are supported")
        d, n, _d1, _d2, _trained, metric = struct.unpack("<iqqqBi", f.read(4 + 8 * 3 + 1 + 4))
        if metric > 1:
            f.read(4)
        (size,) = struct.unpack("<Q", f.read(8))
        if size != n * d:
            raise ValueError(f"{path}: corrupt IndexFlat payload ({size} values for {n}x{d})")
        off = f.tell()
        if mmap:
            x = np.memmap(path, dtype=np.float32, mode="r", offset=off, shape=(n, d))
        else:
            x = np.fromfile(f, dtype=np.float32, count=n * d).reshape(n, d)
    return x, metric


def write_index_dir(index_dir: str, embeddings, x_f32: np.ndarray, metric: int, kind: str = FLAT) -> None:
    """kind FLAT writes x_f32 as an IndexFlat; kind SQFP16 writes its fp16 rounding as an IndexScalarQuantizer(QT_fp16)."""
    os.makedirs(index_dir, exist_ok=True)
    with open(f"{index_dir}/vecs", "wb") as fp:
        pickle.dump(embeddings, fp)
    if kind == SQFP16:
        with np.errstate(over="ignore"):
            write_sq_fp16_index(f"{index_dir}/index", np.asarray(x_f32, dtype=np.float32).astype(np.float16), metric)
    else:
        write_flat_index(f"{index_dir}/index", x_f32, metric)


def read_index_dir(index_dir: str, with_kind: bool = False):
    """-> (vecs as stored by the caller of index(), x, metric), plus the index kind (FLAT / SQFP16) when with_kind. x is float32
    for FLAT and np.float16 for SQFP16. `vecs` falls back to x when the pickle is absent."""
    if not os.path.isdir(index_dir):
        raise ValueError(f"Index directory {index_dir} not found")
    x, metric, kind = read_index(f"{index_dir}/index")
    vecs = None
    vp = f"{index_dir}/vecs"
    if os.path.exists(vp):
        with open(vp, "rb") as fp:
            vecs = pickle.load(fp)
    out = (vecs if vecs is not None else x), x, metric
    return (*out, kind) if with_kind else out
