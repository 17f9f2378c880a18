"""deepgrp_b200.preprocessing -- the data formats either side of the prediction path (SURVEY.md
section 8f rank 4): the ``Data`` tuple ``predict_complete`` takes, the edge-N cut and the label matrix the
reference's evaluation builds it from (``deepgrp/preprocessing.py``), and the ``.npz`` one-hot file
``preprocess_sequence`` writes (``deepgrp/_scripts/preprocess_sequence.py``).  The label / file handling here
is host-side numpy; the one-hot matrix itself comes from the GPU encode kernel (no CPU fallback).

    python -m deepgrp_b200.preprocessing FASTAFILE.gz [--force]      # writes FASTAFILE.gz.npz
"""
import argparse
import gzip
import hashlib
import os
import sys
from typing import BinaryIO, Dict, List, NamedTuple, Tuple

import numpy as np

# Collection of forward one hot encoded sequence and true annotations (deepgrp/preprocessing.py:72)
Data = NamedTuple("Data", [("fwd", np.ndarray), ("truelbl", np.ndarray)])


def read_annotation(filename, repeats_to_search: List[int]) -> Dict[str, np.ndarray]:
    """The whitespace-separated table ``parse_rm`` writes (chromosome, begin, end, repeat number; further columns are
    ignored, no header) -> ``{chromosome: int64[n, 3]}`` of (begin, end, number), in file order, for the lines whose
    repeat number is searched for.  Coordinates are 0-based and half-open as ``preprocess_y`` indexes them.  A
    non-integer begin, end or number, or a negative coordinate, on any line is a ``ValueError``."""
    import pandas as pd
    try:
        table = pd.read_csv(filename, sep=r"\s+", header=None, index_col=False, usecols=[0, 1, 2, 3],
                            names=["chromosom", "begin", "end", "repeatnumber"], dtype=str)
    except pd.errors.EmptyDataError:
        return {}
    cols = ("begin", "end", "repeatnumber")
    for col in cols:
        ok = table[col].str.fullmatch(r"[+-]?[0-9]+").fillna(False).to_numpy(bool)
        if not ok.all():
            line = int(np.argmin(ok))
            raise ValueError("annotation row %d: %s %r is not an integer" % (line + 1, col, table[col].iloc[line]))
    values = table[list(cols)].to_numpy().astype(np.int64)
    negative = (values[:, :2] < 0).any(axis=1)
    if negative.any():
        line = int(np.argmax(negative))
        raise ValueError("annotation row %d: negative coordinate %d %d" % (line + 1, values[line, 0], values[line, 1]))
    keep = np.isin(values[:, 2], np.asarray(list(repeats_to_search), dtype=np.int64))
    chrom = table["chromosom"].to_numpy()[keep]
    values = values[keep]
    out = {}
    if len(chrom):
        names, first, inverse = np.unique(chrom, return_index=True, return_inverse=True)
        order = np.argsort(inverse, kind="stable")
        bounds = np.searchsorted(inverse[order], np.arange(len(names) + 1))
        for k in np.argsort(first):
            out[str(names[k])] = np.ascontiguousarray(values[order[bounds[k]:bounds[k + 1]]])
    return out


def preprocess_y(filename, chromosom: str, length: int, repeats_to_search: List[int]) -> np.ndarray:
    """Reference ``deepgrp/preprocessing.py:9-46``: the annotation table (:func:`read_annotation`) -> one-hot
    annotations int8[len(repeats) + 1, length]; row ``r`` is set on [begin, end) of every line of ``chromosom`` whose
    repeat number ``r`` is searched for (the number itself is the row index, as in the reference), row 0 wherever no
    other row is."""
    lines = read_annotation(filename, repeats_to_search).get(chromosom, np.zeros((0, 3), np.int64))
    yarray = np.zeros((len(repeats_to_search) + 1, length), dtype=np.int8)
    for begin, end, number in lines:
        yarray[number, begin:end] = 1
    yarray[0, ~yarray[1:].any(axis=0)] = 1
    return yarray


def drop_start_end_n(fwd: np.ndarray, array: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Reference ``deepgrp/preprocessing.py:49-68``: cut both arrays to the columns between the first and
    the last column with an A/C/G/T bit -- ``[first, last)``: the slice end is the last such column itself,
    so that column is dropped too (the reference's behaviour, pinned by its test)."""
    has_base = fwd[0:4].sum(axis=0) > 0
    first = int(np.argmax(has_base))
    last = fwd.shape[1] - 1 - int(np.argmax(has_base[::-1]))
    return fwd[:, first:last], array[:, first:last]


def fastaparser(filestream: BinaryIO) -> Tuple[str, str, str]:
    """Reference ``deepgrp/_scripts/preprocess_sequence.py:19-38``: single-record FASTA (bytes lines) ->
    (header, md5 of the stripped sequence lines as they are in the file, upper-cased sequence)."""
    md5 = hashlib.md5()
    header, parts = "", []
    for line in filestream:
        line = line.strip()
        if line[0] == ord(">"):
            header = line[1:].decode()
        else:
            parts.append(line.decode().upper())
            md5.update(line)
    return header, md5.hexdigest(), "".join(parts)


def one_hot_untrimmed(seq: str) -> np.ndarray:
    """int8[5, len(seq)] with rows A, C, G, T, N as ``preprocess_sequence`` builds it (:69-72): nothing is
    trimmed, and a character outside ``ACGTN`` is a ``KeyError`` as in the reference's ``_ENCODEDICT``.  The
    matrix of the trimmed sequence comes from the GPU encode kernel; the edge-N columns are put back here."""
    from . import sequence as dgsequence
    raw = np.frombuffer(seq.encode("latin-1"), dtype=np.uint8)
    bad = ~np.isin(raw, np.frombuffer(b"ACGTN", dtype=np.uint8))
    if bad.any():
        raise KeyError(seq[int(np.argmax(bad))])
    out = np.zeros((5, raw.size), dtype=np.int8)
    if raw.size == 0:
        return out
    if (raw == ord("N")).all():
        out[4] = 1
        return out
    start, fwd = dgsequence.one_hot_encode_dna_sequence(seq)
    out[4, :start] = 1
    out[:, start:start + fwd.shape[1]] = fwd
    out[4, start + fwd.shape[1]:] = 1
    return out


def load_onehot_npz(path) -> Tuple[np.ndarray, str]:
    """The file ``preprocess_sequence`` writes: ``fwd`` int8[5, L] and ``hash`` = [md5] -> (fwd, md5)."""
    with np.load(path) as data:
        return np.ascontiguousarray(data["fwd"], dtype=np.int8), str(data["hash"][0])


def preprocess_sequence(fastafile: str, force: bool = False) -> bool:
    """Reference ``preprocess_sequence.main`` (:41-74): gzip FASTA -> ``fastafile + '.npz'`` unless a file with
    the same sequence hash is already there.  Returns whether the file was (re)written."""
    with gzip.open(fastafile, "rb") as fh:
        _, hash_val, seq = fastaparser(fh)
    create_new = force
    try:
        if load_onehot_npz(fastafile + ".npz")[1] != hash_val:
            create_new = True
    except (IOError, KeyError):
        create_new = True
    if create_new:
        np.savez_compressed(fastafile, fwd=one_hot_untrimmed(seq), hash=np.array([hash_val]))
    return create_new


def main(argv=None):
    parser = argparse.ArgumentParser(description="Format fasta file to onehot encoded sequences")
    parser.add_argument("FASTAFILE", type=str, help="Fastafile (gzip)")
    parser.add_argument("--force", action="store_true", help="forces recreation even if files not changed")
    args = parser.parse_args(argv)
    try:
        preprocess_sequence(args.FASTAFILE, args.force)
    except IOError:
        sys.stderr.write("Could not open file!\n")
        sys.exit(1)


if __name__ == "__main__":
    main()
