"""Repeat masking of FASTA text (``deepgrp predict --mask``): the host restatement of its semantics, checked against
the reference reader (CPU only).

``mask_fasta`` below is the checker of the GPU mask kernels (tests/test_gpu_mask.py).  It is written from the
reference reader's rules (``deepgrp/__main__.py:20-43``, restated in ``_read_multi_fasta``), line by line, and not
from the kernel:

* lines end at ``\\n``, ``\\r\\n`` or a lone ``\\r`` (universal newlines);
* a line that is empty after ``str.strip()`` is an error (``IndexError``);
* a stripped line starting with ``>`` opens a record, which is kept when the rest of the line is not empty;
* every other line is sequence text: each byte inside its strip span is a position of the current kept record
  (none before the first ``>`` or in a record with an empty header), internal spaces and any other byte included.

Position ``p`` of kept record ``r`` is masked when a row ``(start, end)`` of ``r`` has ``start <= p < end``.  A
masked ASCII capital is lower-cased (``soft``) or every masked byte becomes ``N`` (``hard``); all other bytes are
copied unchanged."""
import io
import random

import numpy as np
import pytest

from conftest import messy_fasta

WS = frozenset(list(range(9, 14)) + list(range(28, 33)))     # what str.strip() removes from ASCII text


def spans(text: bytes):
    """Byte spans ``(begin, end)`` of the sequence lines of every kept record, line by line: ``[[span, ...], ...]``."""
    out, current = [], None
    off = 0
    for line in text.splitlines(keepends=True):           # bytes.splitlines: exactly \n, \r\n and \r
        body = len(line) - (2 if line.endswith(b"\r\n") else 1 if line.endswith((b"\n", b"\r")) else 0)
        a, b = 0, body
        while a < b and line[a] in WS:
            a += 1
        while b > a and line[b - 1] in WS:
            b -= 1
        if a == b:
            raise IndexError("string index out of range")
        if line[a] == ord(">"):
            current = [] if b > a + 1 else None
            if current is not None:
                out.append(current)
        elif current is not None:
            current.append((off + a, off + b))
        off += len(line)
    return out


def positions(text: bytes):
    """Byte offsets of the positions of every kept record, in order (int64 arrays)."""
    return [np.concatenate([np.arange(a, b, dtype=np.int64) for a, b in sp]) if sp else np.zeros(0, np.int64)
            for sp in spans(text)]


def mask_fasta(text: bytes, rows_by_record, mode: str) -> bytes:
    """``text`` with the positions covered by ``rows_by_record[r]`` (``(start, end)`` pairs of kept record ``r``)
    masked in ``mode`` (``soft`` or ``hard``)."""
    assert mode in ("soft", "hard")
    out = np.frombuffer(text, dtype=np.uint8).copy()
    for r, offs in enumerate(positions(text)):
        for start, end in rows_by_record.get(r, ()):
            idx = offs[start:end]
            if mode == "hard":
                out[idx] = ord("N")
            else:
                v = out[idx]
                out[idx] = np.where((v >= ord("A")) & (v <= ord("Z")), v + 32, v)
    return out.tobytes()


def reader_records(text: bytes):
    from deepgrp_b200.__main__ import _read_multi_fasta
    return list(_read_multi_fasta(io.StringIO(text.decode("latin-1"), newline=None)))


HAND_MADE = [
    b"",
    b">a\nACGT\n",
    b">a\r\nAC GT\r\nacgt\r\n>b\rNNxy\r\n",                       # CRLF, a lone CR, an internal space
    b"\t>a \t\n  AC\tGT  \n>\n TTTT\n>c\nGG",                   # '>' after whitespace, empty header, no final newline
    b"preamble text\nACGT\n>r1\nA\nC\n>r2\n\x1cAC\x1fG\x0b\n",  # preamble, 1-byte lines, strip whitespace 28-31
    b">only headers\n>another\n>\n",
    b">x\nA\x00B\xffC*-\n",                                      # bytes that are not bases are positions too
]


def all_texts():
    texts = list(HAND_MADE)
    for seed in range(60):
        text = messy_fasta(seed).encode()
        try:
            reader_records(text)
        except IndexError:
            continue
        texts.append(text)
    return texts


@pytest.mark.parametrize("text", all_texts())
def test_positions_are_what_the_reader_reads(text):
    recs = reader_records(text)
    pos = positions(text)
    assert len(pos) == len(recs)
    for (_, seq), offs in zip(recs, pos):
        assert bytes(text[int(o)] for o in offs).decode("latin-1").upper() == seq


@pytest.mark.parametrize("text", [b">a\n\nAC\n", b">a\nAC\n \n", b"\n>a\nAC\n", b">a\nAC\n\t"])
def test_blank_lines_are_errors(text):
    with pytest.raises(IndexError):
        reader_records(text)
    with pytest.raises(IndexError):
        positions(text)


def test_mask_fasta_semantics():
    text = b"pre\n>a\r\nAcg T\r\n>\nGGGG\n>b\nTTTT"
    rows = {0: [(0, 2), (3, 5)], 1: [(1, 4)]}
    assert mask_fasta(text, rows, "soft") == b"pre\n>a\r\nacg t\r\n>\nGGGG\n>b\nTttt"
    assert mask_fasta(text, rows, "hard") == b"pre\n>a\r\nNNgNN\r\n>\nGGGG\n>b\nTNNN"
    assert mask_fasta(text, {}, "soft") == text


def test_mask_fasta_random_rows_cover_what_they_say():
    rng = random.Random(7)
    for text in all_texts():
        pos = positions(text)
        rows = {}
        for r, offs in enumerate(pos):
            cuts = sorted(rng.sample(range(len(offs) + 1), min(len(offs) + 1, 6)))
            rows[r] = [(a, b) for a, b in zip(cuts[::2], cuts[1::2]) if a < b]
        hard = mask_fasta(text, rows, "hard")
        covered = {int(pos[r][p]) for r, rr in rows.items() for a, b in rr for p in range(a, b)}
        assert len(hard) == len(text)
        for i, (x, y) in enumerate(zip(text, hard)):
            assert y == (ord("N") if i in covered else x)
