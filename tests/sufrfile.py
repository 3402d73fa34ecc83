"""Minimal parser of the version-6 `.sufr` byte layout (reference: sufr_builder.rs:817-918,
read side sufr_file.rs:145-275).  Test helper only."""
from __future__ import annotations

import struct
from dataclasses import dataclass
from typing import List, Optional

import numpy as np


@dataclass
class SufrFile:
    version: int
    is_dna: bool
    allow_ambiguity: bool
    ignore_softmask: bool
    text_len: int
    text_pos: int
    sa_pos: int
    lcp_pos: int
    num_suffixes: int
    max_query_len: int
    num_sequences: int
    sequence_starts: List[int]
    seed_mask: Optional[str]
    text: bytes
    sa: np.ndarray
    lcp: np.ndarray
    sequence_names: List[str]
    index_bits: int


def parse_sufr(data: bytes) -> SufrFile:
    version, is_dna, amb, soft = data[0], data[1], data[2], data[3]
    text_len, text_pos, sa_pos, lcp_pos, num_suffixes, mql, nseq = struct.unpack_from("<7Q", data, 4)
    # the element width from the section sizes, so u64 files of short texts (--index-bits 64) read right; the text
    # length rule of suffix_array.rs:390-402 only for an empty array
    bits = 8 * (lcp_pos - sa_pos) // num_suffixes if num_suffixes else (32 if text_len < 0xFFFFFFFF else 64)
    w = bits // 8
    dt = np.dtype("<u4") if bits == 32 else np.dtype("<u8")
    off = 60
    starts = np.frombuffer(data, dt, nseq, off).astype(np.uint64).tolist()
    off += nseq * w
    (mask_len,) = struct.unpack_from("<Q", data, off)
    off += 8
    mask = None
    if mask_len:
        mask = "".join("1" if b == 1 else "0" for b in data[off:off + mask_len])
        off += mask_len
    assert off == text_pos, (off, text_pos)
    text = data[text_pos:text_pos + text_len]
    assert sa_pos == text_pos + text_len
    sa = np.frombuffer(data, dt, num_suffixes, sa_pos).copy()
    assert lcp_pos == sa_pos + num_suffixes * w
    lcp = np.frombuffer(data, dt, num_suffixes, lcp_pos).copy()
    off = lcp_pos + num_suffixes * w
    (cnt,) = struct.unpack_from("<Q", data, off)
    off += 8
    names = []
    for _ in range(cnt):
        (ln,) = struct.unpack_from("<Q", data, off)
        off += 8
        names.append(data[off:off + ln].decode())
        off += ln
    assert off == len(data), (off, len(data))
    return SufrFile(version, bool(is_dna), bool(amb), bool(soft), text_len, text_pos, sa_pos, lcp_pos,
                    num_suffixes, mql, nseq, [int(s) for s in starts], mask, text, sa, lcp, names, bits)


def parse_header(data: bytes) -> dict:
    """The fixed part of the header (sufr_builder.rs:826-867): enough to locate the sections of a large file."""
    text_len, text_pos, sa_pos, lcp_pos, num_suffixes, mql, nseq = struct.unpack_from("<7Q", data, 4)
    return {"version": data[0], "is_dna": bool(data[1]), "allow_ambiguity": bool(data[2]), "ignore_softmask": bool(data[3]),
            "text_len": text_len, "text_pos": text_pos, "sa_pos": sa_pos, "lcp_pos": lcp_pos, "num_suffixes": num_suffixes,
            "max_query_len": mql, "num_sequences": nseq, "index_bytes": (lcp_pos - sa_pos) // max(1, num_suffixes)}
