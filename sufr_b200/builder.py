"""Host-side mirror of the reference's `create` interface, on top of the C ABI.

Same names, argument meaning and error behaviour as the reference:

* :class:`SufrBuilderArgs`  -- libsufr/src/types.rs:527-582
* :class:`SufrBuilder`      -- libsufr/src/sufr_builder.rs:38-220 (``SufrBuilder::<T>::new`` builds AND
  writes the file; the public fields of the struct are attributes here)
* :class:`SuffixArray`      -- ``SuffixArray::write`` u32/u64 dispatch, libsufr/src/suffix_array.rs:460-470
* :class:`SeedMask`         -- libsufr/src/types.rs:36-200
* :func:`read_sequence_file`, :func:`find_lcp_full_offset` -- libsufr/src/util.rs:51-89, :19-37

Everything that computes goes through ``libsufr_b200.so`` (CUDA, sm_100a).  Nothing here touches the
oracle and there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import MEM_DEVICE, MEM_HOST

OUTFILE_VERSION = 6          # types.rs:16
SENTINEL_CHARACTER = b"$"    # types.rs:20


class SufrError(RuntimeError):
    """anyhow::Error of the reference; ``code`` is the C ABI return code."""

    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


def _check(rc: int):
    if rc != _lib.OK:
        raise SufrError(rc, _lib.lib().sufr_b200_last_error().decode(errors="replace"))


# ------------------------------------------------------------------ types.rs:36-200
@dataclass
class SeedMask:
    mask: str
    bytes: List[int]
    positions: List[int]
    differences: List[int]
    weight: int

    @staticmethod
    def new(mask: str) -> "SeedMask":
        n = max(1, len(mask))
        b = (C.c_uint8 * n)()
        p = (C.c_uint64 * n)()
        d = (C.c_uint64 * n)()
        w = _lib.lib().sufr_b200_seed_mask(mask.encode(), b, p, d)
        if w < 0:
            raise SufrError(_lib.ERR_ARGUMENT, f"Invalid seed mask '{mask}'")  # types.rs:82
        return SeedMask(mask, list(b)[:len(mask)], list(p)[:w], list(d)[:w], int(w))

    @staticmethod
    def is_valid(mask: str) -> bool:
        return _lib.lib().sufr_b200_seed_mask(mask.encode(), None, None, None) >= 0

    def __str__(self):
        return self.mask


def find_lcp_full_offset(lcp: int, seed_mask: Optional[str]) -> int:
    """util.rs:19-37"""
    return int(_lib.lib().sufr_b200_find_lcp_full_offset(lcp, seed_mask.encode() if seed_mask else None))


# ------------------------------------------------------------------ types.rs:271-282, util.rs:51-89
@dataclass
class SequenceFileData:
    seq: bytes
    start_positions: List[int]
    sequence_names: List[str]


def read_sequence_file(path, sequence_delimiter: bytes = b"%") -> SequenceFileData:
    s = _lib.Sequences()
    _check(_lib.lib().sufr_b200_read_sequence_file(str(path).encode(), sequence_delimiter[0], C.byref(s)))
    try:
        seq = C.string_at(s.seq, s.seq_len)
        starts = [int(s.start_positions[i]) for i in range(s.num_sequences)]
        names = [s.sequence_names[i].decode() for i in range(s.num_sequences)]
    finally:
        _lib.lib().sufr_b200_sequences_free(C.byref(s))
    return SequenceFileData(seq, starts, names)


# ------------------------------------------------------------------ types.rs:527-582
@dataclass
class SufrBuilderArgs:
    text: bytes
    path: Optional[str] = None
    low_memory: bool = True
    max_query_len: Optional[int] = None
    is_dna: bool = False
    allow_ambiguity: bool = False
    ignore_softmask: bool = False
    sequence_starts: Sequence[int] = (0,)
    sequence_names: Sequence[str] = ("1",)
    num_partitions: int = 16
    seed_mask: Optional[str] = None
    random_seed: int = 42


class _CArgs:
    """Keeps the ctypes buffers behind a SufrB200Args alive."""

    def __init__(self, a: SufrBuilderArgs, *, text_ptr: Optional[int] = None, text_len: Optional[int] = None,
                 rank: int = 0, world_size: int = 1):
        self.c = _lib.Args()
        if text_ptr is None:
            self._text = np.frombuffer(a.text, dtype=np.uint8) if len(a.text) else np.zeros(1, np.uint8)
            self.c.text = self._text.ctypes.data
            self.c.text_len = len(a.text)
        else:
            self.c.text = text_ptr
            self.c.text_len = text_len
        self.c.path = a.path.encode() if a.path is not None else None
        self.c.low_memory = int(a.low_memory)
        self.c.has_max_query_len = int(a.max_query_len is not None)
        self.c.max_query_len = int(a.max_query_len or 0)
        self.c.is_dna = int(a.is_dna)
        self.c.allow_ambiguity = int(a.allow_ambiguity)
        self.c.ignore_softmask = int(a.ignore_softmask)
        self._starts = np.asarray(list(a.sequence_starts), dtype=np.uint64)
        self.c.sequence_starts = self._starts.ctypes.data if len(self._starts) else None
        if len(a.sequence_names) != len(a.sequence_starts):
            # the C ABI carries ONE count for both arrays (make_sufr_frame reads num_sequences entries of each)
            raise SufrError(_lib.ERR_ARGUMENT, f"sequence_names has {len(a.sequence_names)} entries but "
                                               f"sequence_starts has {len(a.sequence_starts)}")
        names = [s.encode() for s in a.sequence_names]
        self._names = (C.c_char_p * max(1, len(names)))(*names)
        self.c.sequence_names = self._names
        self.c.num_sequences = len(self._starts)
        self.c.num_partitions = a.num_partitions
        self.c.seed_mask = a.seed_mask.encode() if a.seed_mask is not None else None
        self.c.random_seed = a.random_seed
        self.c.rank = rank
        self.c.world_size = world_size


class Context:
    """One CUDA stream + device memory pool (SufrB200Ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(_lib.lib().sufr_b200_ctx_create(device, C.byref(self._h)))
        self.device = device

    def reserve(self, text_len: int, index_bits: int = 32):
        _check(_lib.lib().sufr_b200_ctx_reserve(self._h, text_len, index_bits))

    def trim(self):
        _lib.lib().sufr_b200_ctx_trim(self._h)

    def close(self):
        if self._h:
            _lib.lib().sufr_b200_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h


_default_ctx = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class BuildResult:
    """Owner of one SufrB200Result (host or device memory)."""

    def __init__(self, ctx: Context, cargs: _CArgs, res: "_lib.Result"):
        self._ctx, self._cargs, self.c = ctx, cargs, res

    # -- scalars
    @property
    def index_bits(self): return int(self.c.index_bits)
    @property
    def text_len(self): return int(self.c.text_len)
    @property
    def num_suffixes(self): return int(self.c.num_suffixes)
    @property
    def total_suffixes(self): return int(self.c.total_suffixes)
    @property
    def shard_offset(self): return int(self.c.shard_offset)
    @property
    def first_suffix(self): return int(self.c.first_suffix)
    @property
    def last_suffix(self): return int(self.c.last_suffix)
    @property
    def on_device(self): return self.c.memory == MEM_DEVICE
    @property
    def timings(self): return self.c.timings.as_dict()
    @property
    def kernel_launches(self): return int(self.c.kernel_launches)
    @property
    def h2d_bytes(self): return int(self.c.h2d_bytes)
    @property
    def d2h_bytes(self): return int(self.c.d2h_bytes)
    @property
    def n_ranges(self) -> List[Tuple[int, int]]:
        return [(int(self.c.n_ranges[2 * i]), int(self.c.n_ranges[2 * i + 1])) for i in range(self.c.num_n_ranges)]

    def _np(self, ptr, count, dtype):
        if self.on_device:
            raise SufrError(_lib.ERR_ARGUMENT, "result lives in device memory")
        if count == 0:
            return np.zeros(0, dtype)
        ct = {np.uint8: C.c_uint8, np.uint32: C.c_uint32, np.uint64: C.c_uint64}[dtype]
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), (count,))

    @property
    def dtype(self):
        return np.uint32 if self.c.index_bits == 32 else np.uint64

    @property
    def text(self) -> bytes:
        if not self.c.text:
            raise SufrError(_lib.ERR_ARGUMENT, "the transformed text is only returned on rank 0 of a sharded build")
        return self._np(self.c.text, self.text_len, np.uint8).tobytes()

    @property
    def sa(self) -> np.ndarray:
        return self._np(self.c.sa, self.num_suffixes, self.dtype)

    @property
    def lcp(self) -> np.ndarray:
        return self._np(self.c.lcp, self.num_suffixes, self.dtype)

    def _tensor(self, ptr, count, typestr):
        """Zero-copy torch view of a device buffer (valid until free())."""
        import torch

        class _Dev:
            pass
        d = _Dev()
        d.__cuda_array_interface__ = {"shape": (max(count, 0),), "typestr": typestr, "data": (int(ptr), False),
                                      "version": 2}
        if count == 0:
            return torch.zeros(0, dtype=torch.int64, device=f"cuda:{self._ctx.device}")
        return torch.as_tensor(d, device=f"cuda:{self._ctx.device}")

    def sa_tensor(self):
        """Device result: the suffix array as an int32 / int64 torch tensor (same bits as u32 / u64)."""
        return self._tensor(self.c.sa, self.num_suffixes, "<i4" if self.c.index_bits == 32 else "<i8")

    def lcp_tensor(self):
        return self._tensor(self.c.lcp, self.num_suffixes, "<i4" if self.c.index_bits == 32 else "<i8")

    def text_tensor(self):
        return self._tensor(self.c.text, self.text_len, "|u1")

    def device_pointers(self):
        """(text, sa, lcp) raw device addresses of a device result."""
        return int(self.c.text or 0), int(self.c.sa or 0), int(self.c.lcp or 0)

    def set_shard_layout(self, shard_offset: int, total_suffixes: int):
        """Sharded builds: position of this shard in the whole suffix array (from the ranks' counts)."""
        self.c.shard_offset = shard_offset
        self.c.total_suffixes = total_suffixes

    def patch_seam(self, prev_last_suffix: int):
        _check(_lib.lib().sufr_b200_patch_seam(self._ctx.handle, C.byref(self._cargs.c), C.byref(self.c),
                                               prev_last_suffix))

    def verify(self, prev_last_suffix: Optional[int] = None) -> dict:
        """Full on-device check of a DEVICE result (sufr_b200_verify): every SA entry indexed and unique, every
        adjacent pair in order, every LCP value exact.  Returns the report with ``ok`` added; for a sharded
        build ``ok`` covers this shard only (the caller sums num_suffixes against expected_suffixes)."""
        rep = _lib.VerifyReport()
        _check(_lib.lib().sufr_b200_verify(self._ctx.handle, C.byref(self._cargs.c), C.byref(self.c),
                                           int(prev_last_suffix is not None), int(prev_last_suffix or 0), C.byref(rep)))
        d = rep.as_dict()
        errors = d["order_errors"] + d["lcp_errors"] + d["out_of_range"] + d["not_indexed"] + d["duplicates"]
        d["ok"] = errors == 0 and (self._cargs.c.world_size > 1 or d["expected_suffixes"] == self.num_suffixes)
        return d

    def write(self):
        _check(_lib.lib().sufr_b200_write(C.byref(self._cargs.c), C.byref(self.c)))

    def free(self):
        if self.c.owner:
            if not self._ctx.handle:  # context already destroyed (interpreter shutdown): nothing left to return to
                self.c.owner = None
                return
            _lib.lib().sufr_b200_result_free(self._ctx.handle, C.byref(self.c))

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def build(args: SufrBuilderArgs, *, index_bits: int = 0, ctx: Optional[Context] = None, device: int = 0,
          result_memory: int = MEM_HOST, device_text: Optional[Tuple[int, int]] = None,
          rank: int = 0, world_size: int = 1) -> BuildResult:
    """SufrBuilder::new up to (not including) write(): sufr_b200_build.

    ``device_text=(ptr, len)`` passes a text that already lives in device memory.
    """
    ctx = ctx or default_context(device)
    if device_text is not None:
        cargs = _CArgs(args, text_ptr=device_text[0], text_len=device_text[1], rank=rank, world_size=world_size)
        text_memory = MEM_DEVICE
    else:
        cargs = _CArgs(args, rank=rank, world_size=world_size)
        text_memory = MEM_HOST
    res = _lib.Result()
    _check(_lib.lib().sufr_b200_build(ctx.handle, C.byref(cargs.c), index_bits, text_memory, result_memory,
                                      C.byref(res)))
    return BuildResult(ctx, cargs, res)


def file_info(path) -> dict:
    """Header, sequence starts / names and seed mask of a version-6 `.sufr` file, validated (sufr_b200_file_info;
    host only).  Raises SufrError (ERR_IO for a malformed file, ERR_UNSUPPORTED for another version)."""
    fi = _lib.FileInfo()
    _check(_lib.lib().sufr_b200_file_info(str(path).encode(), C.byref(fi)))
    try:
        n = int(fi.num_sequences)
        return {"version": int(fi.version), "index_bits": int(fi.index_bits), "is_dna": bool(fi.is_dna),
                "allow_ambiguity": bool(fi.allow_ambiguity), "ignore_softmask": bool(fi.ignore_softmask),
                "text_len": int(fi.text_len), "num_suffixes": int(fi.num_suffixes),
                "max_query_len": int(fi.max_query_len), "num_sequences": n, "text_pos": int(fi.text_pos),
                "sa_pos": int(fi.sa_pos), "lcp_pos": int(fi.lcp_pos), "file_bytes": int(fi.file_bytes),
                "seed_mask": fi.seed_mask.decode() if fi.seed_mask else None,
                "sequence_starts": [int(fi.sequence_starts[i]) for i in range(n)],
                "sequence_names": [fi.sequence_names[i].decode(errors="replace") for i in range(n)]}
    finally:
        _lib.lib().sufr_b200_file_info_free(C.byref(fi))


@dataclass
class ExtractSequence:
    """One hit of :meth:`SufrIndex.extract` (SufrFile::extract): the region around suffix ``suffix`` (rank ``rank``)
    in the record named ``sequence_name`` that starts at text position ``sequence_start`` (None and 0 outside every
    record).  ``sequence_range`` = (start, end) relative to the record start, ``suffix_offset`` = where the suffix
    starts in ``sequence``, the region's bytes."""
    rank: int
    suffix: int
    sequence_name: Optional[str]
    sequence_start: int
    sequence_range: Tuple[int, int]
    suffix_offset: int
    sequence: bytes


@dataclass
class ExtractResult:
    """The hits of one query of :meth:`SufrIndex.extract`, in rank order (empty when it does not occur)."""
    query_num: int
    query: str
    sequences: List[ExtractSequence]


class KmerSpectrum(NamedTuple):
    """:meth:`SufrIndex.kmer_spectrum`: histogram[i] = distinct k-mers with count i + 1 (the last bin: count >= its
    length)."""
    histogram: np.ndarray
    distinct: int
    occurrences: int
    max_count: int


class SufrIndex:
    """Device-resident index: the read side that consumes the LCP array (``SufrFile::subsample_suffix_array``
    sufr_file.rs:429-456, ``suffix_search`` :777-836, ``locate`` :1132-1169, ``SufrSearch`` sufr_search.rs:104-350).
    ``count`` / ``locate`` take a batch of queries; one GPU thread each.

    ``SufrIndex(result, args)`` borrows the arrays of a DEVICE build result; ``SufrIndex.open(path)`` reads a `.sufr`
    file into device memory the index owns (``.info`` holds its header, names, starts and mask)."""

    HITS_WINDOW = 1 << 24  # hits fetched per sufr_b200_index_hits call: bounds device memory for very frequent queries
    EXTRACT_BYTES = 1 << 28  # default byte budget of one extract / list window (host buffer of that size)

    def __init__(self, result: "BuildResult", args: SufrBuilderArgs):
        self._res, self._args, self._ctx = result, args, result._ctx
        self.info = None
        self._h = C.c_void_p()
        _check(_lib.lib().sufr_b200_index_create(result._ctx.handle, C.byref(result._cargs.c), C.byref(result.c),
                                                 C.byref(self._h)))
        self._set_fields(list(args.sequence_names), [int(x) for x in args.sequence_starts], result.text_len,
                         result.num_suffixes, args.seed_mask, args.max_query_len)

    @classmethod
    def open(cls, path, ctx: Optional[Context] = None, device: int = 0) -> "SufrIndex":
        """SufrFile::read + the in-memory arrays (sufr_file.rs:145-275) on the GPU: sufr_b200_index_open."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        self._res, self._args = None, None
        self._ctx = ctx or default_context(device)
        self.info = file_info(path)
        _check(_lib.lib().sufr_b200_index_open(self._ctx.handle, str(path).encode(), C.byref(self._h)))
        fi = self.info
        self._set_fields(fi["sequence_names"], fi["sequence_starts"], fi["text_len"], fi["num_suffixes"], fi["seed_mask"],
                         fi["max_query_len"])
        return self

    def _set_fields(self, names, starts, text_len, num_suffixes, seed_mask, max_query_len):
        self._sub_mql = None
        self._names, self._starts = names, starts
        self._n, self._s = text_len, num_suffixes
        if seed_mask is not None:
            self._built = SeedMask.new(seed_mask).weight        # sufr_file.rs:528
        else:
            self._built = max_query_len or text_len              # sufr_file.rs:521-527

    def close(self):
        if self._h:
            _lib.lib().sufr_b200_index_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def subsample(self, max_query_len: int) -> int:
        kept = C.c_uint64()
        _check(_lib.lib().sufr_b200_index_subsample(self._h, max_query_len, C.byref(kept)))
        self._sub_mql = max_query_len
        return int(kept.value)

    def _subsample_mql(self, max_query_len, low_memory):
        """set_suffix_array_mem (sufr_file.rs:514-560): the max_query_len of the LCP-subsampled array a search in this
        mode uses, or None when it searches the full array.  sufr_b200_index_locate makes the same choice."""
        if low_memory:
            return None
        eff = min(max_query_len, self._built) if max_query_len else self._built
        return eff if eff != self._built else None

    @staticmethod
    def _pack_queries(queries):
        """A batch of queries as the C ABI takes it: (blob, offsets), query i = blob[offsets[i]:offsets[i + 1]]."""
        qs = [q.encode() if isinstance(q, str) else bytes(q) for q in queries]
        offs = np.zeros(len(qs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(q) for q in qs])
        return np.frombuffer(b"".join(qs) or b"\0", dtype=np.uint8), offs

    def search(self, queries: Sequence[str], max_query_len: Optional[int] = None, low_memory: bool = False):
        """SufrFile::suffix_search: per query the half-open rank range in the full suffix array, or None.
        low_memory=False mirrors set_suffix_array_mem (sufr_file.rs:514-560): when the effective max_query_len is
        shorter than what the index was built with, the LCP-subsampled array is searched."""
        blob, offs = self._pack_queries(queries)
        nq = len(offs) - 1
        eff = self._subsample_mql(max_query_len, low_memory)
        if eff is not None and self._sub_mql != eff:
            self.subsample(eff)
        use_sub = int(eff is not None)
        b = np.zeros(max(1, nq), dtype=np.uint64)
        e = np.zeros(max(1, nq), dtype=np.uint64)
        _check(_lib.lib().sufr_b200_index_search(self._h, blob.ctypes.data, offs.ctypes.data, nq,
                                                 int(max_query_len is not None), int(max_query_len or 0), use_sub,
                                                 b.ctypes.data, e.ctypes.data))
        none = np.uint64(0xFFFFFFFFFFFFFFFF)
        return [None if b[i] == none else (int(b[i]), int(e[i])) for i in range(nq)]

    def count(self, queries, max_query_len=None, low_memory=False) -> List[int]:
        return [0 if r is None else r[1] - r[0] for r in self.search(queries, max_query_len, low_memory)]

    def suffixes(self, rank_begin: int, count: int) -> np.ndarray:
        out = np.zeros(max(1, count), dtype=np.uint64)
        _check(_lib.lib().sufr_b200_index_suffixes(self._h, rank_begin, count, out.ctypes.data))
        return out[:count]

    def locate_ranges(self, queries, max_query_len=None, low_memory=False):
        """sufr_b200_index_locate: (rank_begin, rank_end, hit_offsets) as numpy arrays; hits of query i are
        hit_offsets[i] .. hit_offsets[i + 1] in :meth:`hits`.  Absent queries have rank_begin == rank_end == 2**64-1.
        low_memory=False searches the LCP-subsampled array when the effective max_query_len is shorter than the
        build's (sufr_file.rs:514-560), as :meth:`search` does."""
        blob, offs = self._pack_queries(queries)
        nq = len(offs) - 1
        b = np.zeros(max(1, nq), dtype=np.uint64)
        e = np.zeros(max(1, nq), dtype=np.uint64)
        ho = np.zeros(nq + 1, dtype=np.uint64)
        # the library replaces the index's subsample when this mode needs another one: keep the cache of search() true
        eff = self._subsample_mql(max_query_len, low_memory)
        if eff is not None:
            self._sub_mql = None
        _check(_lib.lib().sufr_b200_index_locate(self._h, blob.ctypes.data, offs.ctypes.data, nq,
                                                 int(max_query_len is not None), int(max_query_len or 0),
                                                 int(low_memory), b.ctypes.data, e.ctypes.data, ho.ctypes.data))
        if eff is not None:
            self._sub_mql = eff
        return b[:nq], e[:nq], ho

    def hits(self, first: int, count: int):
        """sufr_b200_index_hits: (suffix, sequence, sequence_pos) of hits [first, first + count) of the last locate,
        :meth:`mems` or :meth:`approx_matches`."""
        suf = np.zeros(max(1, count), dtype=np.uint64)
        seq = np.zeros(max(1, count), dtype=np.uint64)
        pos = np.zeros(max(1, count), dtype=np.uint64)
        _check(_lib.lib().sufr_b200_index_hits(self._h, first, count, suf.ctypes.data, seq.ctypes.data,
                                               pos.ctypes.data))
        return suf[:count], seq[:count], pos[:count]

    def locate(self, queries, max_query_len=None, low_memory=False):
        """SufrFile::locate: per query a list of (rank, suffix, sequence_name, sequence_position) in rank order
        (name None and position = suffix for an index without sequence starts)."""
        b, _, ho = self.locate_ranges(queries, max_query_len, low_memory)
        hits = self._split(self._all_hits(int(ho[-1])), ho)
        return [[(r0 + k,) + h for k, h in enumerate(hs)] for r0, hs in zip(b.tolist(), hits)]

    def _all_hits(self, total: int):
        """The rows (suffix, sequence name or None, sequence position) of all ``total`` hits of the last locate, mems
        or approx, fetched in windows."""
        parts = [self.hits(f, min(self.HITS_WINDOW, total - f)) for f in range(0, total, self.HITS_WINDOW)]
        if not parts:
            return []
        suf, seq, pos = (np.concatenate([p[k] for p in parts]).tolist() for k in range(3))
        names, none = self._names, 0xFFFFFFFFFFFFFFFF
        return [(s, None if q == none else names[q], p) for s, q, p in zip(suf, seq, pos)]

    @staticmethod
    def _split(rows, offsets):
        """``rows`` cut into one list per entry of an offsets array: entry i gets rows[offsets[i]:offsets[i + 1]]."""
        cuts = np.asarray(offsets).astype(np.int64).tolist()
        return [rows[lo:hi] for lo, hi in zip(cuts[:-1], cuts[1:])]

    def matching_statistics(self, queries):
        """sufr_b200_index_matching_stats: per query (lengths, rank_begin, rank_end), numpy uint64 arrays of the
        query's length.  lengths[i] = the longest l (at most the build's max_query_len) such that query[i:i+l] starts
        an indexed suffix; [rank_begin[i], rank_end[i]) = the ranks of those suffixes (2**64-1 both when l = 0).  See
        include/sufr_b200.h for the definitions; an index with a seed mask is refused (ERR_UNSUPPORTED)."""
        blob, offs = self._pack_queries(queries)
        nq, total = len(offs) - 1, int(offs[-1])
        ms, b, e = (np.zeros(max(1, total), dtype=np.uint64) for _ in range(3))
        _check(_lib.lib().sufr_b200_index_matching_stats(self._h, blob.ctypes.data, offs.ctypes.data, nq, ms.ctypes.data,
                                                         b.ctypes.data, e.ctypes.data))
        return list(zip(*(self._split(x, offs) for x in (ms, b, e))))

    def _mems(self, queries, min_len):
        """sufr_b200_index_mems: (query, position, length, rank_begin, rank_end, hit_offsets) as numpy arrays, one entry
        per MEM (hit_offsets one longer).  The MEMs become the hits of :meth:`hits` / :meth:`extract_window`."""
        if min_len < 1:
            raise SufrError(_lib.ERR_ARGUMENT, f"min_len must be at least 1 (got {min_len})")
        blob, offs = self._pack_queries(queries)
        nq, total = len(offs) - 1, int(offs[-1])
        cols = [np.zeros(max(1, total), dtype=np.uint64) for _ in range(5)]
        ho = np.zeros(total + 1, dtype=np.uint64)
        num = C.c_uint64()
        _check(_lib.lib().sufr_b200_index_mems(self._h, blob.ctypes.data, offs.ctypes.data, nq, min_len, C.byref(num),
                                               *[c.ctypes.data for c in cols], ho.ctypes.data))
        k = int(num.value)
        return tuple(c[:k] for c in cols) + (ho[:k + 1],)

    def mems(self, queries, min_len: int):
        """Maximal exact matches of at least ``min_len`` bytes (include/sufr_b200.h): per query a list of
        (query_pos, length, rank_begin, rank_end) in position order.  Afterwards :meth:`hits` and
        :meth:`extract_window` work on these MEMs (in query order, then position order) as on a locate's queries."""
        q, p, ln, b, e, _ = self._mems(queries, min_len)
        out = [[] for _ in range(len(queries))]
        for row in zip(q.tolist(), p.tolist(), ln.tolist(), b.tolist(), e.tolist()):
            out[row[0]].append(row[1:])
        return out

    def locate_mems(self, queries, min_len: int):
        """:meth:`mems` with every occurrence: per query a list of (query_pos, length, hits) with hits a list of
        (suffix, sequence_name, sequence_position) in rank order, as :meth:`locate` gives them."""
        q, p, ln, _, _, ho = self._mems(queries, min_len)
        hits = self._split(self._all_hits(int(ho[-1])), ho)
        out = [[] for _ in range(len(queries))]
        for qi, qp, ml, hs in zip(q.tolist(), p.tolist(), ln.tolist(), hits):
            out[qi].append((qp, ml, hs))
        return out

    APPROX_WINDOW = 1 << 24  # matches fetched per sufr_b200_index_approx_matches call

    def _approx(self, queries, max_mismatches):
        """sufr_b200_index_approx, then every match in windows: (mismatches, rank_begin, rank_end, hit_offsets,
        match_offsets) as numpy arrays (hit_offsets one longer than the matches, match_offsets one longer than the
        queries).  The matches become the hits of :meth:`hits` / :meth:`extract_window`."""
        _non_negative(max_mismatches=max_mismatches)
        blob, offs = self._pack_queries(queries)
        nq = len(offs) - 1
        mo = np.zeros(nq + 1, dtype=np.uint64)
        hits = C.c_uint64()
        L = _lib.lib()
        _check(L.sufr_b200_index_approx(self._h, blob.ctypes.data, offs.ctypes.data, nq, max_mismatches, mo.ctypes.data,
                                        C.byref(hits)))
        total = int(mo[-1])
        cols = [np.zeros(max(1, total), dtype=np.uint64) for _ in range(3)]
        ho = np.zeros(total + 1, dtype=np.uint64)
        for f in range(0, total, self.APPROX_WINDOW):
            c = min(self.APPROX_WINDOW, total - f)
            _check(L.sufr_b200_index_approx_matches(self._h, f, c, *[x[f:].ctypes.data for x in cols],
                                                    ho[f:].ctypes.data))
        return tuple(x[:total] for x in cols) + (ho, mo)

    def approx_matches(self, queries, max_mismatches: int):
        """Search with mismatches (include/sufr_b200.h): per query a list of (mismatches, rank_begin, rank_end) in
        rank order, one per distinct string w of the query's length (capped at the build's max_query_len) that occurs
        in the text within ``max_mismatches`` substitutions of the query, no substitution onto a record separator.
        An index with a seed mask is refused (ERR_UNSUPPORTED)."""
        mis, b, e, _, mo = self._approx(queries, max_mismatches)
        return self._split(list(zip(mis.tolist(), b.tolist(), e.tolist())), mo)

    def locate_approx(self, queries, max_mismatches: int):
        """:meth:`approx_matches` with every occurrence: per query a list of (mismatches, hits) with hits a list of
        (suffix, sequence_name, sequence_position) in rank order, as :meth:`locate_mems` gives them."""
        mis, _, _, ho, mo = self._approx(queries, max_mismatches)
        hits = self._split(self._all_hits(int(ho[-1])), ho)
        return self._split(list(zip(mis.tolist(), hits)), mo)

    def approx_levels(self):
        """The profile of the last search with mismatches: (nodes, steps), numpy arrays indexed by depth."""
        num = C.c_uint64()
        L = _lib.lib()
        _check(L.sufr_b200_index_approx_levels(self._h, 0, C.byref(num), None, None))
        nodes = np.zeros(max(1, num.value), dtype=np.uint64)
        steps = np.zeros(max(1, num.value), dtype=np.uint64)
        _check(L.sufr_b200_index_approx_levels(self._h, num.value, C.byref(num), nodes.ctypes.data, steps.ctypes.data))
        return nodes[:num.value], steps[:num.value]

    def kmer_spectrum(self, k: int, num_bins: int = 10000) -> "KmerSpectrum":
        """sufr_b200_index_kmer_spectrum: histogram[i] = distinct k-mers occurring i + 1 times (the last bin: at least
        num_bins times), with the number of distinct k-mers, of occurrences and the largest count.  A k-mer lies inside
        one record and never includes its last byte; in a DNA index it is made of ACGT only (include/sufr_b200.h)."""
        _positive_k(k)
        _non_negative(num_bins=num_bins)
        hist = np.zeros(max(1, num_bins), dtype=np.uint64)
        d, o, m = C.c_uint64(), C.c_uint64(), C.c_uint64()
        _check(_lib.lib().sufr_b200_index_kmer_spectrum(self._h, k, num_bins, hist.ctypes.data, C.byref(d), C.byref(o),
                                                        C.byref(m)))
        return KmerSpectrum(hist[:num_bins], int(d.value), int(o.value), int(m.value))

    def kmers(self, k: int, min_count: int = 1, max_count: Optional[int] = None, window: int = 1 << 24):
        """sufr_b200_index_kmers over the whole index: the distinct k-mers whose count lies in [min_count, max_count]
        in byte order, as (rank_begin, rank_end, count, kmers) with kmers a (m, k) uint8 array; [rank_begin,
        rank_end) is the k-mer's rank range, as :meth:`search` gives it.  Fetched ``window`` k-mers at a time (fewer
        when their bytes would pass EXTRACT_BYTES)."""
        _positive_k(k)
        _non_negative(min_count=min_count, max_count=max_count, window=window)
        if window < 1:
            raise SufrError(_lib.ERR_ARGUMENT, f"window must be at least 1 (got {window})")
        per = max(1, min(window, self.EXTRACT_BYTES // k))
        hi = _U64_MAX if max_count is None else max_count
        cols = [np.zeros(per, dtype=np.uint64) for _ in range(3)]
        buf = np.zeros(per * k, dtype=np.uint8)
        parts, first = [], 0
        num, nxt = C.c_uint64(), C.c_uint64()
        while True:
            _check(_lib.lib().sufr_b200_index_kmers(self._h, k, min_count, hi, first, per, C.byref(num), C.byref(nxt),
                                                    *[c.ctypes.data for c in cols], buf.ctypes.data))
            m = int(num.value)
            parts.append([c[:m].copy() for c in cols] + [buf[:m * k].reshape(m, k).copy()])
            first = int(nxt.value)
            if first >= self._s:
                break
        return tuple(np.concatenate([p[j] for p in parts]) for j in range(3)) + (
            np.concatenate([p[3] for p in parts]).reshape(-1, k),)

    def kmer_multiplicity(self, k: int, start: int = 0, length: Optional[int] = None, window: int = 1 << 28):
        """sufr_b200_index_kmer_multiplicity: out[i] = the count of the k-mer at text position start + i, 0 where no
        k-mer starts (saturated at 2**32 - 1), as a numpy uint32 array; ``length`` defaults to the end of the text.
        Each window of ``window`` positions is one pass over the ranks."""
        _positive_k(k)
        _non_negative(start=start, length=length, window=window)
        if window < 1:
            raise SufrError(_lib.ERR_ARGUMENT, f"window must be at least 1 (got {window})")
        if length is None:
            length = max(0, self._n - start)
        out = np.zeros(max(1, length), dtype=np.uint32)
        if length == 0:
            _check(_lib.lib().sufr_b200_index_kmer_multiplicity(self._h, k, start, 0, out.ctypes.data))
        for f in range(0, length, window):
            m = min(window, length - f)
            _check(_lib.lib().sufr_b200_index_kmer_multiplicity(self._h, k, start + f, m, out[f:].ctypes.data))
        return out[:length]

    def extract_window(self, first: int, max_hits: int, prefix_len: Optional[int] = None,
                       suffix_len: Optional[int] = None, max_bytes: Optional[int] = None):
        """sufr_b200_index_extract: the regions of the longest leading run of hits [first, first + max_hits) of the
        last locate or :meth:`mems` whose bytes fit in ``max_bytes``.  Returns ((suffix, sequence, region_start, region_end,
        byte_offsets), bytes) with numpy arrays of the run's length (byte_offsets one longer; sequence 2**64-1 outside
        every record).  A first region larger than the budget gets one retry with a buffer of its size."""
        max_bytes = self.EXTRACT_BYTES if max_bytes is None else max_bytes
        _non_negative(first=first, max_hits=max_hits, prefix_len=prefix_len, suffix_len=suffix_len, max_bytes=max_bytes)
        outs = [np.zeros(max(1, max_hits), dtype=np.uint64) for _ in range(4)]
        offs = np.zeros(max_hits + 1, dtype=np.uint64)
        P = 0 if prefix_len is None else prefix_len
        S = _U64_MAX if suffix_len is None else suffix_len
        k, buf = self._fetch_window(_lib.lib().sufr_b200_index_extract, first, max_hits, (P, S), max_bytes, outs, offs)
        return tuple(o[:k] for o in outs) + (offs[:k + 1],), buf[:int(offs[k])].tobytes()

    def _fetch_window(self, fn, first, m, params, max_bytes, outs, offs):
        """sufr_b200_index_extract / _list over entries [first, first + m) into ``outs`` and ``offs`` with a buffer of
        ``max_bytes``: (entries, buffer).  A first entry larger than that gets one retry with a buffer of its size."""
        num, budget = C.c_uint64(), max_bytes
        while True:
            buf = np.empty(max(1, budget), dtype=np.uint8)
            _check(fn(self._h, first, m, *params, budget, C.byref(num), *[o.ctypes.data for o in outs],
                      offs.ctypes.data, buf.ctypes.data))
            k = int(num.value)
            if k or m == 0 or int(offs[1]) <= budget:
                return k, buf
            budget = int(offs[1])

    def extract(self, queries, prefix_len: Optional[int] = None, suffix_len: Optional[int] = None,
                max_query_len: Optional[int] = None, low_memory: bool = False) -> List[ExtractResult]:
        """SufrFile::extract: per query the text around each hit, in rank order.  ``prefix_len`` bytes before the
        suffix (default 0) and ``suffix_len`` from it (default: to the end of its record), clipped to the record;
        see include/sufr_b200.h for the rule."""
        b, _, ho = self.locate_ranges(queries, max_query_len, low_memory)
        total = int(ho[-1])
        parts, first = [], 0
        while first < total:
            arrs, data = self.extract_window(first, min(self.HITS_WINDOW, total - first), prefix_len, suffix_len)
            parts.append((arrs, data))
            first += len(arrs[0])
        names, starts, none = self._names, self._starts, 0xFFFFFFFFFFFFFFFF
        flat = []
        for (suf, seq, rs, re_, offs), data in parts:
            suf, seq, rs, re_, offs = suf.tolist(), seq.tolist(), rs.tolist(), re_.tolist(), offs.tolist()
            for k in range(len(suf)):
                a = 0 if seq[k] == none else starts[seq[k]]
                flat.append(ExtractSequence(0, suf[k], None if seq[k] == none else names[seq[k]], a, (rs[k], re_[k]),
                                            suf[k] - a - rs[k], data[offs[k]:offs[k + 1]]))
        out = []
        for i, q in enumerate(queries):
            lo, hi, r0 = int(ho[i]), int(ho[i + 1]), int(b[i])
            seqs = flat[lo:hi]
            for k, e in enumerate(seqs):
                e.rank = r0 + k
            out.append(ExtractResult(i, q if isinstance(q, str) else bytes(q).decode("latin-1"), seqs))
        return out

    def list(self, first_rank: int = 0, count: Optional[int] = None, len: Optional[int] = None,
             rows_window: int = 1 << 24, max_bytes: Optional[int] = None):
        """SufrFile::list over ranks [first_rank, first_rank + count) (default: to the last rank): (suffix, lcp,
        byte_offsets, bytes) with bytes[byte_offsets[i]:byte_offsets[i + 1]] = the first ``len`` bytes of suffix i
        (default: the whole suffix).  Fetched in windows of ``rows_window`` rows and ``max_bytes`` bytes."""
        _non_negative(first_rank=first_rank, count=count, len=len, max_bytes=max_bytes)
        if count is None:
            count = max(0, self._s - first_rank)
        max_bytes = self.EXTRACT_BYTES if max_bytes is None else max_bytes
        L = _U64_MAX if len is None else len
        sufs, lcps, offs, datas = [], [], [np.zeros(1, np.uint64)], []
        base, r, end = 0, first_rank, first_rank + count
        while True:
            m = min(rows_window, end - r)
            suf, lcp = np.zeros(max(1, m), np.uint64), np.zeros(max(1, m), np.uint64)
            o = np.zeros(m + 1, np.uint64)
            k, buf = self._fetch_window(_lib.lib().sufr_b200_index_list, r, m, (L,), max_bytes, (suf, lcp), o)
            if m == 0:
                break
            sufs.append(suf[:k])
            lcps.append(lcp[:k])
            offs.append(o[1:k + 1] + np.uint64(base))
            datas.append(buf[:int(o[k])].tobytes())
            base += int(o[k])
            r += k
            if r >= end:
                break
        cat = (lambda xs: np.concatenate(xs) if xs else np.zeros(0, np.uint64))
        return cat(sufs), cat(lcps), np.concatenate(offs), b"".join(datas)

    def string_at(self, pos: int, len: Optional[int] = None) -> bytes:
        """SuffixArray::string_at: text[pos : pos + len] (default: to the end of the text); pos > text length raises."""
        _non_negative(pos=pos, len=len)
        want = max(0, self._n - pos) if len is None else min(len, max(0, self._n - pos))
        out = np.empty(max(1, want), np.uint8)
        got = C.c_uint64()
        _check(_lib.lib().sufr_b200_index_string_at(self._h, pos, _U64_MAX if len is None else len, out.ctypes.data,
                                                    C.byref(got)))
        return out[:int(got.value)].tobytes()


_U64_MAX = 0xFFFFFFFFFFFFFFFF


def _positive_k(k):
    if k < 1:
        raise SufrError(_lib.ERR_ARGUMENT, f"k must be at least 1 (got {k})")


def _non_negative(**values):
    """Positions, counts and lengths travel as u64: a negative one would wrap to a huge value instead of failing."""
    for name, v in values.items():
        if v is not None and v < 0:
            raise SufrError(_lib.ERR_ARGUMENT, f"{name} must not be negative (got {v})")


def create_multi(args: SufrBuilderArgs, devices: Sequence[int], index_bits: int = 0) -> dict:
    """``sufr::create`` on several GPUs of one box in one call (sufr_b200_create_multi): builds and writes
    ``args.path``; returns the counts and timings of the whole build."""
    cargs = _CArgs(args)
    res = _lib.Result()
    devs = (C.c_int * len(devices))(*[int(d) for d in devices])
    _check(_lib.lib().sufr_b200_create_multi(C.byref(cargs.c), devs, len(devices), index_bits, C.byref(res)))
    try:
        return {"num_suffixes": int(res.num_suffixes), "text_len": int(res.text_len), "index_bits": int(res.index_bits),
                "timings": res.timings.as_dict(), "kernel_launches": int(res.kernel_launches),
                # (ctypes.string_at takes a C int: texts of 2 GiB and more go through numpy)
                "text": np.ctypeslib.as_array(C.cast(res.text, C.POINTER(C.c_uint8)), (int(res.text_len),)).tobytes()
                if res.text and res.text_len else b"",
                "n_ranges": [(int(res.n_ranges[2 * i]), int(res.n_ranges[2 * i + 1])) for i in range(res.num_n_ranges)]}
    finally:
        _lib.lib().sufr_b200_result_free(None, C.byref(res))


class SufrBuilder:
    """``SufrBuilder::<T>::new(args)``: builds the suffix and LCP arrays on the GPU and writes the
    `.sufr` file at ``args.path`` (default "out.sufr", sufr_builder.rs:215).  ``index_bits`` plays the
    role of the type parameter T (32 -> u32, 64 -> u64)."""

    def __init__(self, args: SufrBuilderArgs, index_bits: int = 32, *, ctx: Optional[Context] = None,
                 device: int = 0, write: bool = True):
        if index_bits not in (32, 64):
            raise SufrError(_lib.ERR_ARGUMENT, "index_bits must be 32 or 64")
        self._res = build(args, index_bits=index_bits, ctx=ctx, device=device)
        r = self._res
        self.version = OUTFILE_VERSION
        self.is_dna = args.is_dna
        self.allow_ambiguity = args.allow_ambiguity
        self.ignore_softmask = args.ignore_softmask
        self.text_len = r.text_len
        self.num_suffixes = r.num_suffixes
        self.num_sequences = len(args.sequence_starts)
        self.sequence_starts = list(args.sequence_starts)
        self.sequence_names = list(args.sequence_names)
        self.text = r.text
        self.sort_type = ("Mask", SeedMask.new(args.seed_mask)) if args.seed_mask is not None else \
            ("MaxQueryLen", args.max_query_len or 0)
        self.n_ranges = r.n_ranges
        self.path = args.path if args.path is not None else "out.sufr"
        self.index_bits = index_bits
        # not part of the reference struct (its arrays live in temp files): kept for library users
        self.suffix_array = r.sa
        self.lcp_array = r.lcp
        self.timings = r.timings
        if write:
            r.write()


class SuffixArray:
    """The write half of libsufr::suffix_array::SuffixArray."""

    @staticmethod
    def write(args: SufrBuilderArgs, **kw) -> str:
        # suffix_array.rs:460-470: u32 iff text.len() < u32::MAX
        bits = 32 if len(args.text) < 0xFFFFFFFF else 64
        return SufrBuilder(args, bits, **kw).path
