"""Texts for the read-side tests, and one text built as every index source a spec lists (device builds indexed in
place, written and reopened `.sufr` files; u32 and u64), checked to hold the same text, suffix array and LCP array."""
import random

import numpy as np

from sufrfile import parse_sufr

ACGT, PROTEIN = b"ACGT", b"ACDEFGHIKLMNPQRSTVWY"
WIDE = bytes(range(1, 97)) + bytes(range(123, 256))  # (lowercase bytes would be uppercased by the build)
ALL = [("built", 32), ("built", 64), ("file", 32), ("file", 64)]


def make_text(seed, n, alphabet, *, copies=0, copy_len=(10, 100), runs=(), rare=b"", rare_p=0.0, dollar=True):
    """n random bytes of `alphabet`, with `copies` segments copied from elsewhere in the text (repeats, long LCPs),
    tandem runs of the given units, and bytes of `rare` sprinkled at rate rare_p."""
    rng = np.random.default_rng(seed)
    t = np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)]
    for _ in range(copies):
        ln = int(rng.integers(copy_len[0], copy_len[1] + 1))
        if ln >= n:
            continue
        src, dst = (int(x) for x in rng.integers(0, n - ln, 2))
        t[dst:dst + ln] = t[src:src + ln].copy()
    for unit, count in runs:
        u = np.frombuffer(unit, np.uint8)
        ln = min(n, len(u) * count)
        dst = int(rng.integers(0, n - ln + 1))
        t[dst:dst + ln] = np.tile(u, count)[:ln]
    if rare:
        hit = np.flatnonzero(rng.random(n) < rare_p)
        t[hit] = np.frombuffer(rare, np.uint8)[rng.integers(0, len(rare), len(hit))]
    return t.tobytes() + (b"$" if dollar else b"")


def with_records(text, k, seed):
    """`text` with k - 1 of its bytes replaced by the delimiter '%': (text, sequence starts, names)."""
    n = len(text)
    if k <= 1 or n < 4 * k:
        return text, [0], ["r0"]
    rng = random.Random(seed)
    cut = sorted(rng.sample(range(1, n - 2), k - 1))
    t = bytearray(text)
    for c in cut:
        t[c] = ord("%")
    return bytes(t), [0] + [c + 1 for c in cut], [f"r{i}" for i in range(k)]


def builder_args(S, text, starts, names, **flags):
    """SufrBuilderArgs with the given records, or with the builder's default record when starts is None."""
    records = {} if starts is None else dict(sequence_starts=starts, sequence_names=names)
    return S.SufrBuilderArgs(text=text, **records, **flags)


def device_index(S, text, starts, names, index_bits=32, **flags):
    """`text` built on the device and indexed in place: (SufrIndex, the build result it borrows from)."""
    import torch
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = builder_args(S, b"", starts, names, **flags)
    r = S.build(args, index_bits=index_bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    r._keep = t
    return S.SufrIndex(r, args), r


class IndexMatrix:
    """One text built as every source of `sources`, a list of (kind, bits) with kind "built" (device_index) or "file"
    (written to `tmp` and opened).  indexes = [(label, SufrIndex)]; arrays = (text, SA, LCP) as the sources hold them
    (SA and LCP as int64), asserted equal across the sources."""

    def __init__(self, S, name, text, starts, names, flags, sources, tmp):
        self.name, self.flags, self.starts, self.names = name, flags, starts, names
        self.indexes, self._results, arrays = [], [], None
        try:
            for kind, bits in sources:
                if kind == "built":
                    index, r = device_index(S, text, starts, names, bits, **flags)
                    self._results.append(r)
                    udt = np.uint32 if bits == 32 else np.uint64  # (the tensors hold the same bits as signed)
                    got = (r.text_tensor().cpu().numpy().tobytes(), r.sa_tensor().cpu().numpy().view(udt),
                           r.lcp_tensor().cpu().numpy().view(udt))
                else:
                    path = tmp / f"{name}_u{bits}.sufr"
                    S.SufrBuilder(builder_args(S, text, starts, names, path=str(path), **flags), bits)._res.free()
                    f = parse_sufr(path.read_bytes())
                    assert f.index_bits == bits
                    got = (f.text, f.sa, f.lcp)
                    index = S.SufrIndex.open(path)
                self.indexes.append((f"{kind}_u{bits}", index))
                got = (got[0], got[1].astype(np.int64), got[2].astype(np.int64))
                if arrays is None:
                    arrays = got
                else:  # every source holds the same index
                    assert got[0] == arrays[0] and np.array_equal(got[1], arrays[1]) and np.array_equal(got[2], arrays[2])
        except BaseException:
            self.close()
            raise
        self.arrays = arrays

    def close(self):
        for _, index in self.indexes:
            index.close()
        for r in self._results:
            r.free()
        self.indexes, self._results = [], []
