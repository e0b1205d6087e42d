"""Read / reference ingest: FASTA and FASTQ files -> byte buffers the device packers take (SURVEY 8f N2).

The reference reads one sequence per file with a Python line loop (SMEM/ExactMatch.py:43-50 for the reference,
:104-108 for a query).  Here a file is mapped once, line ends are found with one vectorised scan, and the sequence
lines are gathered into one contiguous uint8 buffer plus offsets -- exactly what gsm_pack_reads_device /
gsm_text_pack_device (GPU 2-bit packing) and PipelinedEngine.run_ascii consume.  Parsing is host-side numpy; nothing
here computes a search result.

N-base policy (the reference raises KeyError on any character outside ACGT, ExactMatch.py:139):
  "error"  keep every read; the device packer reports the first offending read (BaseError)      [default]
  "drop"   remove reads that hold a character outside ACGT; their indices are returned
"""
import numpy as np

_VALID = np.zeros(256, bool)
_VALID[[65, 67, 71, 84]] = True          # A C G T


def _lines(buf):
    """(start, end) of every line of a uint8 buffer, '\n' / '\r\n' stripped, trailing empty line dropped."""
    nl = np.flatnonzero(buf == 10)
    starts = np.concatenate(([0], nl + 1))
    ends = np.concatenate((nl, [len(buf)]))
    if len(starts) and starts[-1] >= len(buf):
        starts, ends = starts[:-1], ends[:-1]
    cr = (ends > starts) & (buf[np.maximum(ends - 1, 0)] == 13)
    return starts, ends - cr


def _gather(buf, starts, ends, pin):
    """Concatenate buf[starts[i]:ends[i]] -> (flat uint8, offsets int64[n+1])."""
    lens = (ends - starts).astype(np.int64)
    off = np.concatenate(([0], np.cumsum(lens)))
    total = int(off[-1])
    if pin:
        import torch
        out_t = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
        out = out_t.numpy()[:total]
    else:
        out = np.empty(total, np.uint8)
    # index of every output byte in the source = start of its read + position inside it; in blocks of reads so that the
    # index array stays small next to a multi-GB file
    block = 1 << 18
    for a in range(0, len(starts), block):
        b = min(len(starts), a + block)
        o0, o1 = int(off[a]), int(off[b])
        if o1 > o0:
            idx = np.repeat(starts[a:b] - off[a:b], lens[a:b]) + np.arange(o0, o1, dtype=np.int64)
            np.take(buf, idx, out=out[o0:o1])
    return out, off


def read_fasta(path):
    """-> (names, sequences as uint8 arrays).  Multi-record, multi-line FASTA; the reference's files hold one record."""
    buf = np.fromfile(path, dtype=np.uint8)
    starts, ends = _lines(buf)
    keep = ends > starts
    starts, ends = starts[keep], ends[keep]
    is_hdr = buf[starts] == ord(">")
    hdr_idx = np.flatnonzero(is_hdr)
    names, seqs = [], []
    for k, h in enumerate(hdr_idx):
        nxt = hdr_idx[k + 1] if k + 1 < len(hdr_idx) else len(starts)
        names.append(bytes(buf[starts[h] + 1:ends[h]]).decode(errors="replace"))
        seq, _ = _gather(buf, starts[h + 1:nxt], ends[h + 1:nxt], pin=False)
        seqs.append(seq)
    if not len(hdr_idx) and len(starts):          # headerless: one sequence
        seq, _ = _gather(buf, starts, ends, pin=False)
        names.append("")
        seqs.append(seq)
    return names, seqs


class Contigs:
    """Sequence table of a reference built from several sequences laid end to end (as BWA concatenates them):
    names[i], start[i] = first base of sequence i in the concatenated text (uint32, n + 1 entries, start[n] = n_bases;
    empty sequences allowed) and lengths[i] = start[i + 1] - start[i]."""

    def __init__(self, names, start):
        s = np.asarray(start, np.int64).reshape(-1)
        names = [str(x) for x in names]
        if len(names) < 1 or len(s) != len(names) + 1:
            raise ValueError("Contigs: need at least one sequence and one more start entry than names")
        if s[0] != 0 or (np.diff(s) < 0).any() or s[-1] >= 1 << 32:
            raise ValueError("Contigs: start must begin at 0, never decrease and stay below 2^32")
        self.names = names
        self.start = s.astype(np.uint32)
        self.lengths = np.diff(s).astype(np.uint32)

    @classmethod
    def single(cls, n_bases):
        """The whole text as one sequence named ""."""
        return cls([""], [0, int(n_bases)])

    @classmethod
    def from_lengths(cls, names, lengths):
        return cls(names, np.concatenate(([0], np.cumsum(np.asarray(lengths, np.int64)))))

    @property
    def n_bases(self):
        return int(self.start[-1])

    def __len__(self):
        return len(self.names)

    def __eq__(self, other):
        return isinstance(other, Contigs) and self.names == other.names and np.array_equal(self.start, other.start)

    def __repr__(self):
        return f"Contigs({len(self)} sequences, {self.n_bases} bases)"


def read_reference(path):
    """Multi-record FASTA -> (text, Contigs): text = every record's bases concatenated (uint8 ASCII; pass text.tobytes() to
    HostIndex.build or DeviceIndex.build_on_device), Contigs = where each record starts.  A character outside ACGT (N, lower
    case, IUPAC codes) raises BaseError, as building an index from it would."""
    from .engine import BaseError
    names, seqs = read_fasta(path)
    if not names:
        raise ValueError(f"{path}: no sequence")
    contigs = Contigs.from_lengths(names, [len(q) for q in seqs])
    text = np.concatenate(seqs) if seqs else np.zeros(0, np.uint8)
    bad = np.flatnonzero(~_VALID[text])
    if len(bad):
        p = int(bad[0])
        c = int(np.searchsorted(contigs.start, p, side="right")) - 1
        raise BaseError(f"{path}: sequence {names[c]!r} holds {chr(text[p])!r} at offset {p - int(contigs.start[c])}: only ACGT can be indexed")
    return text, contigs


def read_fastq(path, n_policy="error", pin=True, threads=0):
    """4-line FASTQ -> (bases uint8 (pinned when a GPU is present), base_off int64[n+1], dropped read indices).
    The file is cut into records and its sequence lines are gathered by the library's multi-threaded scanner
    (gsm_fastq_scan / gsm_fastq_gather).  bases/base_off go straight into
    ReadBatch.from_device_bases(bases_on_device, base_off=base_off, ascii=True); when all reads have one length,
    bases.reshape(n, L) is what PipelinedEngine.run_ascii takes."""
    import ctypes as C
    from . import _capi as capi
    if n_policy not in ("error", "drop"):
        raise ValueError("n_policy must be 'error' or 'drop'")
    buf = np.fromfile(path, dtype=np.uint8)
    n_rec = C.c_uint64()
    capi.check(capi.lib.gsm_fastq_scan(buf.ctypes.data, len(buf), C.byref(n_rec), None, None, 0, threads))
    n = int(n_rec.value)
    seq_off = np.zeros(max(n, 1), np.uint64)
    seq_len = np.zeros(max(n, 1), np.uint32)
    capi.check(capi.lib.gsm_fastq_scan(buf.ctypes.data, len(buf), C.byref(n_rec), seq_off.ctypes.data, seq_len.ctypes.data, max(n, 1), threads))

    def gather(so, sl):
        k = len(so)
        off = np.zeros(k + 1, np.uint64)
        total = int(sl.astype(np.int64).sum())
        if pin:
            import torch
            out = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=torch.cuda.is_available()).numpy()
        else:
            out = np.empty(max(total, 1), np.uint8)
        capi.check(capi.lib.gsm_fastq_gather(buf.ctypes.data, so.ctypes.data, sl.ctypes.data, k, out.ctypes.data, off.ctypes.data, threads))
        return out[:total], off.astype(np.int64)

    seq_off, seq_len = seq_off[:n], seq_len[:n]
    bases, off = gather(seq_off, seq_len)
    dropped = np.zeros(0, np.int64)
    if n_policy == "drop" and n:
        bad_byte = ~_VALID[bases]
        if bad_byte.any():
            nz = seq_len > 0
            per_read = np.zeros(n, np.int64)
            per_read[nz] = np.add.reduceat(bad_byte.astype(np.int64), off[:-1][nz])
            bad_read = per_read > 0
            dropped = np.flatnonzero(bad_read)
            keep = ~bad_read
            bases, off = gather(np.ascontiguousarray(seq_off[keep]), np.ascontiguousarray(seq_len[keep]))
    return bases, off, dropped


def fastq_cuts(buf, n_chunks):
    """Byte offsets that cut a 4-line FASTQ held in `buf` (uint8 array) into about n_chunks pieces at RECORD boundaries:
    near each even split point, the first line that starts with '@' and whose next-but-one line starts with '+' (a quality
    line may start with '@', but then the line two below it is a sequence line, never '+').  Only a few hundred bytes per
    cut are looked at; everything else of the parse runs on the GPU (PipelinedEngine.run_fastq)."""
    n = len(buf)
    cuts = [0]

    def line_end(p):
        while p < n:
            w = buf[p:p + 4096]
            k = np.flatnonzero(w == 10)
            if len(k):
                return p + int(k[0])
            p += 4096
        return n

    for i in range(1, max(int(n_chunks), 1)):
        p = max((n * i) // n_chunks, cuts[-1])
        while p < n:
            cand = line_end(p) + 1                     # start of the next line
            if cand >= n:
                p = n
                break
            if buf[cand] == 64:                        # '@'
                l2 = line_end(line_end(cand) + 1) + 1  # start of the line two below
                if l2 < n and buf[l2] == 43:           # '+'
                    p = cand
                    break
            p = cand
        if p < n and p > cuts[-1]:
            cuts.append(p)
    cuts.append(n)
    return cuts


def write_fastq(path, reads, names=None):
    """Small helper for tests and examples."""
    with open(path, "w") as f:
        for i, r in enumerate(reads):
            f.write(f"@{names[i] if names else 'r%d' % i}\n{r}\n+\n{'I' * len(r)}\n")
