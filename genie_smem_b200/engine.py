"""Batched device engine: torch owns the buffers, libgenie_smem (ctypes) does the work.

This is the layer the reference-shaped classes in surface.py sit on; bench.py and the parity
tests also call it directly.  Every search goes through the C ABI of include/genie_smem.h and
therefore through the CUDA kernels; nothing here computes a search result in Python.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi as capi
from .ingest import Contigs

RECORD_DTYPE = np.dtype([("read_id", "<u4"), ("qstart", "<u2"), ("qend", "<u2"), ("sa_lo", "<u4"), ("sa_hi", "<u4")])
HIT_DTYPE = np.dtype([("record", "<u4"), ("contig", "<u4"), ("offset", "<u4"), ("flags", "<u4")])
CHAIN_DTYPE = np.dtype([("slot", "<u4"), ("contig", "<u4"), ("rbeg", "<u4"), ("rend", "<u4"), ("q", "<u4"), ("weight", "<u4"),
                        ("n_seeds", "<u4"), ("reserved", "<u4")])
_BASES = np.frombuffer(b"ACGT", dtype=np.uint8)


class BaseError(KeyError, ValueError):
    """A read or reference holds a character outside ACGT (the reference raises KeyError there,
    SMEM/ExactMatch.py:139; SURVEY 8b asks for ValueError up front -- this is both)."""


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    if not torch.cuda.is_available():
        raise capi.GsmError(capi.E_NODEVICE, "no CUDA device visible: genie_smem_b200 has no CPU fallback")


def l2_fetch_granularity(set_bytes=0):
    """Get (and with set_bytes in {32, 64, 128} first request) the device's L2 fetch granularity."""
    require_cuda()
    cur = C.c_uint32()
    capi.check(capi.lib.gsm_device_l2_fetch_granularity(int(set_bytes), C.byref(cur)))
    return int(cur.value)


class HostIndex:
    """Host-side FM index handle (gsm_index).  Replaces ExactMatch.create_fm_index /
    load_fm_index (reference SMEM/ExactMatch.py:22-41)."""

    def __init__(self, handle):
        self._h = handle
        self.info = capi.IndexInfo()
        capi.check(capi.lib.gsm_index_info_get(self._h, C.byref(self.info)))

    @classmethod
    def build(cls, text, reverse=True):
        data = text if isinstance(text, (bytes, bytearray)) else text.encode()
        h = C.c_void_p()
        try:
            capi.check(capi.lib.gsm_index_build(bytes(data), len(data), 1 if reverse else 0, C.byref(h)))
        except ValueError as e:
            raise BaseError(str(e)) from None
        return cls(h)

    @classmethod
    def from_arrays(cls, text, suffix_array_1based, reverse=True):
        data = text if isinstance(text, (bytes, bytearray)) else text.encode()
        sa = np.ascontiguousarray(suffix_array_1based, dtype=np.uint32)
        if sa.shape[0] != len(data) + 1:
            raise ValueError("suffix_array must have len(text)+1 entries")
        h = C.c_void_p()
        try:
            capi.check(capi.lib.gsm_index_from_arrays(bytes(data), len(data), sa.ctypes.data, 1 if reverse else 0, C.byref(h)))
        except ValueError as e:
            if "ACGT" in str(e):
                raise BaseError(str(e)) from None
            raise
        return cls(h)

    @property
    def n_rows(self):
        return int(self.info.n_rows)

    @property
    def n_bases(self):
        return int(self.info.n_bases)

    def export(self):
        """-> (suffix_array uint32[n] 1-based, bwt bytes) in the reference's schema (ExactMatch.py:29-30)."""
        sa = np.zeros(self.n_rows, np.uint32)
        bwt = np.zeros(self.n_rows, np.uint8)
        capi.check(capi.lib.gsm_index_export(self._h, sa.ctypes.data, bwt.ctypes.data))
        return sa, bwt.tobytes()

    def count_dic(self):
        """fm_index["count_dic"] of the reference (ExactMatch.py:92-101)."""
        i = self.info
        return {"": int(i.n_rows), "$": 0, "A": int(i.C[0]), "C": int(i.C[1]), "G": int(i.C[2]), "T": int(i.C[3])}

    def pack(self, with_sa=True, with_text=True):
        i = self.info
        fwd = np.zeros(i.n_buckets * 16, np.uint32)
        rev = np.zeros(i.n_buckets * 16, np.uint32) if i.has_reverse else None
        sa = np.zeros(i.n_rows, np.uint32) if with_sa else None
        text = np.zeros(i.text_words + 2, np.uint32) if with_text else None
        capi.check(capi.lib.gsm_index_pack(self._h, fwd.ctypes.data, rev.ctypes.data if rev is not None else None,
                                           sa.ctypes.data if sa is not None else None, text.ctypes.data if text is not None else None))
        return fwd, rev, sa, text

    def close(self):
        if self._h is not None:
            capi.lib.gsm_index_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _to_dev(a, device):
    if a is None:
        return None
    a = np.asarray(a)
    if not a.flags.writeable:            # memory-mapped file: stage through RAM once
        a = np.array(a)
    t = torch.from_numpy(a.view(np.int32))
    return t.to(device, non_blocking=False)


class PackedIndex:
    """The device layouts of an index as host arrays, with a plain binary on-disk form (one directory:
    meta.json + fwd.npy, rev.npy, sa.npy, text.npy, memory-mappable).  Replaces the reference's
    pretty-printed <ref>-FM.json (SMEM/ExactMatch.py:32-39) for anything beyond toy sizes: a 1 Gbp
    index loads in seconds instead of being rebuilt (164 s of suffix sorting on the 16-core GPU box)."""

    FIELDS = ("n_bases", "n_rows", "n_buckets", "bucket_bytes", "text_words", "primary_fwd", "primary_rev", "has_reverse")

    def __init__(self, info, fwd, rev, sa, text):
        self.info, self.fwd, self.rev, self.sa, self.text = info, fwd, rev, sa, text

    @classmethod
    def from_host(cls, host: HostIndex, with_sa=True, with_text=True):
        return cls(host.info, *host.pack(with_sa, with_text))

    @classmethod
    def from_device(cls, index, with_sa=True, with_text=True):
        """Host copies of a DeviceIndex (e.g. one built on the GPU) so that it can be saved and reloaded."""
        def grab(t):
            return None if t is None else t.cpu().numpy().view(np.uint32)
        return cls(index.info, grab(index.fwd), grab(index.rev), grab(index.sa) if with_sa else None, grab(index.text) if with_text else None)

    def save(self, directory):
        import json as _json
        import os as _os
        _os.makedirs(directory, exist_ok=True)
        meta = {k: int(getattr(self.info, k)) for k in self.FIELDS}
        meta["count"] = [int(x) for x in self.info.count]
        meta["C"] = [int(x) for x in self.info.C]
        meta["format"] = "genie_smem_b200 packed index v1 (64-byte buckets = two 32-byte halves)"
        for name in ("fwd", "rev", "sa", "text"):
            a = getattr(self, name)
            if a is not None:
                np.save(_os.path.join(directory, name + ".npy"), a)
        with open(_os.path.join(directory, "meta.json"), "w") as f:
            _json.dump(meta, f, indent=1)

    @classmethod
    def load(cls, directory, mmap=True):
        import json as _json
        import os as _os
        with open(_os.path.join(directory, "meta.json")) as f:
            meta = _json.load(f)
        info = capi.IndexInfo()
        for k in cls.FIELDS:
            setattr(info, k, meta[k])
        for c in range(4):
            info.count[c] = meta["count"][c]
        for c in range(5):
            info.C[c] = meta["C"][c]
        arrs = []
        for name in ("fwd", "rev", "sa", "text"):
            p = _os.path.join(directory, name + ".npy")
            arrs.append(np.load(p, mmap_mode="r" if mmap else None) if _os.path.exists(p) else None)
        return cls(info, *arrs)


class IndexFile:
    """ONE memory-mappable file holding everything a search process needs, so that loading skips every rebuild: rank
    buckets of both directions, suffix array (full and / or sampled), packed text, the sweep's seed table, the dense LUT,
    the RMI parameters + None rows and (optionally) the RMI probe table.  Replaces the reference's three artefacts --
    <ref>-FM.json (ExactMatch.py:32-39), <ref>-LUT.json (LUT.py:50-63) and rmi_file.pkl (RMI_LUT.py:186-198).

    Layout: 8-byte magic "GSMIDX02", u64 length of a JSON header, the header (index info, per-section name / dtype /
    shape / offset / byte count / CRC-32, table parameters), then the sections, each starting on a 4096-byte boundary.
    """

    MAGIC = b"GSMIDX02"
    ALIGN = 4096

    @staticmethod
    def _sections(index, lut, rmi):
        def host(t):
            return None if t is None else t.detach().cpu().numpy()
        sec = [("fwd", host(index.fwd)), ("rev", host(index.rev)), ("sa", host(index.sa)), ("text", host(index.text)),
               ("ssa", host(getattr(index, "ssa", None))), ("seed_table", host(getattr(index, "seed_table", None))), ("lut", host(lut))]
        if rmi is not None:
            sec += [("rmi_params", host(rmi.params)), ("rmi_probe", host(rmi.probe))]
        return [(n, a) for n, a in sec if a is not None]

    @classmethod
    def save(cls, path, index, lut=None, lut_K=0, rmi=None, contigs=None):
        """index: DeviceIndex; lut: device table of lut_build (K = lut_K); rmi: RmiParams (None rows / probe table kept if built);
        contigs: the reference's sequence table (Contigs), stored as a "contigs" header key (names) and a contig_start section.
        Without contigs the file is exactly what earlier versions wrote."""
        import json as _json
        import zlib
        info = {k: int(getattr(index.info, k)) for k in PackedIndex.FIELDS}
        info["count"] = [int(x) for x in index.info.count]
        info["C"] = [int(x) for x in index.info.C]
        head = {"format": "genie_smem_b200 index file v2", "info": info, "seed_K": int(getattr(index, "seed_K", 0) or 0),
                "sa_sample": int(getattr(index, "sa_sample", 0) or 0), "lut_K": int(lut_K) if lut is not None else 0, "rmi": None, "sections": []}
        if rmi is not None:
            head["rmi"] = {"K": rmi.K, "level_sizes": [int(x) for x in rmi.level_sizes],
                           "none_rows": [int(x) for x in rmi.none_rows] if rmi.none_rows is not None else None,
                           "max_err": float(getattr(rmi, "max_err", -1.0))}
        secs = cls._sections(index, lut, rmi)
        if contigs is not None:
            if contigs.n_bases != int(index.info.n_bases):
                raise ValueError(f"contigs cover {contigs.n_bases} bases, the index {int(index.info.n_bases)}")
            head["contigs"] = list(contigs.names)
            secs.append(("contig_start", contigs.start))
        for n, a in secs:
            head["sections"].append({"name": n, "dtype": str(a.dtype), "shape": list(a.shape), "offset": 0, "nbytes": int(a.nbytes),
                                     "crc32": zlib.crc32(memoryview(np.ascontiguousarray(a)).cast("B")) & 0xFFFFFFFF})
        # offsets depend on the header length, which depends on the offsets' digits: reserve room, then fill
        blob = _json.dumps(head).encode()
        room = ((len(blob) + 16 + 64 * len(secs) + cls.ALIGN - 1) // cls.ALIGN) * cls.ALIGN
        off = room
        for d in head["sections"]:
            d["offset"] = off
            off += ((d["nbytes"] + cls.ALIGN - 1) // cls.ALIGN) * cls.ALIGN
        blob = _json.dumps(head).encode()
        assert 16 + len(blob) <= room
        with open(path, "wb") as f:
            f.write(cls.MAGIC)
            f.write(np.uint64(len(blob)).tobytes())
            f.write(blob)
            for d, (n, a) in zip(head["sections"], secs):
                f.seek(d["offset"])
                np.ascontiguousarray(a).tofile(f)
            f.truncate(off)
        return off

    @classmethod
    def header(cls, path):
        import json as _json
        with open(path, "rb") as f:
            if f.read(8) != cls.MAGIC:
                raise ValueError(f"{path}: not a genie_smem_b200 index file")
            n = int(np.frombuffer(f.read(8), np.uint64)[0])
            return _json.loads(f.read(n).decode())

    @classmethod
    def load(cls, path, device="cuda", verify=False):
        """-> (DeviceIndex, lut table or None, lut_K, RmiParams or None).  Sections are memory-mapped and copied to the
        device; nothing is rebuilt.  verify=True checks every section's CRC-32 first (ValueError on a mismatch).  The index's
        `contigs` is the file's sequence table, or None when it was saved without one."""
        import zlib
        require_cuda()
        head = cls.header(path)
        arrs = {}
        for d in head["sections"]:
            a = np.memmap(path, mode="r", dtype=np.dtype(d["dtype"]), offset=d["offset"], shape=tuple(d["shape"]))
            if verify and (zlib.crc32(memoryview(a).cast("B")) & 0xFFFFFFFF) != d["crc32"]:
                raise ValueError(f"{path}: section {d['name']} is corrupt (CRC-32 mismatch)")
            arrs[d["name"]] = a
        info = capi.IndexInfo()
        for k in PackedIndex.FIELDS:
            setattr(info, k, head["info"][k])
        for c in range(4):
            info.count[c] = head["info"]["count"][c]
        for c in range(5):
            info.C[c] = head["info"]["C"][c]
        dev = torch.device(device)

        def up(name):
            a = arrs.get(name)
            return None if a is None else torch.from_numpy(np.array(a)).to(dev)
        index = DeviceIndex.__new__(DeviceIndex)
        index.device, index.info, index.build_stats = dev, info, None
        index.fwd, index.rev, index.sa, index.text = up("fwd"), up("rev"), up("sa"), up("text")
        if "ssa" in arrs:
            index.ssa, index.sa_sample = up("ssa"), head["sa_sample"]
        if "seed_table" in arrs:
            index.seed_table, index.seed_K = up("seed_table"), head["seed_K"]
        index._bind()
        if "contigs" in head:
            index.set_contigs(Contigs(head["contigs"], np.array(arrs["contig_start"])))
        lut = up("lut")
        rmi = None
        if head["rmi"] is not None:
            p = np.array(arrs["rmi_params"])
            rmi = RmiParams(head["rmi"]["K"], head["rmi"]["level_sizes"], p[:, 0], p[:, 1], dev)
            rmi.max_err = head["rmi"]["max_err"]
            if head["rmi"]["none_rows"] is not None:
                rows = np.asarray(head["rmi"]["none_rows"], np.uint32)
                rmi.none_rows = rows
                rmi.c.none_rows = rows.ctypes.data_as(capi.u32p)
                rmi.c.n_none_rows = len(rows)
            if "rmi_probe" in arrs:
                rmi.probe = up("rmi_probe")
                rmi.c.probe = rmi.probe.data_ptr()
        return index, lut, head["lut_K"], rmi


class DeviceIndex:
    """The index resident in HBM: two bucket arrays (text / reversed text), optionally the full
    suffix array and the 2-bit text (needed by RMI and by position lookups)."""

    contigs = None          # sequence table (set_contigs); None = the text is one sequence
    _contig_start = None

    def __init__(self, host, device="cuda", with_sa=True, with_text=True):
        """host: a HostIndex (arrays are packed now) or a PackedIndex (arrays loaded from disk)."""
        require_cuda()
        self.device = torch.device(device)
        self.info = host.info
        if isinstance(host, PackedIndex):
            fwd, rev = host.fwd, host.rev
            sa, text = (host.sa if with_sa else None), (host.text if with_text else None)
        else:
            fwd, rev, sa, text = host.pack(with_sa, with_text)
        self.fwd = _to_dev(fwd, self.device)
        self.rev = _to_dev(rev, self.device)
        self.sa = _to_dev(sa, self.device)
        self.text = _to_dev(text, self.device)
        self.build_stats = None
        self._bind()

    def _bind(self):
        info = self.info
        d = capi.DevIndex()
        d.n_rows, d.n_buckets = info.n_rows, info.n_buckets
        d.fwd_buckets, d.rev_buckets = self.fwd.data_ptr(), (self.rev.data_ptr() if self.rev is not None else None)
        d.sa = self.sa.data_ptr() if self.sa is not None else None
        d.text2bit = self.text.data_ptr() if self.text is not None else None
        for c in range(5):
            d.C[c] = info.C[c]
        d.primary_fwd, d.primary_rev = info.primary_fwd, info.primary_rev
        seed = getattr(self, "seed_table", None)
        d.seed_K = getattr(self, "seed_K", 0) if seed is not None else 0
        d.seed_table = seed.data_ptr() if seed is not None else None
        self.c = d
        self.n_rows = int(info.n_rows)
        self.n_bases = int(info.n_bases)
        self.all_bases_present = all(int(info.count[c]) > 0 for c in range(4))

    @classmethod
    def build_on_device(cls, text, device="cuda", reverse=True):
        """Construct the whole index ON THE GPU (gsm_index_build_device: radix sort of 32-mer keys + prefix
        doubling, BWT planes, checkpoints) -- the large-reference replacement of ExactMatch.create_fm_index
        (reference SMEM/ExactMatch.py:22-33).  text: str / bytes of ACGT, or a uint8 array of codes 0..3
        (numpy or torch).  Arrays are bit-identical to HostIndex.build's."""
        require_cuda()
        self = cls.__new__(cls)
        self.device = dev = torch.device(device)
        if isinstance(text, str):
            text = text.encode()
        if isinstance(text, (bytes, bytearray)):
            src, ascii_ = torch.frombuffer(bytearray(text), dtype=torch.uint8), 1
        elif isinstance(text, np.ndarray):
            src, ascii_ = torch.from_numpy(np.ascontiguousarray(text, np.uint8)), 0
        else:
            src, ascii_ = text.contiguous(), 0
        n_bases = int(src.numel())
        if n_bases == 0:
            raise ValueError("empty reference")
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        with torch.cuda.device(dev):
            src = src.to(dev)
            words = (n_bases + 15) // 16 + 2
            self.text = torch.zeros(words + 2, dtype=torch.int32, device=dev)
            scratch = torch.zeros(1, dtype=torch.int64, device=dev)
            e0.record()
            try:
                capi.check(capi.lib.gsm_text_pack_device(_ptr(src), n_bases, ascii_, _ptr(self.text), _ptr(scratch), _stream()))
            except ValueError as e:
                raise BaseError(str(e)) from None
            del src
            n_rows = n_bases + 1
            nb = n_rows // 192 + 1
            flags = 1 if reverse else 0
            need = C.c_uint64()
            capi.check(capi.lib.gsm_index_build_device_workspace(n_bases, flags, C.byref(need)))
            self.sa = torch.empty(n_rows, dtype=torch.int32, device=dev)
            self.fwd = torch.empty(nb * 16, dtype=torch.int32, device=dev)
            self.rev = torch.empty(nb * 16, dtype=torch.int32, device=dev) if reverse else None
            ws = torch.empty(int(need.value), dtype=torch.uint8, device=dev)
            self.info = capi.IndexInfo()
            e1.record()
            capi.check(capi.lib.gsm_index_build_device(_ptr(self.text), n_bases, flags, _ptr(self.sa), _ptr(self.fwd), _ptr(self.rev),
                                                       _ptr(ws), int(need.value), C.byref(self.info), _stream()))
            e2.record()
            torch.cuda.synchronize(dev)
            del ws
            torch.cuda.empty_cache()
        self.build_stats = {"pack_ms": e0.elapsed_time(e1), "build_ms": e1.elapsed_time(e2), "workspace_bytes": int(need.value),
                            "doubling_rounds": int(self.info.reserved)}
        self.info.reserved = 0
        self._bind()
        return self

    def build_seed_table(self, K=None):
        """Seed table of the sweep kernel (gsm_seed_table_build): 4^K x 16 bytes; K defaults to the largest value that
        still leaves 2+ expected occurrences per k-mer (14 at 1-3 Gbp: 4.3 GB, 12 at 100 Mbp; measured on B200 at 1 Gbp:
        round-1 k_sweep 127 / 88 / 82 / 77 / 76 ms per 10 M reads for K = none / 11 / 12 / 13 / 14).  Results never depend on it."""
        if K is None:
            K = 1
            while K < 14 and self.n_rows / 4.0 ** (K + 1) >= 2.0:
                K += 1
        if self.rev is None:
            raise ValueError("the seed table needs the reverse-text buckets")
        K = int(K)
        self.seed_table, self.seed_K = None, 0
        self._bind()
        t = torch.empty((1 << (2 * K)) * 4, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            capi.check(capi.lib.gsm_seed_table_build(C.byref(self.c), K, _ptr(t), _stream()))
        self.seed_table, self.seed_K = t, K
        self._bind()
        return self

    def build_sampled_sa(self, sample=32, drop_full=False):
        """Keep every `sample`-th suffix-array value (gsm_sa_sample_build); positions then come from locate() by LF
        walking.  drop_full releases the 4-byte-per-base suffix array (RMI-SMEM and sa_lookup need it)."""
        if self.sa is None:
            raise ValueError("the sampled suffix array is derived from the full one")
        n = (self.n_rows + sample - 1) // sample
        self.ssa = torch.empty(n, dtype=torch.int32, device=self.device)
        self.sa_sample = int(sample)
        with torch.cuda.device(self.device):
            capi.check(capi.lib.gsm_sa_sample_build(C.byref(self.c), self.sa_sample, _ptr(self.ssa), _stream()))
        if drop_full:
            torch.cuda.synchronize(self.device)
            self.sa = None
            self._bind()
        return self

    def locate(self, rows):
        """rows -> 1-based text positions (ExactMatch.get_position(s), ExactMatch.py:191-199): direct suffix-array reads
        when the full array is resident, else LF walks to the sampled rows."""
        rows = np.ascontiguousarray(rows, np.uint32)
        if rows.size == 0:
            return np.zeros(0, np.uint32)
        if self.sa is not None:
            return sa_lookup(self, rows)
        if getattr(self, "ssa", None) is None:
            raise ValueError("no suffix array on the device: call build_sampled_sa() before dropping it")
        with torch.cuda.device(self.device):
            r = torch.from_numpy(rows.view(np.int32)).to(self.device)
            out = torch.empty_like(r)
            capi.check(capi.lib.gsm_locate_sampled_batch(C.byref(self.c), _ptr(self.ssa), self.sa_sample, rows.size, _ptr(r), _ptr(out), _stream()))
        return out.cpu().numpy().view(np.uint32)

    def set_contigs(self, contigs):
        """Attach the reference's sequence table (ingest.Contigs, e.g. from read_reference): hits are then reported as
        (sequence, offset).  Its start[n] must equal the index's base count.  None detaches it."""
        if contigs is None:
            self.contigs, self._contig_start, self._contigs_c = None, None, None
            return self
        if contigs.n_bases != self.n_bases:
            raise ValueError(f"contigs cover {contigs.n_bases} bases, the index {self.n_bases}")
        self._contig_start = torch.from_numpy(contigs.start.view(np.int32).copy()).to(self.device)
        self._contigs_c = capi.DevContigs(len(contigs), self._contig_start.data_ptr())
        self.contigs = contigs
        return self

    def drop_seed_table(self):
        self.seed_table, self.seed_K = None, 0
        self._bind()
        return self

    def suffix_array_host(self):
        """fm_index["suffix_array"] (1-based values, ExactMatch.py:66) copied back from the device."""
        return self.sa.cpu().numpy().view(np.uint32)

    def count_dic(self):
        i = self.info
        return {"": int(i.n_rows), "$": 0, "A": int(i.C[0]), "C": int(i.C[1]), "G": int(i.C[2]), "T": int(i.C[3])}

    def bytes(self):
        return sum(t.numel() * t.element_size() for t in (self.fwd, self.rev, self.sa, self.text, getattr(self, "seed_table", None)) if t is not None)


class ReadBatch:
    """Reads packed 2 bits/base, MSB-first, 16-byte aligned per read (include/genie_smem.h)."""

    def __init__(self, packed_u8, chunk_off, lens, max_len, read_id_base=0):
        self.packed_host, self.chunk_off_host, self.len_host = packed_u8, chunk_off, lens
        self.n = int(lens.shape[0])
        self.max_len = int(max_len)
        self.read_id_base = int(read_id_base)
        self.packed = self.chunk_off = self.len = None

    @classmethod
    def from_strings(cls, reads, read_id_base=0, pin=False):
        lens = np.asarray([len(r) for r in reads], np.uint32)
        joined = "".join(reads).encode()
        return cls._pack(joined, lens, read_id_base, pin)

    @classmethod
    def from_codes(cls, codes_u8, read_len, read_id_base=0, pin=False):
        """codes_u8: (n, read_len) array of base codes 0..3 (synthetic batches)."""
        n = codes_u8.shape[0]
        lens = np.full(n, read_len, np.uint32)
        joined = _BASES[np.ascontiguousarray(codes_u8).reshape(-1)].tobytes()
        return cls._pack(joined, lens, read_id_base, pin)

    @classmethod
    def _pack(cls, joined, lens, read_id_base, pin):
        n = int(lens.shape[0])
        off = np.zeros(n + 1, np.uint32)
        try:
            capi.check(capi.lib.gsm_pack_reads(joined, lens.ctypes.data, n, off.ctypes.data, None))
            nbytes = int(off[n]) * 16 + 16          # one readable pad chunk
            if pin and torch.cuda.is_available():
                packed_t = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
                packed = packed_t.numpy()
            else:
                packed = np.zeros(nbytes, np.uint8)
            capi.check(capi.lib.gsm_pack_reads(joined, lens.ctypes.data, n, off.ctypes.data, packed.ctypes.data))
        except ValueError as e:
            raise BaseError(str(e)) from None
        if pin and torch.cuda.is_available():          # offsets and lengths travel with every batch too
            off_t = torch.from_numpy(off.view(np.int32)).pin_memory()
            len_t = torch.from_numpy(np.ascontiguousarray(lens).view(np.int32)).pin_memory()
            off, lens = off_t.numpy().view(np.uint32), len_t.numpy().view(np.uint32)
        return cls(packed, off, lens, max(1, int(lens.max())) if n else 1, read_id_base)

    @classmethod
    def from_device_bases(cls, bases, read_len=None, base_off=None, ascii=False, read_id_base=0, check=True):
        """Pack ON THE GPU (gsm_pack_reads_device).  bases: torch uint8 on the device -- an (n, read_len) matrix of
        codes 0..3 / ASCII bytes, or a flat buffer with base_off (n+1 int64 offsets, numpy or torch).  The batch
        lives on the device; to_host() makes the (pinned) host copies the end-to-end paths start from."""
        require_cuda()
        dev = bases.device
        if base_off is None:
            if bases.dim() == 2:
                read_len = int(bases.shape[1])
            n = bases.numel() // int(read_len)
            lens = np.full(n, int(read_len), np.uint32)
            cpr = (int(read_len) + 63) // 64
            off = (np.arange(n + 1, dtype=np.int64) * cpr)
            boff_t = None
        else:
            boff = np.asarray(base_off.cpu() if isinstance(base_off, torch.Tensor) else base_off, np.int64)
            n = len(boff) - 1
            lens = np.diff(boff).astype(np.uint32)
            off = np.concatenate([[0], np.cumsum((lens.astype(np.int64) + 63) // 64)])
            boff_t = torch.from_numpy(boff).to(dev)
        if n and int(off[-1]) >= 1 << 32:
            raise capi.GsmError(capi.E_CAPACITY, "read batch too large for 32-bit chunk offsets")
        self = cls(None, off.astype(np.uint32), lens, max(1, int(lens.max())) if n else 1, read_id_base)
        with torch.cuda.device(dev):
            self.chunk_off = torch.from_numpy(self.chunk_off_host.view(np.int32)).to(dev)
            self.packed = torch.empty(int(off[-1]) * 16 + 16, dtype=torch.uint8, device=dev)
            self.packed[int(off[-1]) * 16:].zero_()
            self.len = torch.empty(max(n, 1), dtype=torch.int32, device=dev)[:n]
            scratch = torch.zeros(1, dtype=torch.int64, device=dev)
            flat = bases.contiguous().view(-1)
            capi.check(capi.lib.gsm_pack_reads_device(_ptr(flat), _ptr(boff_t), 0 if boff_t is not None else int(read_len), _ptr(self.chunk_off), n,
                                                      1 if ascii else 0, _ptr(self.packed), _ptr(self.len), _ptr(scratch), _stream()))
            if check:
                try:
                    capi.check(capi.lib.gsm_pack_reads_device_check(_ptr(scratch), _stream()))
                except ValueError as e:
                    raise BaseError(str(e)) from None
        return self

    def to_host(self, pin=True):
        """Host copies of a device-built batch (pinned by default): what Engine.run / PipelinedEngine.run copy in."""
        def grab(t):
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=bool(pin))
            h.copy_(t)
            return h.numpy()
        self.packed_host = grab(self.packed)
        self.chunk_off_host = grab(self.chunk_off).view(np.uint32)
        self.len_host = grab(self.len).view(np.uint32)
        return self

    def to(self, device, non_blocking=False):
        self.packed = torch.from_numpy(self.packed_host).to(device, non_blocking=non_blocking)
        self.chunk_off = torch.from_numpy(self.chunk_off_host.view(np.int32)).to(device, non_blocking=non_blocking)
        self.len = torch.from_numpy(self.len_host.view(np.int32)).to(device, non_blocking=non_blocking)
        return self

    def h2d_bytes(self):
        return self.packed_host.nbytes + self.chunk_off_host.nbytes + self.len_host.nbytes

    def cstruct(self):
        r = capi.DevReads()
        r.n_reads = self.n
        r.packed, r.chunk_off, r.len = self.packed.data_ptr(), self.chunk_off.data_ptr(), self.len.data_ptr()
        r.max_len, r.read_id_base = self.max_len, self.read_id_base
        return r

    def both_strands(self):
        """The strand-doubled batch, built on the device (gsm_reads_both_strands_device): 2n reads, slot 2i = read i as
        given, slot 2i+1 = its reverse complement, read_id_base = 2 * self.read_id_base, so that a record's read_id >> 1
        is the read and read_id & 1 its strand.  A batch that only lives on the host is copied to the current CUDA
        device first.  Raises ValueError when the doubled read ids would reach 2^32."""
        require_cuda()
        _check_doubled_ids(self.read_id_base, self.n)
        if self.packed is None:
            self.to(torch.device("cuda"))
        dev = self.packed.device
        n = self.n
        co = self.chunk_off_host if self.chunk_off_host is not None else self.chunk_off.cpu().numpy().view(np.uint32)
        c = co[: n + 1].astype(np.int64) - int(co[0])
        coff = np.empty(2 * n + 1, np.int64)
        coff[0::2], coff[1::2] = 2 * c, c[:-1] + c[1:]
        if coff[-1] >= 1 << 32:
            raise capi.GsmError(capi.E_CAPACITY, "strand-doubled batch too large for 32-bit chunk offsets")
        lens = self.len_host if self.len_host is not None and len(self.len_host) == n else self.len[:n].cpu().numpy().view(np.uint32)
        out = ReadBatch(None, coff.astype(np.uint32), np.repeat(np.asarray(lens, np.uint32), 2), self.max_len, 2 * self.read_id_base)
        with torch.cuda.device(dev):
            out.packed = torch.empty(int(coff[-1]) * 16 + 16, dtype=torch.uint8, device=dev)
            out.chunk_off = torch.empty(2 * n + 1, dtype=torch.int32, device=dev)
            out.len = torch.empty(max(2 * n, 1), dtype=torch.int32, device=dev)[: 2 * n]
            capi.check(capi.lib.gsm_reads_both_strands_device(C.byref(self.cstruct()), _ptr(out.packed), _ptr(out.chunk_off), _ptr(out.len), _stream()))
        return out


def _check_doubled_ids(read_id_base, n):
    if 2 * (int(read_id_base) + int(n)) >= 1 << 32:
        raise ValueError(f"strands=2: read ids 2 * ({read_id_base} + {n}) do not fit in 32 bits")


class RmiParams:
    """(coef, intercept) per linear model of an RMI (reference SMEM/RMI.py), on the device."""

    def __init__(self, K, level_sizes, coef, intercept, device="cuda"):
        self.K = int(K)
        self.level_sizes = np.asarray(level_sizes, np.uint32)
        self.coef_host = np.ascontiguousarray(coef, np.float64)
        self.intercept_host = np.ascontiguousarray(intercept, np.float64)
        assert self.coef_host.shape[0] == int(self.level_sizes.sum()) == self.intercept_host.shape[0]
        # one interleaved {coef, intercept} array: a model is one 16-byte line, and one L2 persistence window covers all
        self.params = torch.from_numpy(np.stack([self.coef_host, self.intercept_host], axis=1).copy()).to(device)
        self.coef, self.intercept = self.params[:, 0], self.params[:, 1]
        s = capi.DevRmi()
        s.K, s.n_levels = self.K, len(self.level_sizes)
        s.level_sizes = self.level_sizes.ctypes.data_as(capi.u32p)
        s.coef, s.intercept = self.params.data_ptr(), self.params.data_ptr() + 8
        s.param_stride = 2
        s.probe = None
        s.bounds = None
        s.none_rows, s.n_none_rows = None, 0
        s.hazard_slots, s.hazard_n_slots, s.reserved0 = None, 0, 0
        self.c = s
        self.probe = None
        self.bounds = None
        self.none_rows = None
        self.hazard_slots = None
        self.n_hazards = None

    def persist_in_l2(self, on=True):
        """Pin the model parameters in the persisting L2 for kernels of the current stream (gsm_l2_persist): every
        prediction reads one random 16-byte line of this array per level."""
        with torch.cuda.device(self.params.device):
            if on:
                capi.check(capi.lib.gsm_l2_persist(_ptr(self.params), self.params.numel() * 8, _stream()))
            else:
                capi.check(capi.lib.gsm_l2_persist(None, 0, _stream()))
        return self

    def build_none_rows(self, index):
        """The K rows where get_ref_seq returns None (gsm_rmi_none_rows): lets the selection kernel run the
        error-bounded fast search wherever it provably equals the literal one.  Results never depend on it."""
        rows = np.zeros(self.K, np.uint32)
        scratch = torch.zeros(33, dtype=torch.int32, device=index.device)
        with torch.cuda.device(index.device):
            capi.check(capi.lib.gsm_rmi_none_rows(C.byref(index.c), self.K, rows.ctypes.data, _ptr(scratch), _stream()))
        self.none_rows = rows
        self.c.none_rows = rows.ctypes.data_as(capi.u32p)
        self.c.n_none_rows = self.K
        return self

    def build_bounds_table(self, index):
        """Dense {first row >= k-mer, occurrences} pair per K-mer code (gsm_rmi_bounds_build; 4^K x 8 B of HBM, 8.6 GB for
        K = 15): with the None rows, every RMI lookup of the selection kernel is the model prediction plus ONE fetch.
        Results never depend on it."""
        if self.K > 16:
            raise ValueError("bounds table: K must be <= 16")
        self.bounds = torch.empty((1 << (2 * self.K)) * 2, dtype=torch.int32, device=index.device)
        with torch.cuda.device(index.device):
            capi.check(capi.lib.gsm_rmi_bounds_build(C.byref(index.c), self.K, _ptr(self.bounds), _stream()))
        self.c.bounds = self.bounds.data_ptr()
        if self.none_rows is not None and self.K <= 15:
            self.build_hazard_filter(index)
        return self

    def drop_bounds_table(self):
        self.bounds = None
        self.c.bounds = None
        return self.drop_hazard_filter()

    def build_hazard_filter(self, index, max_codes=1 << 18):
        """The model's HAZARD codes -- the K-mers whose last-mile search is not certified to return the true interval, a few
        per million for a model worth using -- as a hash set on the device (gsm_rmi_hazard_scan over all 4^K codes, then
        gsm_rmi_hazard_hash on the host).  With it gsm_smem_select(RMI) hands every read without a hazard window to the
        BWA-SMEM selection (same records, include/genie_smem.h) and runs the frame machine on the others only.  Needs the
        None rows and the bounds table (build_bounds_table calls this).  A model with more than max_codes hazards gets no
        filter (self.n_hazards says how many there were).  Results never depend on it."""
        if self.bounds is None or self.none_rows is None:
            raise ValueError("hazard filter: build_none_rows and build_bounds_table first")
        if self.K > 15:
            raise ValueError("hazard filter: K must be <= 15")
        self.drop_hazard_filter()
        codes = torch.empty(max_codes, dtype=torch.int32, device=index.device)
        count = torch.zeros(1, dtype=torch.int64, device=index.device)
        found = C.c_uint64(0)
        with torch.cuda.device(index.device):
            capi.check(capi.lib.gsm_rmi_hazard_scan(C.byref(index.c), C.byref(self.c), _ptr(codes), max_codes, _ptr(count), C.byref(found), _stream()))
        self.n_hazards = int(found.value)
        if self.n_hazards > max_codes:
            return self
        host = codes[:self.n_hazards].cpu().numpy().view(np.uint32)
        n_slots = 1024
        while n_slots < 4 * self.n_hazards + 4:
            n_slots *= 2
        slots = np.empty(n_slots, np.uint32)
        capi.check(capi.lib.gsm_rmi_hazard_hash(host.ctypes.data, self.n_hazards, slots.ctypes.data, n_slots))
        self.hazard_slots = torch.from_numpy(slots.view(np.int32)).to(index.device)
        self.c.hazard_slots = self.hazard_slots.data_ptr()
        self.c.hazard_n_slots = n_slots
        return self

    def drop_hazard_filter(self):
        self.hazard_slots = None
        self.c.hazard_slots = None
        self.c.hazard_n_slots = 0
        return self

    def build_probe_table(self, index):
        """16-byte {SA value, 32-mer code} record per row: one fetch per last-mile probe (n_rows x 16 B of HBM)."""
        self.probe = torch.empty(index.n_rows * 16, dtype=torch.uint8, device=index.device)
        capi.check(capi.lib.gsm_rmi_probe_build(C.byref(index.c), _ptr(self.probe), _stream()))
        self.c.probe = self.probe.data_ptr()
        return self


class SmemResult:
    """Records of one batch in (read, emission) order + CSR offsets per read.

    strands = 2 (an engine built with strands=2): the batch was searched strand-doubled, so offsets, status and the records'
    read ids are per SLOT -- slot 2i is read i as given, slot 2i+1 its reverse complement, read_id = 2 * (read_id_base + i)
    + strand, and a strand-1 record's qstart / qend are in the reverse complement's coordinates.  `lengths` then holds the
    length of every read (uint32), which read_coords() needs.

    Lifetime: by default the arrays are the caller's own copies.  With reuse_host_buffers=True (Engine.run /
    PipelinedEngine.run*) they are VIEWS of the engine's pinned staging buffers and are overwritten by that engine's
    next run -- the zero-copy mode bench.py times; copy what you keep."""

    def __init__(self, records, offsets, status, n_mems, strands=1, lengths=None):
        self.records, self.offsets, self.status, self.n_mems = records, offsets, status, n_mems
        self.strands, self.lengths = strands, lengths

    def detach(self):
        self.records, self.offsets, self.status = self.records.copy(), self.offsets.copy(), self.status.copy()
        if self.lengths is not None:
            self.lengths = self.lengths.copy()
        return self

    def _slots(self, i, strand):
        """Slot range [a, b) of read i: both strands (strand None) or one."""
        if strand not in (None, 0, 1) or (self.strands == 1 and strand == 1):
            raise ValueError(f"strand must be None, 0{' or 1' if self.strands == 2 else ''}")
        if self.strands == 1:
            return i, i + 1
        return (2 * i, 2 * i + 2) if strand is None else (2 * i + strand, 2 * i + strand + 1)

    def for_read(self, i, strand=None):
        """Records of read i; with strands = 2 those of both its slots (strand None, slot 2i first) or of one strand."""
        a, b = self._slots(i, strand)
        return self.records[self.offsets[a]:self.offsets[b]]

    def read_coords(self):
        """Per-record arrays in the ORIGINAL read's orientation: `read` (read_id >> 1 with strands = 2, else read_id),
        `strand` (0 / 1), and the matched bases read[qbeg:qend] -- for a strand-1 record qbeg = L - qend, qend = L - qstart,
        the same bases seen on the reverse strand."""
        rid = self.records["read_id"]
        qs, qe = self.records["qstart"].astype(np.uint32), self.records["qend"].astype(np.uint32)
        if self.strands == 1:
            return {"read": rid.copy(), "strand": np.zeros(len(rid), np.uint8), "qbeg": qs, "qend": qe}
        slot = np.repeat(np.arange(len(self.offsets) - 1), np.diff(self.offsets))
        strand = (rid & 1).astype(np.uint8)
        L = np.asarray(self.lengths, np.uint32)[slot >> 1]
        rev = strand == 1
        return {"read": rid >> 1, "strand": strand, "qbeg": np.where(rev, L - qe, qs), "qend": np.where(rev, L - qs, qe)}


class HitResult:
    """Hits of a record array (HIT_DTYPE: record, contig, offset, flags), in record order and within a record in
    suffix-array row order, + CSR offsets per record (int64, one entry per record plus one).  Host arrays of their own."""

    def __init__(self, hits, offsets):
        self.hits, self.offsets = hits, offsets

    def for_record(self, k):
        return self.hits[self.offsets[k]:self.offsets[k + 1]]

    def for_read(self, result, i, strand=None):
        """Hits of read i of `result`, the SmemResult whose records these hits were located from (strand as in
        SmemResult.for_read)."""
        a, b = result._slots(i, strand)
        return self.hits[self.offsets[result.offsets[a]]:self.offsets[result.offsets[b]]]

    def __len__(self):
        return len(self.hits)


class ChainResult:
    """BWA-MEM's co-linear chains of every slot (chain_seeds has the semantics): `chains` (CHAIN_DTYPE) in slot order, within
    a slot in (contig, rbeg) order; `offsets` (int64, one entry per slot plus one); `hits`, the HitResult of the slots'
    records; `hit_chain` (u32 per hit): the index within its slot of the chain the hit belongs to, | CHAIN_CONTAINED when it
    was contained in that chain rather than appended, CHAIN_NONE for a spanning hit; `rec_offsets`: the records of each slot
    (the SmemResult's offsets).  strands / lengths as in SmemResult.  Host arrays of their own."""

    def __init__(self, chains, offsets, hits, hit_chain, rec_offsets, strands=1, lengths=None):
        self.chains, self.offsets, self.hits, self.hit_chain = chains, offsets, hits, hit_chain
        self.rec_offsets, self.strands, self.lengths = rec_offsets, strands, lengths

    def __len__(self):
        return len(self.chains)

    def for_read(self, i, strand=None):
        """Chains of read i: with strands = 2 those of both its slots (strand None, slot 2i first) or of one strand."""
        a, b = SmemResult._slots(self, i, strand)
        return self.chains[self.offsets[a]:self.offsets[b]]

    def seeds(self, k):
        """Indices into hits.hits of the member seeds of chain k, in member order (contained seeds are not members)."""
        s = int(self.chains["slot"][k])
        a, b = int(self.hits.offsets[self.rec_offsets[s]]), int(self.hits.offsets[self.rec_offsets[s + 1]])
        return a + np.flatnonzero(self.hit_chain[a:b] == np.uint32(k - int(self.offsets[s])))

    def read_coords(self):
        """Per-chain arrays in the ORIGINAL read's orientation: `read` (the read's index in the batch), `strand`, and qbeg /
        qend -- for a strand-1 chain qbeg = L - qend, qend = L - qbeg of its reverse-complement coordinates."""
        slot = self.chains["slot"].astype(np.int64)
        q = self.chains["q"]
        qb, qe = (q & 0xFFFF).astype(np.uint32), (q >> 16).astype(np.uint32)
        if self.strands == 1:
            return {"read": slot, "strand": np.zeros(len(slot), np.uint8), "qbeg": qb, "qend": qe}
        strand = (slot & 1).astype(np.uint8)
        L = np.asarray(self.lengths, np.uint32)[slot >> 1]
        rev = strand == 1
        return {"read": slot >> 1, "strand": strand, "qbeg": np.where(rev, L - qe, qb), "qend": np.where(rev, L - qb, qe)}

    def best(self):
        """Per read, the index of its heaviest chain over its slots, or -1 without chains; ties go to the lower slot, then to
        the earlier chain."""
        n_reads = (len(self.offsets) - 1) // self.strands
        out = np.full(n_reads, -1, np.int64)
        if len(self.chains):
            read = self.chains["slot"].astype(np.int64) // self.strands
            order = np.lexsort((np.arange(len(read)), -self.chains["weight"].astype(np.int64), read))
            first = order[np.r_[True, read[order][1:] != read[order][:-1]]]
            out[read[first]] = first
        return out


class Engine:
    """Owns the workspace for batches of up to `max_reads` reads of up to `max_len` bases.

    strands = 2: run() searches every read and its reverse complement in one batch.  The batch is strand-doubled on the
    device (ReadBatch.both_strands: slot 2i = read i, slot 2i+1 = its reverse complement) into buffers of this engine,
    so the workspace holds 2 * max_reads slots, and the result is per slot (SmemResult.strands = 2).  sweep / select /
    launch take the batch they are given, doubled or not."""

    def __init__(self, index: DeviceIndex, max_reads, max_len, mems_per_read=24, recs_per_read=16, strands=1):
        require_cuda()
        if strands not in (1, 2):
            raise ValueError("strands must be 1 or 2")
        self.index = index
        self.device = index.device
        self.max_reads, self.max_len = int(max_reads), int(max_len)
        self.strands = int(strands)
        self.slots = self.strands * self.max_reads
        wi = capi.WorkspaceInfo()
        capi.check(capi.lib.gsm_smem_workspace_info(self.slots, self.max_len, C.byref(wi)))
        self.grid = (int(wi.grid_blocks), int(wi.block_threads))
        dev = self.device
        n = max(self.slots, 1)
        self.mem_cap = min(max(n * mems_per_read, 4096), (1 << 32) - 1)
        self.rec_cap = min(max(n * recs_per_read, 4096), (1 << 32) - 1)
        self.mem_pool = torch.empty(self.mem_cap * 16, dtype=torch.uint8, device=dev)
        self.scratch = torch.empty(int(wi.quad_scratch_bytes), dtype=torch.uint8, device=dev)
        self.mem_off = torch.empty(n, dtype=torch.int32, device=dev)
        self.mem_cnt = torch.empty(n, dtype=torch.int32, device=dev)
        self.rec_tmp = torch.empty(self.rec_cap * 16, dtype=torch.uint8, device=dev)
        self.rec_tmp_off = torch.empty(n, dtype=torch.int32, device=dev)
        self.rec_cnt = torch.empty(n, dtype=torch.int32, device=dev)
        self.rec_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
        self.read_status = torch.empty(n, dtype=torch.uint8, device=dev)
        self.counters = torch.zeros(8, dtype=torch.int64, device=dev)
        self.scan_tmp = torch.empty(int(wi.scan_tmp_bytes), dtype=torch.uint8, device=dev)
        self.records = torch.empty(self.rec_cap * 16, dtype=torch.uint8, device=dev)
        w = capi.Workspace()
        w.mem_pool, w.mem_cap = self.mem_pool.data_ptr(), self.mem_cap
        w.quad_scratch, w.quad_scratch_bytes = self.scratch.data_ptr(), self.scratch.numel()
        w.mem_off, w.mem_cnt = self.mem_off.data_ptr(), self.mem_cnt.data_ptr()
        w.rec_tmp, w.rec_cap = self.rec_tmp.data_ptr(), self.rec_cap
        w.rec_tmp_off, w.rec_cnt, w.rec_off = self.rec_tmp_off.data_ptr(), self.rec_cnt.data_ptr(), self.rec_off.data_ptr()
        w.read_status, w.counters = self.read_status.data_ptr(), self.counters.data_ptr()
        w.scan_tmp, w.scan_tmp_bytes = self.scan_tmp.data_ptr(), self.scan_tmp.numel()
        self.ws = w
        self.kernel_launches = 0
        self._pin = {}
        self.last_d2h_bytes = 0
        if self.strands == 2:                     # the strand-doubled batch: 2 * max_reads reads of up to max_len bases
            m = max(self.max_reads, 1)
            self.ds_packed = torch.empty(2 * m * ((self.max_len + 63) // 64) * 16 + 16, dtype=torch.uint8, device=dev)
            self.ds_chunk_off = torch.empty(2 * m + 1, dtype=torch.int32, device=dev)
            self.ds_len = torch.empty(2 * m, dtype=torch.int32, device=dev)

    def _both_strands(self, reads):
        """Strand-double reads (a ReadBatch or a view of one on the device) into this engine's buffers, on the current
        stream; -> the doubled batch as a view, read_id_base and lo doubled."""
        if reads.n > self.max_reads or reads.max_len > self.max_len:
            raise ValueError("batch exceeds the engine's workspace")
        _check_doubled_ids(reads.read_id_base, reads.n)
        capi.check(capi.lib.gsm_reads_both_strands_device(C.byref(reads.cstruct()), _ptr(self.ds_packed), _ptr(self.ds_chunk_off),
                                                          _ptr(self.ds_len), _stream()))
        self.kernel_launches += 1
        return _ChunkView(self.ds_packed, self.ds_chunk_off, self.ds_len, 2 * reads.n, reads.max_len, 2 * reads.read_id_base,
                          2 * getattr(reads, "lo", 0))

    # -- device-resident phases: kernels only (bench.py times these as `value`)
    def _check_batch(self, reads):
        if reads.n > self.slots or reads.max_len > self.max_len:
            raise ValueError("batch exceeds the engine's workspace")
        self._reads_c = reads.cstruct()
        return self._reads_c

    def sweep(self, reads: ReadBatch):
        """k_sweep1: every maximal exact match of every read (method-independent FM walk; also leaves the BWA-SMEM picks)."""
        r = self._check_batch(reads)
        capi.check(capi.lib.gsm_smem_sweep(C.byref(self.index.c), C.byref(r), C.byref(self.ws), _stream()))
        self.kernel_launches += 1 if reads.n else 0

    def select(self, method, reads: ReadBatch, min_len=1, K=0, lut=None, rmi: RmiParams = None, gatherer=None):
        """k_select + scan + ordered write: the reference's records for one method, in (read, emission) order -- into
        this engine's `records` buffer, or with a sharding.RecordGatherer straight into the gathering rank's HBM."""
        if gatherer is not None and self.strands == 2:
            raise ValueError("strands=2 does not support a gatherer")
        r = self._check_batch(reads)
        capi.check(capi.lib.gsm_smem_select(method, C.byref(self.index.c), C.byref(r), int(min_len), int(K), _ptr(lut),
                                            C.byref(rmi.c) if rmi is not None else None, C.byref(self.ws), _stream()))
        # RMI with a hazard filter: + k_rmi_prefilter and k_select<BWA> for the reads without a hazard window (the library
        # applies the same conditions; a workspace too small for the read queue only makes this count two too high)
        pre = 2 if (reads.n and method == capi.METHOD_RMI and rmi is not None and rmi.hazard_slots is not None and rmi.bounds is not None
                    and capi.lib.gsm_option_rmi_prefilter(-1) != 0) else 0
        if gatherer is not None:
            gatherer.collect(self, r)
            self.kernel_launches += ((8 if self._picks_path(method) else 7) + pre) if reads.n else 1
            return
        capi.check(capi.lib.gsm_smem_collect(C.byref(r), C.byref(self.ws), _ptr(self.records), self.rec_cap, _stream()))
        # BWA: picked / queued / finish; LUT, RMI: select + the deferred explicit searches; then 3 scan kernels, ordered write
        self.kernel_launches += ((7 if self._picks_path(method) else 6) + pre) if reads.n else 0

    @staticmethod
    def _picks_path(method):
        """BWA-SMEM, and LUT-SMEM unless the frame machine is asked for: picked / queued / finish kernels."""
        return method == capi.METHOD_BWA or (method == capi.METHOD_LUT and capi.lib.gsm_option_lut_frame_machine(-1) == 0)

    def collect_local(self, reads: ReadBatch):
        """(Re)write the records of the batch just selected into this engine's own `records` buffer."""
        r = self._check_batch(reads)
        capi.check(capi.lib.gsm_smem_collect(C.byref(r), C.byref(self.ws), _ptr(self.records), self.rec_cap, _stream()))

    def launch(self, method, reads: ReadBatch, min_len=1, K=0, lut=None, rmi: RmiParams = None, gatherer=None):
        self.sweep(reads)
        self.select(method, reads, min_len, K, lut, rmi, gatherer)

    def check_overflow(self):
        c = self.counters.cpu().numpy()
        if c[2] != 0:
            raise capi.GsmError(capi.E_CAPACITY, f"workspace overflow (flags {int(c[2])}): mems {int(c[0])}/{self.mem_cap}, "
                                                 f"records {int(c[1])}/{self.rec_cap}")
        return int(c[0]), int(c[1])

    def _pinned(self, name, nbytes):
        buf = self._pin.get(name)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8).pin_memory()
            self._pin[name] = buf
        return buf

    # -- end-to-end step: host reads in (H2D), host records out (D2H)
    def run(self, method, reads: ReadBatch, min_len=1, K=0, lut=None, rmi: RmiParams = None, grow=True, reuse_host_buffers=False):
        """Host reads in (H2D), host records out (D2H).  With strands=2 the batch is strand-doubled on the device first and
        the result is per slot (SmemResult.strands = 2)."""
        reads.to(self.device, non_blocking=True)
        if self.strands == 2:
            reads = self._both_strands(reads)
        while True:
            self.launch(method, reads, min_len, K, lut, rmi)
            try:
                n_mems, n_rec = self.check_overflow()
                break
            except capi.GsmError as e:
                if e.code != capi.E_CAPACITY or not grow:
                    raise
                self._grow()
        n = reads.n
        hrec = self._pinned("rec", n_rec * 16)
        hoff = self._pinned("off", (n + 1) * 8)
        hst = self._pinned("st", max(n, 1))
        hrec[: n_rec * 16].copy_(self.records[: n_rec * 16], non_blocking=True)
        hoff[: (n + 1) * 8].copy_(self.rec_off[: n + 1].view(torch.uint8), non_blocking=True)
        hst[:n].copy_(self.read_status[:n], non_blocking=True)
        lengths = None
        if self.strands == 2:
            hlen = self._pinned("len", max(n, 1) * 4)
            hlen[: n * 4].copy_(self.ds_len[:n].view(torch.uint8), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last_d2h_bytes = n_rec * 16 + (n + 1) * 8 + n + 64
        if self.strands == 2:
            lengths = hlen.numpy()[: n * 4].view(np.uint32)[0::2]
            self.last_d2h_bytes += n * 4
        recs = hrec.numpy()[: n_rec * 16].view(RECORD_DTYPE)
        offs = hoff.numpy()[: (n + 1) * 8].view(np.int64)
        res = SmemResult(recs, offs, hst.numpy()[:n], n_mems, self.strands, lengths)
        return res if reuse_host_buffers else res.detach()

    def locate_hits(self, max_occ=500, min_len=0, hit_cap=None):
        """Hits of the records of the batch this engine selected last, located on the device straight from its record
        buffer (locate_hits has the semantics)."""
        _, n_rec = self.check_overflow()
        return _expand_hits(self.index, self.records, n_rec, max_occ, min_len, hit_cap)

    def chain_seeds(self, max_occ=500, min_len=19, w=100, max_gap=10000):
        """Chains of the batch this engine selected last (chain_seeds has the semantics): hits are located from the engine's
        record buffer into device memory and chained there; only the results are copied back."""
        r = getattr(self, "_reads_c", None)
        if r is None:
            raise ValueError("no batch has been selected yet")
        _, n_rec = self.check_overflow()
        n = int(r.n_reads)
        rec_offsets = self.rec_off[: n + 1].cpu().numpy()
        lengths = self.ds_len[:n].cpu().numpy().view(np.uint32)[0::2].copy() if self.strands == 2 else None
        return _chain(self.index, self.records, n_rec, self.rec_off, rec_offsets, max_occ, min_len, w, max_gap, self.strands, lengths)

    def _grow(self):
        dev = self.device
        self.mem_cap = min(self.mem_cap * 4, (1 << 32) - 1)
        self.rec_cap = min(self.rec_cap * 4, (1 << 32) - 1)
        self.mem_pool = torch.empty(self.mem_cap * 16, dtype=torch.uint8, device=dev)
        self.rec_tmp = torch.empty(self.rec_cap * 16, dtype=torch.uint8, device=dev)
        self.records = torch.empty(self.rec_cap * 16, dtype=torch.uint8, device=dev)
        self.ws.mem_pool, self.ws.mem_cap = self.mem_pool.data_ptr(), self.mem_cap
        self.ws.rec_tmp, self.ws.rec_cap = self.rec_tmp.data_ptr(), self.rec_cap


# ---------------------------------------------------------------------------- batched primitives
def backsearch_batch(index: DeviceIndex, reads: ReadBatch):
    """exact_match_back_prop for every read -> (lo, cnt) uint32 arrays; cnt == 0 <=> reference -1."""
    require_cuda()
    reads.to(index.device)
    lo = torch.empty(max(reads.n, 1), dtype=torch.int32, device=index.device)
    cnt = torch.empty(max(reads.n, 1), dtype=torch.int32, device=index.device)
    r = reads.cstruct()
    capi.check(capi.lib.gsm_backsearch_batch(C.byref(index.c), C.byref(r), _ptr(lo), _ptr(cnt), _stream()))
    return lo[: reads.n].cpu().numpy().view(np.uint32), cnt[: reads.n].cpu().numpy().view(np.uint32)


def add_one_batch(index: DeviceIndex, bases, lo, cnt):
    """exact_match_back_prop_add_one for a batch of (base code, interval)."""
    require_cuda()
    n = len(bases)
    b = torch.from_numpy(np.ascontiguousarray(bases, np.uint8)).to(index.device)
    lo_t = torch.from_numpy(np.ascontiguousarray(lo, np.uint32).view(np.int32)).to(index.device)
    cnt_t = torch.from_numpy(np.ascontiguousarray(cnt, np.uint32).view(np.int32)).to(index.device)
    capi.check(capi.lib.gsm_backsearch_add_one_batch(C.byref(index.c), n, _ptr(b), _ptr(lo_t), _ptr(cnt_t), _stream()))
    return lo_t.cpu().numpy().view(np.uint32), cnt_t.cpu().numpy().view(np.uint32)


def sa_lookup(index: DeviceIndex, rows):
    """suffix-array rows -> 1-based text positions (ExactMatch.get_positions)."""
    require_cuda()
    rows = np.ascontiguousarray(rows, np.uint32)
    if rows.size == 0:
        return np.zeros(0, np.uint32)
    r = torch.from_numpy(rows.view(np.int32)).to(index.device)
    out = torch.empty_like(r)
    capi.check(capi.lib.gsm_sa_lookup_batch(C.byref(index.c), rows.size, _ptr(r), _ptr(out), _stream()))
    return out.cpu().numpy().view(np.uint32)


def locate_hits(index: DeviceIndex, records, max_occ=500, min_len=0, hit_cap=None):
    """SMEM records (RECORD_DTYPE, e.g. SmemResult.records) -> HitResult: every record's occurrences on the reference as
    (sequence, offset), BWA's mem_collect_seeds sampling.  A record of len = qend - qstart < min_len has no hits; otherwise
    min(cnt, max_occ) of its cnt rows (max_occ = 0: all), row lo + k * (cnt // max_occ) for hit k when cnt > max_occ
    (flag HIT_SAMPLED).  HIT_SPANS flags a match that runs past the end of its sequence.  Sequences: index.contigs, else
    one sequence.  Positions from the full suffix array when resident, else from the sampled one (build_sampled_sa).
    The hits are expanded on the device in slices of at most hit_cap hits (default: all at once; never fewer than the
    largest record's count) and copied to pinned host memory slice by slice."""
    require_cuda()
    recs = np.ascontiguousarray(records).view(RECORD_DTYPE).reshape(-1)
    n_rec = len(recs)
    _validate_records(index, recs)
    dev =torch.from_numpy(recs.view(np.uint8).reshape(-1)).to(index.device) if n_rec else torch.empty(16, dtype=torch.uint8, device=index.device)
    return _expand_hits(index, dev, n_rec, max_occ, min_len, hit_cap)


def _hit_params(index, max_occ, min_len):
    if index.sa is None and getattr(index, "ssa", None) is None:
        raise ValueError("no suffix array on the device: call build_sampled_sa() before dropping it")
    max_occ, min_len = int(max_occ), int(min_len)
    if max_occ < 0 or min_len < 0:
        raise ValueError("max_occ and min_len must be >= 0")
    return max_occ, min_len


def _count_hits(index, recs, n_rec, max_occ, min_len):
    """gsm_hits_count over records on the device -> hit_off (device int64, n_rec + 1 entries) and its host copy."""
    dev = index.device
    counts = torch.empty(max(n_rec, 1), dtype=torch.int32, device=dev)
    off = torch.empty(n_rec + 1, dtype=torch.int64, device=dev)
    tmp_bytes = C.c_uint64()
    capi.check(capi.lib.gsm_hits_workspace_info(n_rec, C.byref(tmp_bytes)))
    tmp = torch.empty(max(int(tmp_bytes.value), 8), dtype=torch.uint8, device=dev)
    capi.check(capi.lib.gsm_hits_count(_ptr(recs), n_rec, max_occ, min_len, _ptr(counts), _ptr(off), _ptr(tmp), int(tmp_bytes.value), _stream()))
    return off, off.cpu().numpy()


def _locate_range(index, recs, off, a, b, max_occ, min_len, out, cap, status):
    """gsm_hits_locate: the hits of records [a, b) to out (device, cap hits)."""
    ssa = getattr(index, "ssa", None)
    contigs = C.byref(index._contigs_c) if index.contigs is not None else None
    ssa_p, sample = (_ptr(ssa), int(index.sa_sample)) if ssa is not None else (C.c_void_p(0), 0)
    capi.check(capi.lib.gsm_hits_locate(C.byref(index.c), ssa_p, sample, contigs, _ptr(recs), _ptr(off), a, b, max_occ, min_len,
                                        _ptr(out), cap, _ptr(status), _stream()))


def _expand_hits(index, recs, n_rec, max_occ, min_len, hit_cap):
    """gsm_hits_count + gsm_hits_locate over records already on the device (recs: uint8 tensor, n_rec x 16 bytes)."""
    max_occ, min_len = _hit_params(index, max_occ, min_len)
    with torch.cuda.device(index.device):
        dev = index.device
        off, offsets = _count_hits(index, recs, n_rec, max_occ, min_len)
        total = int(offsets[-1])
        if total == 0:
            return HitResult(np.zeros(0, HIT_DTYPE), offsets)
        cap = total if hit_cap is None else max(int(hit_cap), int(np.diff(offsets).max()))
        cap = min(cap, total)
        out = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
        status = torch.zeros(1, dtype=torch.int64, device=dev)
        host = torch.empty(total * 16, dtype=torch.uint8, pin_memory=True)
        a = 0
        while a < n_rec:
            # records [a, b): as many as fit in cap hits (one at least)
            b = max(int(np.searchsorted(offsets, offsets[a] + cap, side="right")) - 1, a + 1)
            b = min(b, n_rec)
            h0, h1 = int(offsets[a]), int(offsets[b])
            if h1 > h0:
                _locate_range(index, recs, off, a, b, max_occ, min_len, out, cap, status)
                host[h0 * 16:h1 * 16].copy_(out[:(h1 - h0) * 16], non_blocking=True)
            a = b
        torch.cuda.current_stream().synchronize()
        if int(status.item()) != 0:
            raise capi.GsmError(capi.E_CAPACITY, "gsm_hits_locate: hit buffer overflow")
    return HitResult(host.numpy().view(HIT_DTYPE), offsets)


def _device_hits(index, recs, n_rec, max_occ, min_len):
    """Every hit of records on the device, left on the device: -> (hit_off device, its host copy, hits uint8 tensor of
    total x 16 bytes, total)."""
    off, offsets = _count_hits(index, recs, n_rec, max_occ, min_len)
    total = int(offsets[-1])
    hits = torch.empty(max(total, 1) * 16, dtype=torch.uint8, device=index.device)
    if total:
        status = torch.zeros(1, dtype=torch.int64, device=index.device)
        _locate_range(index, recs, off, 0, n_rec, max_occ, min_len, hits, total, status)
    return off, offsets, hits, total


def _validate_records(index, recs):
    if len(recs) and int((recs["sa_hi"][recs["sa_hi"] >= recs["sa_lo"]]).max(initial=0)) >= index.n_rows:
        raise ValueError("a record's interval lies outside the index")


def _chain_params(w, max_gap):
    w, max_gap = int(w), int(max_gap)
    if not (0 <= w < 1 << 32 and 0 <= max_gap < 1 << 32):
        raise ValueError("w and max_gap must be in [0, 2^32)")
    return w, max_gap


def _chain(index, recs, n_rec, rec_off, rec_offsets, max_occ, min_len, w, max_gap, strands, lengths):
    """Hits of the records on the device (never copied to the host in between), chained per slot (gsm_chain_seeds +
    gsm_chains_collect); recs: uint8 tensor (n_rec x 16 bytes), rec_off: device int64 per slot, rec_offsets: its host copy."""
    max_occ, min_len = _hit_params(index, max_occ, min_len)
    w, max_gap = _chain_params(w, max_gap)
    n_slots = len(rec_offsets) - 1
    dev = index.device
    with torch.cuda.device(dev):
        off, offsets, hits, total = _device_hits(index, recs, n_rec, max_occ, min_len)
        hit_chain = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        cnt = torch.empty(max(n_slots, 1), dtype=torch.int32, device=dev)
        coff = torch.empty(n_slots + 1, dtype=torch.int64, device=dev)
        need = C.c_uint64()
        capi.check(capi.lib.gsm_chains_workspace_info(n_slots, total, C.byref(need)))
        ws = torch.empty(max(int(need.value), 8), dtype=torch.uint8, device=dev)
        capi.check(capi.lib.gsm_chain_seeds(_ptr(recs), _ptr(rec_off), n_slots, _ptr(hits), _ptr(off), total, w, max_gap, _ptr(hit_chain), _ptr(cnt),
                                            _ptr(coff), _ptr(ws), int(need.value), _stream()))
        chain_off = coff.cpu().numpy()
        n_ch = int(chain_off[-1])
        out = torch.empty(max(n_ch, 1) * 32, dtype=torch.uint8, device=dev)
        status = torch.zeros(1, dtype=torch.int64, device=dev)
        capi.check(capi.lib.gsm_chains_collect(_ptr(rec_off), n_slots, _ptr(off), total, _ptr(coff), _ptr(ws), int(need.value), _ptr(out), n_ch,
                                               _ptr(status), _stream()))
        h_chains = torch.empty(n_ch * 32, dtype=torch.uint8, pin_memory=True)
        h_hits = torch.empty(total * 16, dtype=torch.uint8, pin_memory=True)
        h_ids = torch.empty(total, dtype=torch.int32, pin_memory=True)
        h_chains.copy_(out[:n_ch * 32], non_blocking=True)
        h_hits.copy_(hits[:total * 16], non_blocking=True)
        h_ids.copy_(hit_chain[:total], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        if int(status.item()) != 0:
            raise capi.GsmError(capi.E_CAPACITY, "gsm_chains_collect: chain buffer overflow")
    hr = HitResult(h_hits.numpy().view(HIT_DTYPE), offsets)
    return ChainResult(h_chains.numpy().view(CHAIN_DTYPE), chain_off, hr, h_ids.numpy().view(np.uint32), rec_offsets, strands, lengths)


def chain_seeds(index: DeviceIndex, result, max_occ=500, min_len=19, w=100, max_gap=10000):
    """BWA-MEM's seed chaining (mem_chain) of every slot of an SmemResult (Engine.run, PipelinedEngine.run*): its records
    are expanded into hits on the device (locate_hits with max_occ / min_len, BWA's -c and -k), and each slot's hits -- in
    record order, then suffix-array row order -- are grouped into co-linear chains on one sequence (test_and_merge with band
    w and max_gap, BWA's -w and max_chain_gap; hits that span two sequences are skipped).  A slot's chains are ordered by
    (contig, rbeg of the first seed), ties in creation order; `lower` among tied chains is the one created first.  Only the
    chains, the hits and their chain ids come back to the host -> ChainResult."""
    require_cuda()
    recs = np.ascontiguousarray(result.records).view(RECORD_DTYPE).reshape(-1)
    _validate_records(index, recs)
    rec_offsets = np.ascontiguousarray(result.offsets, np.int64)
    if len(rec_offsets) < 1 or rec_offsets[0] != 0 or rec_offsets[-1] != len(recs) or (np.diff(rec_offsets) < 0).any():
        raise ValueError("result.offsets must rise from 0 to the number of records")
    if result.strands == 2 and result.lengths is None:
        raise ValueError("a strands=2 result needs its read lengths")
    n_rec = len(recs)
    with torch.cuda.device(index.device):
        dev = torch.from_numpy(recs.view(np.uint8).reshape(-1)).to(index.device) if n_rec else torch.empty(16, dtype=torch.uint8, device=index.device)
        rec_off = torch.from_numpy(rec_offsets).to(index.device)
        return _chain(index, dev, n_rec, rec_off, rec_offsets, max_occ, min_len, w, max_gap, result.strands,
                      None if result.lengths is None else np.asarray(result.lengths, np.uint32).copy())


def set_rmi_prefilter(on=True):
    """RMI-SMEM selection: True (default) = reads without a hazard window take their records from the BWA-SMEM selection when
    the model carries a hazard filter (RmiParams.build_hazard_filter); False = every read runs the reference's frame machine
    (k_select_seeded<RMI>, the cross-check: same records).  Process-wide (gsm_option_rmi_prefilter); returns the previous
    setting."""
    return bool(capi.lib.gsm_option_rmi_prefilter(1 if on else 0))


def set_lut_frame_machine(on=True):
    """LUT-SMEM selection: False (default) = the records are the sweep's picks (get_smems_lut emits exactly get_SMEMS's
    records with min_len 1 for reads of at least K bases); True = run the reference's frame machine itself
    (k_select_seeded<LUT>, the cross-check: same records).  Process-wide (gsm_option_lut_frame_machine); returns the
    previous setting."""
    return bool(capi.lib.gsm_option_lut_frame_machine(1 if on else 0))


def lut_build(index: DeviceIndex, K):
    """Dense device table (4^K x {lo, cnt}); replaces LUT.generate_lut (reference SMEM/LUT.py:15-35)."""
    require_cuda()
    t = torch.empty((1 << (2 * K)) * 2, dtype=torch.int32, device=index.device)
    capi.check(capi.lib.gsm_lut_build(C.byref(index.c), int(K), _ptr(t), _stream()))
    return t


def rmi_lookup_batch(index: DeviceIndex, rmi: RmiParams, codes):
    """get_suffix_rmi for a batch of k-mer codes -> (pred f64, lo i64, hi i64, status u8)."""
    require_cuda()
    codes = np.ascontiguousarray(codes, np.uint64)
    n = codes.size
    dev = index.device
    c = torch.from_numpy(codes.view(np.int64)).to(dev)
    pred = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
    lo = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    hi = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    st = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
    capi.check(capi.lib.gsm_rmi_lookup_batch(C.byref(index.c), C.byref(rmi.c), n, _ptr(c), _ptr(pred), _ptr(lo), _ptr(hi), _ptr(st), _stream()))
    return pred[:n].cpu().numpy(), lo[:n].cpu().numpy(), hi[:n].cpu().numpy(), st[:n].cpu().numpy()


def gather_probe(buf: torch.Tensor, n_fetch, dependent):
    """Random aligned 64-byte gather over `buf`; returns (#fetches, seconds) timed with CUDA events."""
    require_cuda()
    sink = torch.zeros(1, dtype=torch.int64, device=buf.device)
    done = C.c_uint64()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nbytes = buf.numel() * buf.element_size()
    capi.check(capi.lib.gsm_gather_probe(_ptr(buf), nbytes, max(n_fetch // 8, 1), int(dependent), _ptr(sink), C.byref(done), _stream()))
    torch.cuda.synchronize()
    e0.record()
    capi.check(capi.lib.gsm_gather_probe(_ptr(buf), nbytes, int(n_fetch), int(dependent), _ptr(sink), C.byref(done), _stream()))
    e1.record()
    torch.cuda.synchronize()
    return int(done.value), e0.elapsed_time(e1) * 1e-3


def gather_probe2(buf: torch.Tensor, n_fetch, fetch_bytes=64, in_flight=4):
    """Random gather ceiling with the kernels' access shapes (gsm_gather_probe2); returns (#fetches, seconds)."""
    require_cuda()
    sink = torch.zeros(1, dtype=torch.int64, device=buf.device)
    done = C.c_uint64()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nbytes = buf.numel() * buf.element_size()
    capi.check(capi.lib.gsm_gather_probe2(_ptr(buf), nbytes, max(n_fetch // 8, 1), int(fetch_bytes), int(in_flight), _ptr(sink), C.byref(done), _stream()))
    torch.cuda.synchronize()
    e0.record()
    capi.check(capi.lib.gsm_gather_probe2(_ptr(buf), nbytes, int(n_fetch), int(fetch_bytes), int(in_flight), _ptr(sink), C.byref(done), _stream()))
    e1.record()
    torch.cuda.synchronize()
    return int(done.value), e0.elapsed_time(e1) * 1e-3


# ---------------------------------------------------------------------------- pipelined end-to-end path
class _ReadView:
    """Reads [lo, hi) of a ReadBatch whose buffers are (being) copied to the device."""

    def __init__(self, parent, lo, hi):
        self.p, self.lo, self.hi = parent, lo, hi
        self.n = hi - lo
        self.max_len = parent.max_len
        self.read_id_base = parent.read_id_base + lo

    def cstruct(self):
        r = capi.DevReads()
        r.n_reads = self.n
        r.packed = self.p.packed.data_ptr()
        r.chunk_off = self.p.chunk_off.data_ptr() + 4 * self.lo
        r.len = self.p.len.data_ptr() + 4 * self.lo
        r.max_len, r.read_id_base = self.max_len, self.read_id_base
        return r


class _ChunkView:
    """One self-contained chunk of reads on the device (its own packed buffer, offsets and lengths)."""

    def __init__(self, packed, chunk_off, lens, n, max_len, read_id_base, lo):
        self.packed, self.chunk_off, self.len = packed, chunk_off, lens
        self.n, self.max_len, self.read_id_base = int(n), int(max_len), int(read_id_base)
        self.lo, self.hi = int(lo), int(lo) + int(n)

    def cstruct(self):
        r = capi.DevReads()
        r.n_reads = self.n
        r.packed, r.chunk_off, r.len = self.packed.data_ptr(), self.chunk_off.data_ptr(), self.len.data_ptr()
        r.max_len, r.read_id_base = self.max_len, self.read_id_base
        return r


class PipelinedEngine:
    """Host reads in, host records out, with the PCIe copies hidden behind the kernels.  The batch is cut into
    chunks; three CUDA streams run concurrently:
      copy-in   every chunk's H2D is queued up front (the device input buffers hold the whole batch),
      compute   [2-bit packing,] sweep, select, scan, gather of chunk i, in order, alternating between two workspaces,
      copy-out  records / offsets / status of chunk i to pinned host memory as soon as its record count is known.
    The compute stream only waits for chunk i's H2D and for the D2H that frees its workspace (chunk i-2), so neither
    copy direction ever sits between two sweeps.  Inputs must be pinned.

    strands = 2: every chunk is strand-doubled on the compute stream right after packing (Engine strands=2: each workspace
    holds 2 * chunk_reads slots and its own doubled-batch buffers), and the result is per slot (SmemResult.strands = 2)."""

    def __init__(self, index: DeviceIndex, max_reads, max_len, n_chunks=8, mems_per_read=24, recs_per_read=16, strands=1):
        require_cuda()
        if strands not in (1, 2):
            raise ValueError("strands must be 1 or 2")
        self.index, self.device = index, index.device
        self.strands = int(strands)
        self.n_chunks = max(2, int(n_chunks))
        self.chunk_reads = (int(max_reads) + self.n_chunks - 1) // self.n_chunks
        self.engines = [Engine(index, self.chunk_reads, max_len, mems_per_read, recs_per_read, self.strands) for _ in range(2)]
        self.s_in, self.s_comp, self.s_out = (torch.cuda.Stream(device=self.device) for _ in range(3))
        self.max_reads, self.max_len = int(max_reads), int(max_len)
        self._dev = {}
        self._pin = {}
        self._cnt_pin = [torch.zeros(8, dtype=torch.int64).pin_memory() for _ in range(2)]
        self.last_d2h_bytes = 0
        self.last_h2d_bytes = 0
        self.kernel_launches = 0
        self.pack_launches = 0

    def _buf(self, store, name, nbytes, pinned):
        b = store.get(name)
        if b is None or b.numel() < nbytes:
            b = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, device="cpu" if pinned else self.device)
            if pinned:
                b = b.pin_memory()
            store[name] = b
        return b

    def _chunk_bounds(self, n):
        """Chunk boundaries: full chunks of chunk_reads in the middle, a geometric ramp (1/8, 1/8, 1/4, 1/2) at both ends,
        because the first chunk's H2D and the last chunk's D2H are the only copies nothing can hide (chunks of a million
        reads and more; smaller ones are equal)."""
        c = self.chunk_reads
        ramp = [max(c // 8, 1), max(c // 8, 1), max(c // 4, 1), max(c // 2, 1)]
        # small chunks (a batch sharded over many GPUs) are launch-latency bound already: no ramp below 1 M reads per chunk
        if n <= 4 * c or c < 1_000_000:
            return sorted(set(min(n, i * c) for i in range((n + c - 1) // c + 1))) if n else [0]
        head, pos = [0], 0
        for r in ramp:
            pos += r
            head.append(pos)
        tail, end = [n], n
        for r in ramp:
            end -= r
            tail.append(end)
        tail.reverse()
        mid = list(range(head[-1] + c, tail[0], c))
        return head + mid + tail

    def run(self, method, reads: ReadBatch, min_len=1, K=0, lut=None, rmi: RmiParams = None, reuse_host_buffers=False, gatherer=None):
        """Packed host reads in (pinned), host records out -- or, with a sharding.RecordGatherer, records written straight
        into the gathering rank's HBM (the result then carries offsets and status only)."""
        self._check_gatherer(gatherer)
        n = reads.n
        if n > self.max_reads or reads.max_len > self.max_len:
            raise ValueError("batch exceeds the engine's workspace")
        hp = torch.from_numpy(reads.packed_host)
        hco = torch.from_numpy(reads.chunk_off_host.view(np.int32))
        hln = torch.from_numpy(reads.len_host.view(np.int32))
        reads.packed = self._buf(self._dev, "packed", hp.numel(), False)[: hp.numel()]
        reads.chunk_off = self._buf(self._dev, "coff", hco.numel() * 4, False)[: hco.numel() * 4].view(torch.int32)
        reads.len = self._buf(self._dev, "len", max(hln.numel(), 1) * 4, False)[: hln.numel() * 4].view(torch.int32)
        co = reads.chunk_off_host

        def copy_in(lo, hi):
            b0, b1 = int(co[lo]) * 16, int(co[hi]) * 16 + 16
            reads.packed[b0:b1].copy_(hp[b0:b1], non_blocking=True)
            reads.chunk_off[lo:hi + 1].copy_(hco[lo:hi + 1], non_blocking=True)
            reads.len[lo:hi].copy_(hln[lo:hi], non_blocking=True)

        self.last_h2d_bytes = reads.h2d_bytes()
        res = self._run_chunks(method, n, copy_in, lambda lo, hi: _ReadView(reads, lo, hi), min_len, K, lut, rmi, gatherer)
        return res if reuse_host_buffers else res.detach()

    def run_ascii(self, method, bases, read_len, min_len=1, K=0, lut=None, rmi: RmiParams = None, read_id_base=0, reuse_host_buffers=False,
                  gatherer=None):
        """RAW read bytes in, host records out: `bases` is a pinned uint8 tensor of n x read_len ASCII characters
        (what a FASTQ parser hands over).  Each chunk crosses PCIe as 1 byte/base and is 2-bit packed on the GPU
        (gsm_pack_reads_device) right before its sweep.  Raises BaseError if a read holds a non-ACGT character
        (the reference's KeyError, ExactMatch.py:139)."""
        self._check_gatherer(gatherer)
        read_len = int(read_len)
        n = bases.numel() // read_len
        if n > self.max_reads or read_len > self.max_len:
            raise ValueError("batch exceeds the engine's workspace")
        flat = bases.view(-1)
        cpr = (read_len + 63) // 64
        key = (cpr, n)
        if self._dev.get("coff_key") != key:                 # chunk offsets of a fixed-length batch are arithmetic: built once
            self._dev["coff_fixed"] = (torch.arange(n + 1, dtype=torch.int64, device=self.device) * cpr).to(torch.int32)
            self._dev["coff_key"] = key
        coff = self._dev["coff_fixed"]
        packed = self._buf(self._dev, "packed", n * cpr * 16 + 16, False)
        lens = self._buf(self._dev, "len", max(n, 1) * 4, False)[: n * 4].view(torch.int32)
        raw = self._buf(self._dev, "raw", max(n * read_len, 1), False)
        n_slots = len(self._chunk_bounds(n))
        bad = self._buf(self._dev, "bad", 8 * n_slots, False)[: 8 * n_slots].view(torch.int64)
        slot = {}
        holder = ReadBatch(None, None, np.zeros(0, np.uint32), read_len, read_id_base)
        holder.n, holder.packed, holder.chunk_off, holder.len = n, packed, coff, lens

        def copy_in(lo, hi):
            raw[lo * read_len: hi * read_len].copy_(flat[lo * read_len: hi * read_len], non_blocking=True)

        def prep(lo, hi):
            capi.check(capi.lib.gsm_pack_reads_device(C.c_void_p(raw.data_ptr() + lo * read_len), None, read_len, C.c_void_p(coff.data_ptr() + 4 * lo),
                                                      hi - lo, 1, _ptr(packed), C.c_void_p(lens.data_ptr() + 4 * lo),
                                                      C.c_void_p(bad.data_ptr() + 8 * len(slot)), _stream()))
            slot[len(slot)] = lo
            self.pack_launches += 1
            return _ReadView(holder, lo, hi)

        self.last_h2d_bytes = n * read_len
        res = self._run_chunks(method, n, copy_in, prep, min_len, K, lut, rmi, gatherer)
        b = bad.cpu().numpy()[: len(slot)]
        if (b != -1).any():
            k = int(np.nonzero(b != -1)[0][0])
            raise BaseError(f"non-ACGT base in read {slot[k] + int(b[k])}")
        return res if reuse_host_buffers else res.detach()

    def run_fastq(self, method, fq, min_len=1, K=0, lut=None, rmi: RmiParams = None, read_id_base=0, reuse_host_buffers=False, n_chunks=None):
        """FASTQ FILE BYTES in (a pinned uint8 tensor holding a 4-line FASTQ), host records out.  The host only looks for
        a record boundary near each chunk cut (ingest.fastq_cuts: a few hundred bytes per cut); every chunk crosses PCIe
        as raw file bytes and is cut into records and 2-bit packed ON THE GPU (gsm_fastq_count_device /
        gsm_fastq_records_device / gsm_pack_reads_scattered_device) on the copy-in stream, ahead of the sweeps.  Read
        lengths may differ.  Raises BaseError for a non-ACGT base (ExactMatch.py:139), ValueError for a malformed file."""
        from . import ingest
        fq = fq.view(-1)
        nb_total = int(fq.numel())
        n_ch = int(n_chunks or 2 * self.n_chunks)
        cuts = ingest.fastq_cuts(fq.numpy(), n_ch)
        n_ch = len(cuts) - 1
        TILE = 16384
        cap = self.chunk_reads
        chunks = [None] * n_ch
        stats_pin = self._buf(self._pin, "fq_stats", 8 * 8 * max(n_ch, 1), True)[: 64 * n_ch].view(torch.int64).view(n_ch, 8)
        ev_parse = [None] * n_ch

        def copy_in(i):
            c0, c1 = cuts[i], cuts[i + 1]
            nb = c1 - c0
            raw = torch.empty(nb + 16, dtype=torch.uint8, device=self.device)
            raw[:nb].copy_(fq[c0:c1], non_blocking=True)
            tiles = (nb + TILE - 1) // TILE
            cnt = torch.empty(max(tiles, 1), dtype=torch.int32, device=self.device)
            capi.check(capi.lib.gsm_fastq_count_device(_ptr(raw), nb, _ptr(cnt), _stream()))
            incl = torch.cumsum(cnt[:tiles].to(torch.int64), 0)
            prefix = (incl - cnt[:tiles]).contiguous()
            seq_start = torch.zeros(cap, dtype=torch.int64, device=self.device)
            seq_end = torch.zeros(cap, dtype=torch.int64, device=self.device)
            flags = torch.empty(2, dtype=torch.int64, device=self.device)          # [0] structure error offset, [1] first bad read
            capi.check(capi.lib.gsm_fastq_records_device(_ptr(raw), nb, _ptr(prefix), cap, _ptr(seq_start), _ptr(seq_end), _ptr(flags), _stream()))
            # a record counts only if both ends of its sequence line were seen (a truncated file leaves the last one open);
            # anything else packs as an empty read, so no length derived from the input can send the packer out of bounds
            whole = (seq_start > 0) & (seq_end >= seq_start) & (seq_end <= nb)
            lens = torch.where(whole, seq_end - seq_start, torch.zeros_like(seq_end)).to(torch.int32)
            coff = torch.zeros(cap + 1, dtype=torch.int32, device=self.device)
            coff[1:] = torch.cumsum((lens + 63) // 64, 0).to(torch.int32)
            packed = torch.empty(nb // 4 + 16 * cap + 32, dtype=torch.uint8, device=self.device)
            capi.check(capi.lib.gsm_pack_reads_scattered_device(_ptr(raw), _ptr(seq_start), _ptr(lens), _ptr(coff), cap, 1, _ptr(packed),
                                                                C.c_void_p(flags.data_ptr() + 8), _stream()))
            st = torch.stack([incl[-1] if tiles else incl.new_zeros(()), lens.max().to(torch.int64), flags[0], flags[1],
                              coff[-1].to(torch.int64)])
            stats_pin[i, :5].copy_(st, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            ev_parse[i] = ev
            chunks[i] = (packed, coff, lens, raw)
            self.pack_launches += 3

        seen = [0]

        def prep(i):
            ev_parse[i].synchronize()
            n_nl, max_len, err, bad, _ = (int(x) for x in stats_pin[i, :5])
            c0, c1 = cuts[i], cuts[i + 1]
            n_lines = n_nl + (0 if c1 == c0 or int(fq[c1 - 1]) == 10 else 1)
            if err != -1:
                raise ValueError(f"malformed FASTQ near byte {c0 + err}: a record must start with '@' and its third line with '+'")
            if n_lines % 4:
                raise ValueError(f"truncated FASTQ: {n_lines} lines in the chunk starting at byte {c0}")
            n_i = n_lines // 4
            if n_i > cap:
                raise capi.GsmError(capi.E_CAPACITY, f"a FASTQ chunk holds {n_i} reads, more than the engine's chunk capacity {cap}: raise n_chunks")
            if bad != -1 and bad < n_i:
                raise BaseError(f"non-ACGT base in read {seen[0] + bad}")
            if max_len > self.max_len:
                raise ValueError(f"a read of {max_len} bases exceeds the engine's max_len {self.max_len}")
            packed, coff, lens, _raw = chunks[i]
            v = _ChunkView(packed, coff, lens, n_i, self.max_len, read_id_base + seen[0], seen[0])
            seen[0] += n_i
            return v

        self.last_h2d_bytes = nb_total
        res = self._run_chunks(method, self.max_reads, copy_in, prep, min_len, K, lut, rmi, None, dynamic_chunks=n_ch)
        return res if reuse_host_buffers else res.detach()

    def _check_gatherer(self, gatherer):
        if gatherer is not None and self.strands == 2:
            raise ValueError("strands=2 does not support a gatherer")

    def _run_chunks(self, method, n, copy_in, prep, min_len, K, lut, rmi, gatherer=None, dynamic_chunks=0):
        """dynamic_chunks = 0: the batch of n reads is cut by _chunk_bounds; copy_in(lo, hi) / prep(lo, hi) take read ranges.
        dynamic_chunks = k: k chunks whose read counts are only known once they are prepared (FASTQ bytes): copy_in(i) /
        prep(i) take the chunk index, prep's view carries .lo / .hi, and n is the capacity the outputs are sized for.
        With strands = 2 each prepared chunk is strand-doubled and everything downstream is in slot space (2 lo .. 2 hi)."""
        if dynamic_chunks:
            bounds, n_ch = None, int(dynamic_chunks)
        else:
            bounds = self._chunk_bounds(n)
            n_ch = len(bounds) - 1
        ns = self.strands
        n_cap = n * ns                                          # slots the outputs are sized for
        est = self.engines[0].rec_cap * 16
        out_rec = self._buf(self._pin, "rec", max(est, 1 << 20), True)
        out_off = self._buf(self._pin, "off", (n_cap + 1) * 8, True)
        out_st = self._buf(self._pin, "st", max(n_cap, 1), True)
        out_len = self._buf(self._pin, "len", max(n_cap, 1) * 4, True) if ns == 2 else None
        start_ev = torch.cuda.Event()
        start_ev.record(torch.cuda.current_stream())
        ev_in = []
        with torch.cuda.stream(self.s_in):                     # every chunk's H2D, queued up front
            self.s_in.wait_event(start_ev)
            for i in range(n_ch):
                if dynamic_chunks:
                    copy_in(i)
                else:
                    copy_in(bounds[i], bounds[i + 1])
                ev = torch.cuda.Event()
                ev.record(self.s_in)
                ev_in.append(ev)
        self.s_comp.wait_event(start_ev)
        self.s_out.wait_event(start_ev)
        pending = []      # (engine idx, lo, hi, compute-done event)
        ev_out = {}       # chunk index -> its D2H-done event
        rec_total = 0
        mems_total = 0
        chunk_rec = []

        def drain(item):
            nonlocal rec_total, mems_total, out_rec
            i, e, lo, hi, ev = item
            ev.synchronize()
            c = self._cnt_pin[e].numpy()
            if c[2] != 0:
                raise capi.GsmError(capi.E_CAPACITY, f"workspace overflow in chunk [{lo},{hi}): mems {int(c[0])}, records {int(c[1])}; "
                                                     "raise mems_per_read / recs_per_read")
            n_rec = int(c[1])
            mems_total += int(c[0])
            if (rec_total + n_rec) * 16 > out_rec.numel():
                grown = torch.empty(max((rec_total + n_rec) * 32, out_rec.numel() * 2), dtype=torch.uint8).pin_memory()
                torch.cuda.synchronize()
                grown[: rec_total * 16] = out_rec[: rec_total * 16]
                out_rec = grown
                self._pin["rec"] = grown
            eng = self.engines[e]
            with torch.cuda.stream(self.s_out):                # the host has seen ev: the chunk's kernels are done
                if gatherer is None:
                    out_rec[rec_total * 16:(rec_total + n_rec) * 16].copy_(eng.records[: n_rec * 16], non_blocking=True)
                if rec_total:                                  # chunk-local offsets -> global offsets, on the device
                    eng.rec_off[: hi - lo].add_(rec_total)
                out_off[lo * 8:hi * 8].copy_(eng.rec_off[: hi - lo].view(torch.uint8), non_blocking=True)
                out_st[lo:hi].copy_(eng.read_status[: hi - lo], non_blocking=True)
                if out_len is not None:
                    out_len[lo * 4:hi * 4].copy_(eng.ds_len[: hi - lo].view(torch.uint8), non_blocking=True)
                d = torch.cuda.Event()
                d.record(self.s_out)
                ev_out[i] = d
            chunk_rec.append((lo, hi, rec_total, n_rec))
            rec_total += n_rec

        n_seen = 0
        for i in range(n_ch):
            e = i % 2
            if len(pending) == 2:                 # workspace e still holds chunk i-2: drain it (count -> D2H) first
                drain(pending.pop(0))
            eng = self.engines[e]
            with torch.cuda.stream(self.s_comp):
                self.s_comp.wait_event(ev_in[i])
                if i - 2 in ev_out:
                    self.s_comp.wait_event(ev_out[i - 2])
                if dynamic_chunks:
                    view = prep(i)
                    lo, hi = view.lo, view.hi
                    if hi > n:
                        raise capi.GsmError(capi.E_CAPACITY, f"the input holds more than the engine's {n} reads")
                else:
                    lo, hi = bounds[i], bounds[i + 1]
                    view = prep(lo, hi)
                if ns == 2:
                    view = eng._both_strands(view)
                    lo, hi = 2 * lo, 2 * hi
                n_seen = max(n_seen, hi)
                eng.launch(method, view, min_len, K, lut, rmi, gatherer)
                self._cnt_pin[e].copy_(eng.counters, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.s_comp)
            pending.append((i, e, lo, hi, ev))
        while pending:
            drain(pending.pop(0))
        self.s_out.synchronize()
        self.s_comp.synchronize()
        torch.cuda.current_stream().wait_stream(self.s_out)
        n = n_seen if dynamic_chunks else n_cap                 # slots
        offs = out_off.numpy()[: (n + 1) * 8].view(np.int64)
        offs[n] = rec_total
        self.kernel_launches = sum(e.kernel_launches for e in self.engines) + self.pack_launches
        self.last_d2h_bytes = (rec_total * 16 if gatherer is None else 0) + (n + 1) * 8 + n + 64 * len(chunk_rec)
        recs = out_rec.numpy()[: (rec_total if gatherer is None else 0) * 16].view(RECORD_DTYPE)
        lengths = None
        if out_len is not None:
            lengths = out_len.numpy()[: n * 4].view(np.uint32)[0::2]
            self.last_d2h_bytes += n * 4
        return SmemResult(recs, offs, out_st.numpy()[:n], mems_total, ns, lengths)
