"""ctypes bindings of libgenie_smem.so (include/genie_smem.h).  Thin: no logic lives here.

The library is built in-tree by genie_smem_b200/build.py (nvcc, sm_100a) and must be present:
there is no CPU fallback for any search routine -- a missing library is an ImportError, a missing
GPU is GSM_E_NODEVICE from every device entry point.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgenie_smem.so")

OK, E_INVALID, E_NOMEM, E_CUDA, E_CAPACITY, E_NODEVICE = 0, -1, -2, -3, -4, -5
METHOD_BWA, METHOD_LUT, METHOD_RMI = 0, 1, 2
READ_OK, READ_REF_RAISES, READ_TOO_SHORT = 0, 1, 2

u8p, u32p, u64p, i64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_int64, C.c_double))


class IndexInfo(C.Structure):
    _fields_ = [("n_bases", C.c_uint64), ("n_rows", C.c_uint64), ("n_buckets", C.c_uint64), ("bucket_bytes", C.c_uint64),
                ("text_words", C.c_uint64), ("count", C.c_uint32 * 4), ("C", C.c_uint32 * 5), ("primary_fwd", C.c_uint32),
                ("primary_rev", C.c_uint32), ("has_reverse", C.c_uint32), ("reserved", C.c_uint32)]


class DevIndex(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_buckets", C.c_uint64), ("fwd_buckets", C.c_void_p), ("rev_buckets", C.c_void_p),
                ("sa", C.c_void_p), ("text2bit", C.c_void_p), ("C", C.c_uint32 * 5), ("primary_fwd", C.c_uint32),
                ("primary_rev", C.c_uint32), ("seed_K", C.c_uint32), ("seed_table", C.c_void_p)]


class DevReads(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("packed", C.c_void_p), ("chunk_off", C.c_void_p), ("len", C.c_void_p),
                ("max_len", C.c_uint32), ("read_id_base", C.c_uint32)]


class DevRmi(C.Structure):
    _fields_ = [("K", C.c_uint32), ("n_levels", C.c_uint32), ("level_sizes", u32p), ("coef", C.c_void_p), ("intercept", C.c_void_p), ("probe", C.c_void_p),
                ("none_rows", u32p), ("n_none_rows", C.c_uint32), ("param_stride", C.c_uint32), ("bounds", C.c_void_p),
                ("hazard_slots", C.c_void_p), ("hazard_n_slots", C.c_uint32), ("reserved0", C.c_uint32)]


class Workspace(C.Structure):
    _fields_ = [("mem_pool", C.c_void_p), ("mem_cap", C.c_uint64), ("quad_scratch", C.c_void_p), ("quad_scratch_bytes", C.c_uint64),
                ("mem_off", C.c_void_p), ("mem_cnt", C.c_void_p), ("rec_tmp", C.c_void_p), ("rec_cap", C.c_uint64),
                ("rec_tmp_off", C.c_void_p), ("rec_cnt", C.c_void_p), ("rec_off", C.c_void_p), ("read_status", C.c_void_p),
                ("counters", C.c_void_p), ("scan_tmp", C.c_void_p), ("scan_tmp_bytes", C.c_uint64)]


class WorkspaceInfo(C.Structure):
    _fields_ = [("quad_scratch_bytes", C.c_uint64), ("scan_tmp_bytes", C.c_uint64), ("grid_blocks", C.c_uint32), ("block_threads", C.c_uint32)]


class DevContigs(C.Structure):
    _fields_ = [("n", C.c_uint64), ("start", C.c_void_p)]


class Hit(C.Structure):
    _fields_ = [("record", C.c_uint32), ("contig", C.c_uint32), ("offset", C.c_uint32), ("flags", C.c_uint32)]


HIT_SPANS, HIT_SAMPLED = 1, 2


class Chain(C.Structure):
    _fields_ = [("slot", C.c_uint32), ("contig", C.c_uint32), ("rbeg", C.c_uint32), ("rend", C.c_uint32), ("q", C.c_uint32),
                ("weight", C.c_uint32), ("n_seeds", C.c_uint32), ("reserved", C.c_uint32)]


CHAIN_NONE, CHAIN_CONTAINED = 0xFFFFFFFF, 0x80000000

EXPORTS = {
    # name: (restype, argtypes)
    "gsm_index_build": (C.c_int, [C.c_char_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_void_p)]),
    "gsm_index_from_arrays": (C.c_int, [C.c_char_p, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "gsm_index_info_get": (C.c_int, [C.c_void_p, C.POINTER(IndexInfo)]),
    "gsm_index_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_index_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_index_free": (None, [C.c_void_p]),
    "gsm_pack_reads": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "gsm_text_pack_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_index_build_device_workspace": (C.c_int, [C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]),
    "gsm_index_build_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                         C.POINTER(IndexInfo), C.c_void_p]),
    "gsm_fastq_scan": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]),
    "gsm_fastq_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32]),
    "gsm_pack_reads_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "gsm_fastq_count_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "gsm_fastq_records_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_pack_reads_scattered_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p,
                                                  C.c_void_p]),
    "gsm_pack_reads_device_check": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gsm_reads_both_strands_device": (C.c_int, [C.POINTER(DevReads), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_smem_workspace_info": (C.c_int, [C.c_uint64, C.c_uint32, C.POINTER(WorkspaceInfo)]),
    "gsm_backsearch_batch": (C.c_int, [C.POINTER(DevIndex), C.POINTER(DevReads), C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_backsearch_add_one_batch": (C.c_int, [C.POINTER(DevIndex), C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_sa_lookup_batch": (C.c_int, [C.POINTER(DevIndex), C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_sa_sample_build": (C.c_int, [C.POINTER(DevIndex), C.c_uint32, C.c_void_p, C.c_void_p]),
    "gsm_locate_sampled_batch": (C.c_int, [C.POINTER(DevIndex), C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_lut_build": (C.c_int, [C.POINTER(DevIndex), C.c_uint32, C.c_void_p, C.c_void_p]),
    "gsm_seed_table_build": (C.c_int, [C.POINTER(DevIndex), C.c_uint32, C.c_void_p, C.c_void_p]),
    "gsm_smem_batch": (C.c_int, [C.c_int, C.POINTER(DevIndex), C.POINTER(DevReads), C.c_uint32, C.c_uint32, C.c_void_p,
                                 C.POINTER(DevRmi), C.POINTER(Workspace), C.c_void_p]),
    "gsm_smem_sweep": (C.c_int, [C.POINTER(DevIndex), C.POINTER(DevReads), C.POINTER(Workspace), C.c_void_p]),
    "gsm_smem_select": (C.c_int, [C.c_int, C.POINTER(DevIndex), C.POINTER(DevReads), C.c_uint32, C.c_uint32, C.c_void_p,
                                  C.POINTER(DevRmi), C.POINTER(Workspace), C.c_void_p]),
    "gsm_smem_collect": (C.c_int, [C.POINTER(DevReads), C.POINTER(Workspace), C.c_void_p, C.c_uint64, C.c_void_p]),
    "gsm_rmi_probe_build": (C.c_int, [C.POINTER(DevIndex), C.c_void_p, C.c_void_p]),
    "gsm_rmi_bounds_build": (C.c_int, [C.POINTER(DevIndex), C.c_uint32, C.c_void_p, C.c_void_p]),
    "gsm_option_lut_frame_machine": (C.c_int, [C.c_int]),
    "gsm_option_rmi_prefilter": (C.c_int, [C.c_int]),
    "gsm_rmi_hazard_scan": (C.c_int, [C.POINTER(DevIndex), C.POINTER(DevRmi), C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "gsm_rmi_hazard_hash": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32]),
    "gsm_rmi_none_rows": (C.c_int, [C.POINTER(DevIndex), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_rmi_lookup_batch": (C.c_int, [C.POINTER(DevIndex), C.POINTER(DevRmi), C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_comm_unique_id": (C.c_int, [C.c_void_p]),
    "gsm_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "gsm_comm_free": (C.c_int, [C.c_void_p]),
    "gsm_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "gsm_comm_allgather_u64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "gsm_gather_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gsm_peer_export": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "gsm_peer_open": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "gsm_peer_close": (C.c_int, [C.c_void_p, C.c_uint64]),
    "gsm_smem_collect_gathered": (C.c_int, [C.POINTER(DevReads), C.POINTER(Workspace), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32,
                                            C.c_void_p, C.c_void_p]),
    "gsm_gather_advance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "gsm_gather_probe": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "gsm_gather_probe2": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "gsm_l2_persist": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p]),
    "gsm_device_l2_fetch_granularity": (C.c_int, [C.c_int32, C.POINTER(C.c_uint32)]),
    "gsm_last_error": (C.c_char_p, []),
    "gsm_version": (C.c_int, []),
    "gsm_hits_workspace_info": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint64)]),
    "gsm_hits_count": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "gsm_hits_locate": (C.c_int, [C.POINTER(DevIndex), C.c_void_p, C.c_uint32, C.POINTER(DevContigs), C.c_void_p, C.c_void_p, C.c_uint64,
                                  C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "gsm_chains_workspace_info": (C.c_int, [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]),
    "gsm_chain_seeds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "gsm_chains_collect": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                     C.c_void_p, C.c_void_p]),
}


class GsmError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libgenie_smem error {code}: {text}")
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -m genie_smem_b200.build` (nvcc, sm_100a). "
                          "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(status):
    if status != OK:
        text = lib.gsm_last_error().decode(errors="replace")
        if status == E_INVALID:
            raise ValueError(text)
        raise GsmError(status, text)
