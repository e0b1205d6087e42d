"""B200-native SMEM-seeding engine: a drop-in for GENIE-SMEM's search path.

Importing this package loads libgenie_smem.so (built in-tree by genie_smem_b200/build.py with
nvcc for sm_100a).  There is no CPU fallback: without the library the import fails, without a
GPU every search call raises.
"""
from . import _capi  # noqa: F401  (fails loudly when the CUDA library is missing)
from .engine import (BaseError, CHAIN_DTYPE, ChainResult, DeviceIndex, Engine, HIT_DTYPE, HitResult, HostIndex, IndexFile, PackedIndex, PipelinedEngine, ReadBatch, RmiParams,  # noqa: F401
                     RECORD_DTYPE, SmemResult, add_one_batch, backsearch_batch, chain_seeds, gather_probe, gather_probe2, l2_fetch_granularity, lut_build, rmi_lookup_batch, locate_hits, sa_lookup, set_lut_frame_machine, set_rmi_prefilter)
from .ingest import Contigs, read_fasta, read_fastq, read_reference, write_fastq  # noqa: F401
from .surface import (ExactMatch, LUT, RMI, RMI_LUT, SMEM, create_query_from_ref, create_random_query)  # noqa: F401
from ._capi import CHAIN_CONTAINED, CHAIN_NONE, HIT_SAMPLED, HIT_SPANS, METHOD_BWA, METHOD_LUT, METHOD_RMI, READ_OK, READ_REF_RAISES, READ_TOO_SHORT, GsmError  # noqa: F401

__version__ = "0.1.0"
