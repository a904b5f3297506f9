"""nafcodec_b200 -- B200-native backend for the nafcodec decode hot path (zstd NAF sections -> per-record ASCII).

Surface mirrors `nafcodec` (Rust crate) / `nafcodec` (Python binding) for the decode path:
Decoder, DecoderBuilder, Record, Header, Flag, Flags, SequenceType, FormatVersion, open.
The compute runs in hand-written sm_100a kernels behind the C ABI of include/nafgpu.h; there is no CPU fallback.
"""
from .data import Flag, Flags, FormatVersion, Header, Record, SequenceType
from .decoder import (ArchiveResult, Context, Decoder, DecoderBuilder, Pipeline, decode_batch, parse_archive, shared_context,
                      to_fasta, to_fastq, to_text)
from .device import TABLES, DeviceRecords, DeviceStream, decode_to_device, stream_to_device
from .encoder import Encoder, pack_sequences
from .errors import NafArgumentError, NafDeviceError, NafError, NafIoError, NafParseError, NafUnicodeError

__version__ = "0.1.0"


def open(file, mode="r", **options):
    """nafcodec.open (nafcodec-py/nafcodec/lib.rs:641-653): 'r' -> Decoder, 'w' -> Encoder."""
    if mode == "r":
        return Decoder(file, **options)
    if mode == "w":
        return Encoder(file, **options)
    raise ValueError(f"invalid mode: {mode!r}")


__all__ = ["Decoder", "DecoderBuilder", "Record", "Header", "Flag", "Flags", "SequenceType", "FormatVersion", "Encoder", "open",
           "pack_sequences", "Context", "Pipeline", "ArchiveResult", "decode_batch", "to_text", "to_fasta", "to_fastq", "parse_archive", "shared_context",
           "decode_to_device", "DeviceRecords", "stream_to_device", "DeviceStream", "TABLES", "NafError", "NafArgumentError", "NafIoError", "NafParseError", "NafUnicodeError", "NafDeviceError"]
