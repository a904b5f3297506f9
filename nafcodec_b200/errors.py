"""Status code -> exception mapping, mirroring nafcodec::error::Error (nafcodec/src/error.rs:4-11) and the
Python binding's convert_error (nafcodec-py/nafcodec/lib.rs:39-77)."""
from . import _ffi


class NafError(Exception):
    """Base class; `.status` holds the nafgpu_status code."""
    status = 0


class NafIoError(NafError, OSError):
    """Error::Io -- truncated or corrupt data (convert_error raises OSError for these)."""


class NafParseError(NafError, ValueError):
    """Error::Nom -- header could not be parsed (convert_error raises ValueError)."""


class NafUnicodeError(NafError, UnicodeError):
    """Error::Utf8 / Io(InvalidData) from String::from_utf8 (reader.rs:108-109)."""


class NafArgumentError(NafError, ValueError):
    """A device export the library refused (NAFGPU_ERR_ARGUMENT): no run, a field that was not decoded, too small an output."""


class NafDeviceError(NafError, RuntimeError):
    """CUDA failure, missing device or missing library: there is no CPU fallback."""


def raise_for_status(lib, code, ctx=None, what=""):
    if code == _ffi.OK:
        return
    detail = ""
    if ctx is not None:
        detail = lib.dll.nafgpu_last_error(ctx).decode()
    msg = lib.strerror(code) + (": " + detail if detail else "") + ((" [" + what + "]") if what else "")
    if code in (_ffi.ERR_UNEXPECTED_EOF, _ffi.ERR_INVALID_DATA, _ffi.ERR_UNSUPPORTED):
        exc = NafIoError(msg)
    elif code == _ffi.ERR_PARSE:
        exc = NafParseError("parser failed: " + msg)
    elif code == _ffi.ERR_UTF8:
        exc = NafUnicodeError("failed to decode UTF-8 data")
    elif code == _ffi.ERR_ARGUMENT:
        exc = ValueError(msg)
        exc.status = code
        raise exc
    elif code == _ffi.ERR_NOMEM:
        exc = MemoryError(msg)
        exc.status = code
        raise exc
    else:
        exc = NafDeviceError(msg)
    exc.status = code
    raise exc
