"""Packed Domain values on the device (qf_domain_encode_dev / qf_domain_decode_dev): the Golomb-Rice code of DESIGN 4.11
for int32 rows held in torch CUDA tensors, on the current torch stream.  For the format see include/qfall_b200.h."""
import torch

from . import _ffi


def _stream():
    return _ffi.ptr(int(torch.cuda.current_stream().cuda_stream)) if torch.cuda.current_stream().cuda_stream else None


def encode(x: torch.Tensor, k: int, slot_bytes: int):
    """x: rows x dim int32 (CUDA, contiguous) -> (packed uint8 rows x slot_bytes, nbytes int32 rows); nbytes -1 and a zero
    slot for a row whose code does not fit or that holds INT32_MIN."""
    assert x.is_cuda and x.dtype == torch.int32 and x.dim() == 2 and x.is_contiguous()
    rows, dim = x.shape
    out = torch.empty((rows, int(slot_bytes)), dtype=torch.uint8, device=x.device)
    nbytes = torch.empty(rows, dtype=torch.int32, device=x.device)
    st = _ffi.lib().qf_domain_encode_dev(_ffi.ptr(x.data_ptr()), rows, dim, int(k), int(slot_bytes), _ffi.ptr(out.data_ptr()),
                                         _ffi.ptr(nbytes.data_ptr()), _stream())
    if st != _ffi.QF_OK:
        raise _ffi.QfError(st, "qf_domain_encode_dev")
    return out, nbytes


def decode(packed: torch.Tensor, dim: int, k: int):
    """packed: rows x slot_bytes uint8 (CUDA, contiguous) -> (values int32 rows x dim, ok bool rows); a row that is not a
    canonical code has ok False and unspecified values."""
    assert packed.is_cuda and packed.dtype == torch.uint8 and packed.dim() == 2 and packed.is_contiguous()
    rows, slot_bytes = packed.shape
    out = torch.empty((rows, int(dim)), dtype=torch.int32, device=packed.device)
    ok = torch.empty(rows, dtype=torch.uint8, device=packed.device)
    st = _ffi.lib().qf_domain_decode_dev(_ffi.ptr(packed.data_ptr()), rows, int(dim), int(k), slot_bytes,
                                         _ffi.ptr(out.data_ptr()), _ffi.ptr(ok.data_ptr()), _stream())
    if st != _ffi.QF_OK:
        raise _ffi.QfError(st, "qf_domain_decode_dev")
    return out, ok.bool()
