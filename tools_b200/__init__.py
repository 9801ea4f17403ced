"""tools_b200 -- B200 (sm_100a) backend for the batched PSF / FIPS 203 hot path of qfall/tools.

Host-side mirror of the reference's interface for that path only:
  primitive.psf   : PSF, PSFGPV, PSFGPVRing, PSFPerturbation        (src/primitive/psf/)
  sample.g_trapdoor: GadgetParameters(Ring), gen_trapdoor, short bases (src/sample/g_trapdoor/)
  compression     : LossyCompressionFIPS203                          (src/compression/)
  utils           : rot_minus, rot_minus_matrix                      (src/utils/rotation_matrix.rs), rot_f
                    encode / decode_value_*_polynomialringzq         (src/utils/common_encodings.rs)
  serde_io        : serde-JSON / typetag / FLINT-string import of parameters and keys
All arithmetic on the hot path runs in the CUDA library behind include/qfall_b200.h.
"""
from . import _ffi  # noqa: F401
from .gadget import (GadgetParameters, GadgetParametersRing, find_solution_gadget_mat, find_solution_gadget_vec,  # noqa: F401
                     gen_gadget_mat, gen_gadget_vec, rot_f, rot_minus, rot_minus_matrix, short_basis_gadget)
from ._ffi import NotInDomain, QfError  # noqa: F401
from .psf import PSFGPV, PolyTags, PSFGPVRing, PSFPerturbation  # noqa: F401
from .compression import lossy_compress, lossy_decompress  # noqa: F401
from .encodings import decode_value_from_polynomialringzq, encode_value_in_polynomialringzq  # noqa: F401
