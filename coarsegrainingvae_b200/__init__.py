"""coarsegrainingvae_b200 -- B200 (sm_100a) implementation of the CGVAE equivariant message-passing
hot path behind the reference's Python API (same class names, constructor / forward signatures and
state_dict layout as ``CoarseGrainingVAE.{modules,conv,cgvae,data}``).

All arithmetic runs in hand-written CUDA kernels (csrc/, built into libcgvae_sm100.so, C ABI in
include/cgvae_b200.h).  There is no CPU or PyTorch-eager fallback.
"""
from .cgvae import (BatchGraphs, CGequiVAE, CGprior, EquiEncoder, EquivariantDecoder,  # noqa: F401
                    EquivariantPsuedoDecoder, PCN)
from .conv import (ContractiveMessageBlock, EquiMessageBlock, EquiMessageCross, EquiMessagePsuedo,  # noqa: F401
                   InvariantMessage, PseudoUpdateBlock, UpdateBlock)
from .data import (CG_collate, CGDataset, DeviceCGDataset, DeviceProteinDataset, batch_to, get_neighbor_list,  # noqa: F401
                   get_neighbor_list_batch)
from .modules import Dense, DistanceEmbed, make_directed  # noqa: F401
from .ops import get_matmul_precision, matmul_precision, set_matmul_precision  # noqa: F401

__version__ = "0.1.0"
