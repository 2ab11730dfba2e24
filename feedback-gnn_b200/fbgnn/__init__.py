"""fbgnn -- B200-native BP -> feedback-GNN -> BP decoder behind Feedback-GNN's layer API.

The names below are the ones the reference exports from ``sionna.fec.ldpc``, ``sionna.channel``
and ``sionna.utils`` for this path, so ``n1270.py`` / ``n882.py`` only change their imports.
Everything numerical runs in ``libfbgnn.so`` (CUDA, sm_100a); there is no CPU fallback.
"""
from .codes_q import (css_code, create_circulant_matrix, create_generalized_bicycle_codes,
                      hypergraph_product, hamming_code, rep_code, create_surface_codes,
                      create_rotated_surface_codes, create_checkerboard_toric_codes,
                      create_QC_GHP_codes, create_cyclic_permuting_matrix,
                      create_bivariate_QC_codes, readAlist, alistToNumpy)
from .gf2 import row_echelon, rank, kernel, row_basis, compute_code_distance, inverse, int2bin, int_mod_2
from .gnn import load_weights, save_weights, read_weights, WEIGHTS_DIR, GNN_BP4
from .decoding_q import QLDPCBPDecoder
from .decoding import LDPCBPDecoder
from .pauli import Pauli, pauli_thresholds
from .feedback_gnn import (Feedback_GNN, Sandwich_BP_GNN_Evaluation_Model, BP_BSC_Model, ErrorIndicator, pack_bits,
                           unpack_bits, packed_words)
from .bp_osd import OSD_Decoder, OSD0_Decoder, LSD_Decoder, BP4_OSD_Model, BP2_OSD_Model
from .utils import count_block_errors, count_errors, compute_bler, compute_ber, zeros_like, sim_ber, PlotBER, BinarySource
from .training import (First_Stage_BP_Model, Second_Stage_GNN_BP_Model, Adam, CosineDecay, clip_by_value, train_step,
                       BP4_Error_Model, Feedback_GNN_Error_Model)
from ._ffi import (FbgnnError, Context, DeviceArray, default_context, device_count, from_dlpack)

__version__ = "0.1.0"
