"""rwkv_lm_ext_b200 -- B200-native (sm_100a) WKV6 hot path behind yynil/RWKV_LM_EXT's operator surface.

Importing the package does not touch the GPU or the shared library; the first operator call loads
``libwkv6_b200.so`` and raises if it is missing (there is no CPU / eager fallback)."""
from ._lib import LIB_PATH, Wkv6B200Error, launch_count, load, set_decay_clamp, set_impl  # noqa: F401
from .ops import (HEAD_SIZE, RUN_CUDA_RWKV6, RUN_CUDA_RWKV6_BI, RUN_CUDA_RWKV6_STATE, RUN_RWKV_6, RWKV_6,  # noqa: F401
                  RUN_CUDA_RWKV6_STATE_BPTT, WKV_6, WKV_6_BI, WKV_6STATE, WKV_6STATE_BPTT, WKV_6STATE_INFCTX,
                  exact_route_report, install, rwkv6, wkv6_bi_cuda, wkv6_cuda,
                  wkv6infctx_cuda, wkv6state_cuda)
from .heads import (add_layernorm, create_mask_and_rev_idx, eos_gather, eos_index, gather_rows, groupnorm_gate, groupnorm_gate_pair, pooling,  # noqa: F401
                    reverse_x, tmix_ddlerp_lora, tmix_ddlerp_mix, tmix_shift_lerp)
from .cmix import cmix_shift_lerp2, cmix_x060_forward, relu_sq, sigmoid_mul  # noqa: F401
from .encoders import (GraphedForward, bi_encoder_encode, bi_encoder_hidden, bi_tmix_forward, blocks_forward, causal_hidden, classification_logits,  # noqa: F401
                       cross_encoder_rows, encode_corpus, length_buckets, sequence_embedding)
from .infctx import (BlockState, BlockStateList, ChannelMixState, TimeMixState, infctx_forward,  # noqa: F401
                     infctx_train_step)
from .tmix import Tmix_x060, tmix_x060_finish, tmix_x060_forward, tmix_x060_project  # noqa: F401

__version__ = "0.1.0"
