"""video-pre-training_b200 -- B200-native (sm_100a) implementation of the VPT policy forward path.

The directory name carries a hyphen (it is fixed by the project layout), so import it through the root-level shim:

    import vpt_b200                      # == this package
    pol = vpt_b200.MinecraftAgentPolicy(action_space, policy_kwargs, pi_head_kwargs).cuda()

Host code here is plumbing (parameter storage, weight re-layout, buffer allocation, launch order); all arithmetic
of the forward path runs in csrc/*.cuh behind the C ABI of include/vpt_b200.h.  No CPU fallback exists.
"""
from . import _native  # noqa: F401
from .types import DictType, Discrete, TensorType, idm_action_space, minecraft_action_space  # noqa: F401
from .agent import ActionCodec, IDMAgent, MineRLAgent, composite_cursor, ingest_frames, resize_frames  # noqa: F401
from .policy import InverseActionNet, InverseActionPolicy, MinecraftAgentPolicy, MinecraftPolicy, NetConfig  # noqa: F401
from .checkpoint import load_model_parameters, load_training_state, load_weights, save_training_state, save_weights  # noqa: F401
from .training import BCTrainer, RLTrainer  # noqa: F401
from .parallel import FlatAdamDP  # noqa: F401

POLICY_KWARGS_2X = dict(  # agent.py:16-36
    attention_heads=16, attention_mask_style="clipped_causal", attention_memory_size=256, diff_mlp_embedding=False,
    hidsize=2048, img_shape=[128, 128, 3], impala_chans=[16, 32, 32], impala_kwargs={"post_pool_groups": 1}, impala_width=8,
    init_norm_kwargs={"batch_norm": False, "group_norm_groups": 1}, n_recurrence_layers=4, only_img_input=True,
    pointwise_ratio=4, pointwise_use_activation=False, recurrence_is_residual=True, recurrence_type="transformer",
    timesteps=128, use_pointwise_layer=True, use_pre_lstm_ln=False,
)
PI_HEAD_KWARGS = dict(temperature=2.0)  # agent.py:38


def idm_net_kwargs(**over):
    """The released IDM (README model zoo "4x_idm"; kwargs inferred in SURVEY.md section 0 and confirmed by its parameter
    count): conv3d 3->128 pre-stage, 4x-width CNN, hidsize 4096, 32 heads, 2 unmasked layers over 128-frame chunks."""
    kw = dict(attention_heads=32, attention_mask_style="none", attention_memory_size=128,
              conv3d_params=dict(inchan=3, outchan=128, kernel_size=[5, 1, 1], padding=[2, 0, 0]), hidsize=4096,
              img_shape=[128, 128, 128], impala_chans=[16, 32, 32], impala_kwargs={"post_pool_groups": 1}, impala_width=16,
              init_norm_kwargs={"batch_norm": False, "group_norm_groups": 1}, n_recurrence_layers=2, only_img_input=True,
              pointwise_ratio=4, pointwise_use_activation=False, recurrence_is_residual=True, recurrence_type="transformer",
              single_output=True, timesteps=128, use_pointwise_layer=True, use_pre_lstm_ln=False)
    kw.update(over)
    return kw


def policy_kwargs(width="2x", **over):
    """The released model family (README model zoo): 1x / 2x / 3x = impala_width 4/8/12, hidsize 1024/2048/3072."""
    w = {"1x": (4, 1024, 8), "2x": (8, 2048, 16), "3x": (12, 3072, 24)}[width]
    kw = dict(POLICY_KWARGS_2X, impala_width=w[0], hidsize=w[1], attention_heads=w[2])
    kw.update(over)
    return kw
