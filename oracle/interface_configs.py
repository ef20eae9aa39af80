"""The configurations whose state-dict layout and initial values tests/test_model_interface.py checks against
tests/golden/init_state.json (recorded by oracle/make_init_golden.py)."""
from dl4vc_b200.config import min_config, small_config

CONFIGS = {"prod_small": small_config(), "min_small": min_config(layer_sizes=(64, 32), pool_combine_dimension=96),
           "variant": small_config(total_conv_layers=4, residual_layer_start=3, conv_1d_pool_layers=(1, 3), concat_hw_reads=False,
                                   skip_final_maxpool=True, use_strands=False, hidden_dropout=0.0)}
