"""CPU: every entry point of the C-ABI library is exercised on the GPU, either called by name in a
tests/test_*_gpu.py file or reached through a composed path that an existing GPU test checks against a reference.
A new kernel that is bound in dquartic/_native.py but reached by no test fails here."""
import glob
import os
import re

from _util import ROOT

from dquartic import _native

# entry point -> the GPU test that checks it through composition (file::function)
COVERED_BY = {
    "dq_qsample": "test_kernels_gpu.py::test_scheduler_kernels_bit_exact",
    "dq_mix_affine": "test_model_gpu.py::test_train_step_loss_and_gradients_match_reference_golden",
    "dq_mse": "test_model_gpu.py::test_train_step_loss_and_gradients_match_reference_golden",
    "dq_scale_by": "test_model_gpu.py::test_train_step_loss_and_gradients_match_reference_golden",
    "dq_add_inplace": "test_model_gpu.py::test_train_step_loss_and_gradients_match_reference_golden",
    "dq_ncl_nlc": "test_model_gpu.py::test_train_step_loss_and_gradients_match_reference_golden",
    "dq_block_bwd": "test_updown_convs_gpu.py::test_attn_cond_proj_convs_and_gelu_block_backward_over_rt",
    "dq_add_mul": "test_model_gpu.py::test_ddim_sampling_matches_reference_golden",
    "dq_ddim_step_x0": "test_round2_gpu.py::test_secondary_modes_vs_oracle",
    "dq_cosine_sums": "test_round2_gpu.py::test_predict_returns_reference_dicts_and_predict_batch_scores_every_window",
    "dq_map_scores": "test_validation_gpu.py::test_map_scores_match_the_float64_oracle",
    "dq_initconv_bwd": "test_updown_convs_gpu.py::test_init_conv_forward_and_one_pass_backward_per_element",
    "dq_sample_dot": "test_round2_gpu.py::test_initconv_one_pass_backward_matches_generic_path",
    "dq_conv1d_fwd": "test_updown_convs_gpu.py::test_resampling_and_plain_conv_per_element_at_training_shape",
    "dq_conv1d_bwd_data": "test_kernels_gpu.py::test_resample_convs",
    "dq_conv1d_bwd_weight": "test_updown_convs_gpu.py::test_attn_cond_proj_convs_and_gelu_block_backward_over_rt",
    "dq_resblock_fwd": "test_updown_convs_gpu.py::test_resnet_block_per_element_at_training_shape",
    "dq_conv_bwd_fused": "test_updown_convs_gpu.py::test_resnet_block_per_element_at_training_shape",
    "dq_conv_bwd_fused_res": "test_updown_convs_gpu.py::test_resnet_block_per_element_at_training_shape",
    "dq_upconv_bwd_fused": "test_updown_convs_gpu.py::test_resampling_and_plain_conv_per_element_at_training_shape",
    "dq_upsample2x": "test_round2_gpu.py::test_upsample_backward_one_pass_matches_three_pass_composition",
    "dq_fold2x": "test_round2_gpu.py::test_upsample_backward_one_pass_matches_three_pass_composition",
    "dq_downconv_bwd_fused": "test_updown_convs_gpu.py::test_resampling_and_plain_conv_per_element_at_training_shape",
    "dq_s2d": "test_round2_gpu.py::test_downsample_backward_one_pass_matches_reindexing_composition",
    "dq_d2s": "test_round2_gpu.py::test_downsample_backward_one_pass_matches_reindexing_composition",
    "dq_down_w": "test_round2_gpu.py::test_downsample_backward_one_pass_matches_reindexing_composition",
    "dq_linattn_fwd": "test_kernels_gpu.py::test_linear_attention_fwd_bwd",
    "dq_linattn_bwd": "test_kernels_gpu.py::test_linear_attention_fwd_bwd",
    "dq_sumsq": "test_kernels_gpu.py::test_fused_adamw_and_clip",
    "dq_clip_coef": "test_kernels_gpu.py::test_fused_adamw_and_clip",
    "dq_multiplex": "test_kernels_gpu.py::test_multiplex_bit_exact_against_reference_golden",
    "dq_gemm_bf16_tn": "test_mid_stage_gpu.py::test_gemm_mid_conv_fwd_dgrad",
}


def _gpu_sources():
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "test_*_gpu.py")))
    assert files
    return {os.path.basename(f): open(f).read() for f in files}


def test_every_entry_point_is_tested_on_the_gpu():
    src = _gpu_sources()
    called = {name for name in _native._SIGS
              if any(re.search(r"[\"']%s[\"']" % name, text) for text in src.values())}
    missing = sorted(set(_native._SIGS) - called - set(COVERED_BY))
    assert not missing, f"entry points no GPU test calls or covers: {missing}"


def test_composition_map_names_existing_tests():
    src = _gpu_sources()
    for name, where in COVERED_BY.items():
        assert name in _native._SIGS, f"{name} is not an entry point any more"
        fname, func = where.split("::")
        assert fname in src, where
        assert re.search(r"^def %s\(" % func, src[fname], flags=re.M), where
