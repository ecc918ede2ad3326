"""Import alias so that the reference's own scripts run unmodified against the B200 path:

    from audioset_convnext_inf.pytorch.convnext import ConvNeXt, convnext_tiny      # demo_convnext.py:13,
                                                                                    # evaluate_convnext_on_audioset.py:14,
                                                                                    # pytorch/extract_embeddings.py:12
    from audioset_convnext_inf.pytorch.pytorch_utils import forward, move_data_to_device
    from audioset_convnext_inf.pytorch.evaluate import Evaluator                   # evaluate_convnext_on_audioset.py

resolves to audioset_convnext_inf_b200 (libacx kernels; Evaluator scores the tags on the GPU instead of with sklearn).
Only the hot-path modules and the evaluation harness are aliased; the reference's training / dataset / PANNs modules
are out of scope (SURVEY.md section 2) and are deliberately absent."""
