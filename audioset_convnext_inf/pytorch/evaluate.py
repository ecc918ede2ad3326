"""`audioset_convnext_inf.pytorch.evaluate`: the reference's `Evaluator` (evaluate.py:12-60).  `evaluate(data_loader)`
runs the batch loop and scores the clipwise output against the targets on the GPU; it returns per-class
"average_precision", "auc" and "d_prime"."""
from audioset_convnext_inf_b200.evalloop import Evaluator  # noqa: F401

__all__ = ["Evaluator"]
