"""adaprox_b200 -- B200-native AdaProx iteration hot path (host-side mirror).

``import adaprox_b200 as AdaProx`` gives the reference's entry points
(src/AdaProx.jl) backed by libadaprox_cuda.so; see INTEGRATION.md for the Julia
``ccall`` shim that binds the same C ABI.
"""
from . import synth, sharding, records                           # noqa: F401  (numpy only; no GPU needed)
from .records import JsonlSink, read_jsonl, find_best, is_logstep, load_libsvm_dataset   # noqa: F401
from ._lib import AdaproxError, LIB_PATH, SYMBOLS, load          # noqa: F401
from .core import (                                               # noqa: F401
    Device, DeviceMatrix, DeviceVector, default_device, set_default_device,
    Counting, without_counting, is_counting_enabled,
    grad_count, prox_count, mul_count, amul_count, eval_count,
    LinearLeastSquares, LogisticLoss, Quadratic, QuadraticGram, Cubic, logistic_loss_grad_Hessian, WorstQuadratic, Simple2DObjective, Simple2DBox,
    Zero, IndZero, NormL1, NormL2, IndBox, Translate, convex_conjugate, prox,
    eval_with_pullback, eval_with_gradient,
    FixedStepsize, MalitskyMishchenkoRule, OurRule, OurRulePlus, stepsize,
    adaptive_primal_dual, adaptive_primal_dual_path, adaptive_primal_dual_lambda_path, condat_vu, adaptive_proxgrad, auto_adaptive_proxgrad, adaptive_proxgrad_path, fixed_proxgrad, adaptive_linesearch_primal_dual, malitsky_pock,
    backtracking_proxgrad, backtracking_nesterov, fixed_nesterov, agraal,
    generate_planted_lasso, last_solve_info,
)
