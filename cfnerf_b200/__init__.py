"""cfnerf_b200 — B200-native (sm_100a) implementation of CF-NeRF's per-ray K-sample render / train hot path.

Public surface = the reference's own callables (see api.py) over the C-ABI in include/cfnerf_b200.h.
Importing the package does not load the CUDA library; the first call does, and fails loudly if it is missing.
"""
from .api import (configure, gemm, gemm_bf16, install, kde_nll_loss, mean_over_k, merge_sorted, raw2outputs, rays_from_pose, reference_t_schedule,
                  render_image, render_rays, render_rays_host, run_network, sample_pdf, test_latents, trainer_loss)
from .engine import Engine, engine_for
from .evaluate import evaluate_view, evaluate_views, sparsification
from .field import field_grid, query_field
from .network import NeRFFlowsParams

__all__ = ["render_rays", "run_network", "raw2outputs", "sample_pdf", "merge_sorted", "mean_over_k", "install", "configure",
           "kde_nll_loss", "trainer_loss", "rays_from_pose", "gemm", "gemm_bf16", "render_image", "render_rays_host", "Engine", "engine_for", "NeRFFlowsParams", "reference_t_schedule", "test_latents",
           "evaluate_view", "evaluate_views", "sparsification", "query_field", "field_grid"]
__version__ = "0.1.0"
