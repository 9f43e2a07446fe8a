"""extrack_b200 — B200-native (sm_100a CUDA) track-likelihood engine behind ExTrack's Python API.

Only the hot path of ``extrack.tracking`` is provided: ``param_fitting`` / ``cum_Proba_Cs`` /
``Proba_Cs`` / ``predict_Bs`` and the parameter builders (plus ``predict_transitions`` / ``transition_summary``: the
per-step two-state posteriors of the same annotation, and ``predict_residuals``: its one-step-ahead predictive
densities and PIT values, ``predict_path`` / ``path_segments``: its most probable state paths and their dwell
times, and ``sample_paths`` / ``sample_segments``: posterior draws of whole state paths and their dwell times), and ``param_uncertainty``: standard errors of fitted parameters from per-track scores along the frozen grouping
plan, plus the data formats either side of it:
``readers.read_table`` (table -> length-bucketed ``all_tracks``) and ``simulate.sim_tracks``.  See DESIGN.md.
"""
from . import readers, tracking  # noqa: F401
from .tracking import (  # noqa: F401
    Proba_Cs,
    cum_Proba_Cs,
    extract_params,
    generate_params,
    get_2DSPT_params,
    get_params,
    ParamUncertainty,
    param_fitting,
    param_uncertainty,
    path_segments,
    predict_Bs,
    predict_path,
    predict_residuals,
    predict_transitions,
    sample_paths,
    sample_segments,
    transition_summary,
)

__version__ = "0.1.0"
