"""Run configuration: a flat attribute bag filled from a sectioned YAML file.

Drop-in for reference src/config.py:4-50 — same field names, same
`PINNConfig.from_yaml(file='./src/parameters.yml')` entry, sections merged into one
namespace, unknown or missing keys are a TypeError.  Keys that only this implementation
knows (B200 section) are optional so an unmodified reference YAML still loads.
"""
import yaml

REQUIRED_FIELDS = (
    "mesh_file", "n_modes", "hierarchy", "k_neighbors", "epochs", "learning_rate", "corrector_scale",
    "weight_residual", "weight_orthogonal", "weight_projection", "weight_trace", "w_order", "w_eigen",
    "gradient_clipping", "weight_decay", "log_every", "hidden_layers", "dropout", "normalization_eps",
    "prolongation_neighbors", "knn_graph_neighbors", "verbose", "do_extensive_visuals", "diagnostics_viz",
    "vtu_file", "coarse_mesh_files", "sampler_type", "edge_computation_type", "model_type",
)

OPTIONAL_FIELDS = {
    "mlp_mode": "fp32",        # "fp32" parity mode | "bf16" tcgen05 perf mode
    "fps_start": None,         # explicit FPS start vertex (reference draws it unseeded)
    "seed": None,              # torch seed for the corrector initialisation (reference never seeds)
    "cgc_mode": "reference",   # "reference": dense coarse solve as in the reference | "regularized" | "skip"
    "cgc_shift": 1e-3,         # "regularized": coarse solve with K_c + cgc_shift * M_c (block CG on the device)
    "loss_read_delay": 1,      # epochs between launching a step and reading its loss (0 = synchronous like :261)
    "cuda_graph": True,        # replay the epoch body as one CUDA graph after three eager epochs
    "offset_edges": False,     # True: per-level edge lists get node offsets (notebooks); False: reference quirk Q3
    "aggregation": "mean",     # 'mean' (reference) | 'sum' (notebook variant without the degree division)
    "operator_type": "auto",   # level operators of the point samplers: "point_cloud" (robust_laplacian, as the
                               # reference), "fem" (Galerkin P^T K P of the mesh's FEM operators), "auto" (first if installed)
    # notebook variant multigrid_gnn_refine_fixed.ipynb cell 4 (model_type 'adaptive' = learnable per-mode scales)
    "mode_scale_init": 0.01,   # initial value of the AdaptiveCorrector's per-mode scales
    "weight_smooth": 0.0,      # w * sum U_pred o (K U_pred) / (n k) per level
    "weight_smooth_corr": 0.0, # w * sum corr o (K corr) / (n k) per level (the notebook uses one weight for both)
}


class PINNConfig:
    def __init__(self, **fields):
        missing = [f for f in REQUIRED_FIELDS if f not in fields]
        unknown = [f for f in fields if f not in REQUIRED_FIELDS and f not in OPTIONAL_FIELDS]
        if missing:
            raise TypeError("PINNConfig missing required field(s): " + ", ".join(missing))
        if unknown:
            raise TypeError("PINNConfig got unexpected field(s): " + ", ".join(unknown))
        for name in REQUIRED_FIELDS:
            setattr(self, name, fields[name])
        for name, default in OPTIONAL_FIELDS.items():
            setattr(self, name, fields.get(name, default))

    @classmethod
    def from_yaml(cls, file='./src/parameters.yml'):
        with open(file, "r") as handle:
            sections = yaml.safe_load(handle)
        flat = {}
        for body in sections.values():
            flat.update(body)
        return cls(**flat)
