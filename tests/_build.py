"""Build a gnan_b200 module configured like the reference module a golden case was generated from."""
import torch


def build_module(z, device=None, load=True):
    v = z["variant"]
    sd = {k: torch.tensor(val) for k, val in z["sd"].items()}
    if v == "batched":
        from gnan_b200.batched import TensorGNAN
        m = TensorGNAN(z["K"], z["C"], 2, hidden_channels=z["H"], is_graph_task=z["is_graph_task"])
    elif v == "gnanpy_tensor":
        from gnan_b200.GNAN import TensorGNAN
        m = TensorGNAN(z["K"], z["C"], z["L"], z["H"], bias=z["bias"], normalize_rho=z["normalize_rho"],
                       is_graph_task=z["is_graph_task"], rho_per_feature=z["rho_per_feature"])
    elif v == "models_tensor":
        from gnan_b200.models import TensorGNAN
        m = TensorGNAN(z["K"], z["C"], z["L"], z["H"], bias=z["bias"], normalize_rho=z["normalize_rho"],
                       is_graph_task=z["is_graph_task"], rho_per_feature=z["rho_per_feature"],
                       readout_n_layers=z["readout_n_layers"])
    else:
        from gnan_b200.models import GNAN
        m = GNAN(z["K"], z["C"], num_layers=z["L"], hidden_channels=z["H"], bias=z["bias"],
                 normalize_rho=z["normalize_rho"], rho_per_feature=z["rho_per_feature"])
    if load:
        m.load_state_dict(sd, strict=True)
    if device is not None:
        m = m.to(device)
    return m
