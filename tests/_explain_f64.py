"""float64 restatement of the per-feature contributions the reference forms before it sums over features: mf = matmul(W, fx) of
GNAN.py:68-70 (oracle/gnan_port.py:62-72, fx from the reference's K-loop) with W from the oracle's table form (oracle/gnan_lut.py),
and the NAM readout of models.py:374-381 applied feature by feature. Each contribution comes with A, the sum of the absolute values
of its terms, the scale its fp32 rounding error is judged against. The terms reach into the shape functions: each f_k(x) enters A
as M = f_k evaluated with absolute weights and biases on |x| (the forward-error scale of the MLP), because an f_k(x) that nearly
cancels inside its own MLP carries an fp32 error far above eps * |f_k(x)|."""
import torch

from oracle import gnan_lut, gnan_port


def params(stacked):
    return gnan_port.to_torch(stacked, torch.float64)


def pair_weights(p_rho, hop, cnt, mode, C):
    """W [R,N,C] float64 (a single-output rho broadcast over the C channels)"""
    W = gnan_lut.pair_weights(p_rho, hop, cnt, mode)
    return W.expand(-1, -1, C) if W.shape[-1] == 1 else W


def shape_terms(p_fs, x):
    """(fx [N,K,C] = f_k(x_jk), M [N,K,C] = the same MLPs with |weights|, |biases| on |x|)"""
    p_abs = {k: (None if v is None else v.abs()) for k, v in p_fs.items()}
    return gnan_port.shape_functions(p_fs, x.double()), gnan_port.shape_functions(p_abs, x.double().abs())


def node_rows(p_fs, p_rho, x, hop, cnt, mode):
    """(features [R,K,C], A [R,K,C], (fx, M), W [R,N,C]) of the rows of `hop` (int64 [R,N], -1 unreachable)"""
    fx, M = shape_terms(p_fs, x)
    C = fx.shape[2]
    if hop.shape[0] == 0:
        empty = fx.new_zeros(0, fx.shape[1], C)
        return empty, empty, (fx, M), fx.new_zeros(0, fx.shape[0], C)
    W = pair_weights(p_rho, hop, cnt, mode, C)
    F = torch.einsum("ijc,jkc->ikc", W, fx)
    A = torch.einsum("ijc,jkc->ikc", W.abs(), M)
    return F, A, (fx, M), W


def colw_nodes(W, terms):
    """(nodes [N,C], A [N,C]): nodes[j,c] = colw[j,c] S[j,c], colw[j,c] = sum_i W[i,j,c], S = sum_k fx"""
    fx, M = terms
    return W.sum(dim=0) * fx.sum(dim=1), W.abs().sum(dim=0) * M.sum(dim=1)


def graph_row(p_fs, p_rho, x, hop, cnt, mode):
    """one graph: (features [K,C], A [K,C], nodes [N,C], A of nodes [N,C]) = mf.sum(dim=1) and colw * S"""
    F, A, terms, W = node_rows(p_fs, p_rho, x, hop, cnt, mode)
    return (F.sum(dim=0), A.sum(dim=0)) + colw_nodes(W, terms)


def nam_features(p_read, hidden):
    """g_k(hidden[b,k]) -> [B,K,C] (models.py:348-350: the readout NAM is additive over k)"""
    return torch.stack([gnan_port.scalar_mlp(p_read, k, hidden[:, k:k + 1]) for k in range(hidden.shape[1])], dim=1)
