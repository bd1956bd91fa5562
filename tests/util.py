"""Shared helpers for the test-suite."""
import os

import numpy as np

from cvxpylayers_b200.problems import Batch
from cvxpylayers_b200.structure import ConeSpec, Structure

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = ["qp_c1", "qp_eq", "lp_dense", "socp", "sdp"]


def load_golden(name: str):
    z = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    cones = ConeSpec(z=int(z["cone_z"]), l=int(z["cone_l"]), q=[int(v) for v in z["cone_q"]], s=[int(v) for v in z["cone_s"]])
    hasP = z["P_indices"].size > 0
    st = Structure(int(z["n"]), int(z["m"]), z["A_indptr"], z["A_indices"], cones,
                   z["P_indptr"] if hasP else None, z["P_indices"] if hasP else None)
    bt = Batch(st, z["A_vals"], z["b"], z["c"], z["P_vals"] if hasP else None, name=name)
    return bt, {k: z[k] for k in ("x", "y", "s", "dx", "dy", "dA", "dP", "db", "dc")}


def rel_err(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ----------------------------------------------------------------------------- the reference's own gradcheck programs
def ref_sdp_batch(C_list):
    """``min tr(C X) s.t. tr(X) = 1, X >> 0`` for 3 x 3 symmetric C -- the program of the reference's PSD
    gradcheck (cvxpylayers ``tests/test_torch.py:233-248``) written directly in solver form with x = svec(X)
    (lower triangle, column-major, off-diagonals * sqrt 2): one zero-cone row for the trace, -x + s = 0 with s in the
    PSD cone.  The optimum is the rank-one projector on the smallest eigenvector of C and is strictly complementary
    when that eigenvalue is simple, so the solution map is differentiable.  One instance per C in ``C_list``."""
    from cvxpylayers_b200.problems import mat_to_svec

    k, n = 3, 6
    diag_idx = [0, 3, 5]   # svec positions of X_00, X_11, X_22
    indptr = [0, 3] + [3 + i + 1 for i in range(n)]
    indices = diag_idx + list(range(n))
    st = Structure(n, 1 + n, np.asarray(indptr, np.int32), np.asarray(indices, np.int32), ConeSpec(z=1, s=[k]))
    B = len(C_list)
    A_vals = np.tile(np.concatenate([np.ones(3), -np.ones(n)]), (B, 1))
    b = np.zeros((B, 1 + n)); b[:, 0] = 1.0
    c = np.stack([mat_to_svec(np.asarray(C, dtype=float)) for C in C_list])
    return Batch(st, A_vals, b, c, None, name="ref_sdp")


def ref_soc_batch(c_list, t_list):
    """``min c'x + 0.1 ||x||^2 s.t. ||x|| <= t`` (n = 3) -- the program of the reference's SOC gradcheck
    (cvxpylayers ``tests/test_dual_variables.py:346-369``) in solver form: P = 0.2 I, one SOC of size 4 with
    s = (t, x).  Outputs of the reference's check: the SOC dual (sum), parameters c and t."""
    n = 3
    indptr = [0, 0, 1, 2, 3]
    st = Structure(n, 4, np.asarray(indptr, np.int32), np.arange(3, dtype=np.int32), ConeSpec(q=[4]),
                   np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32))
    B = len(c_list)
    A_vals = -np.ones((B, 3))
    b = np.zeros((B, 4)); b[:, 0] = np.asarray(t_list, dtype=float)
    return Batch(st, A_vals, b, np.asarray(c_list, dtype=float), np.full((B, n), 0.2), name="ref_soc")


# ----------------------------------------------------------------------------- a cvxpy-free stand-in for the reference package
def install_fake_cvxpylayers(monkeypatch):
    """cvxpy / cvxpylayers are not installable in this image.  This builds just enough of the reference's module
    layout in ``sys.modules`` to drive ``cvxpylayers_b200.interface.register()`` the way the real package would:

    * ``cvxpylayers.interfaces.get_solver_ctx / get_torch_cvxpylayer`` -- closed dispatch that rejects unknown names
      (cvxpylayers ``src/cvxpylayers/interfaces/__init__.py:13-101``);
    * ``cvxpylayers.utils.parse_args.parse_args(problem, variables, parameters, solver, ...)`` -- refuses solver names
      cvxpy does not know (that is what ``problem.get_problem_data(solver=...)`` does, ``parse_args.py:447-462``), then
      calls ``interfaces.get_solver_ctx`` and returns a LayersContext-like dataclass;
    * ``cvxpylayers.torch.cvxpylayer`` with ``CvxpyLayer.forward`` doing the reference's sequence: flatten ->
      three sparse products -> ``_CvxpyLayer.apply`` -> recover (``torch/cvxpylayer.py:434-487``).

    ``problem`` is a dict carrying what cvxpy's canonicalisation would produce (the ParamConeProg pieces)."""
    import dataclasses
    import sys
    import types
    from types import SimpleNamespace

    import torch

    pkg = types.ModuleType("cvxpylayers")
    ifs = types.ModuleType("cvxpylayers.interfaces")
    utils = types.ModuleType("cvxpylayers.utils")
    pa = types.ModuleType("cvxpylayers.utils.parse_args")
    tpk = types.ModuleType("cvxpylayers.torch")
    tl = types.ModuleType("cvxpylayers.torch.cvxpylayer")

    def get_solver_ctx(solver, param_prob, cone_dims, data, kwargs, verbose=False):
        raise RuntimeError("Unknown solver. Check if your solver is supported by CVXPYlayers")

    def get_torch_cvxpylayer(solver):
        raise RuntimeError("Unknown solver. Check if your solver is supported by CVXPYlayers")

    ifs.get_solver_ctx, ifs.get_torch_cvxpylayer = get_solver_ctx, get_torch_cvxpylayer

    @dataclasses.dataclass
    class LayersContext:
        parameters: list
        reduced_P: object
        q: object
        reduced_A: object
        cone_dims: object
        solver_ctx: object
        solver: str
        var_recover: list = dataclasses.field(default_factory=list)
        user_order_to_col_order: tuple = ()
        batch_sizes: list = None
        gp: bool = False

        def validate_params(self, params):   # (the reference records the per-parameter batch sizes here, parse_args.py:102-139)
            batch = (params[0].shape[0],) if params[0].dim() > 1 else ()
            self.batch_sizes = [p.shape[0] if batch else 0 for p in params]
            self.user_order_to_col_order = tuple(range(len(params)))
            return batch

    def parse_args(problem, variables, parameters, solver, gp=False, verbose=False, canon_backend=None, solver_args=None):
        if solver not in ("DIFFCP", "CLARABEL", "SCS"):   # cvxpy: "The solver B200 is not installed"
            raise ValueError(f"The solver {solver} is not installed.")
        pp = problem["param_prob"]
        sctx = ifs.get_solver_ctx(solver, pp, problem["dims"], {}, solver_args, verbose=verbose)
        n_, m_ = pp.q.shape[0] - 1, pp.reduced_A.problem_data_index[2][0]
        rec = [SimpleNamespace(primal=slice(0, n_), dual=None, shape=(n_,), source="primal", unpack_fn="reshape"),
               SimpleNamespace(primal=None, dual=slice(0, m_), shape=(m_,), source="dual", unpack_fn="reshape")]
        return LayersContext(parameters, pp.reduced_P, pp.q, pp.reduced_A, problem["dims"], sctx, solver, var_recover=rec)

    pa.parse_args = parse_args

    class _Spmm(torch.autograd.Function):   # the reference's _ScipySparseMatmul (torch/cvxpylayer.py:12-37)
        @staticmethod
        def forward(ctx, M, x):
            ctx.MT = M.T.tocsr()
            return torch.from_numpy(np.asarray(M @ x.detach().cpu().numpy())).to(x.device)

        @staticmethod
        def backward(ctx, g):
            return None, torch.from_numpy(np.asarray(ctx.MT @ g.cpu().numpy())).to(g.device)

    def _apply_gp_log_transform(params, ctx):
        return params

    def _flatten_and_batch_params(params, ctx, batch):
        B = batch[0] if batch else 1
        flat = [p.reshape(B, -1).T if batch else p.reshape(-1, 1) for p in params]
        ones = torch.ones((1, B), dtype=flat[0].dtype, device=flat[0].device)
        ps = torch.cat(flat + [ones], dim=0)
        return ps if batch else ps.squeeze(1)

    def _recover_results(primal, dual, ctx, batch):
        return (primal, dual) if batch else (primal[0], dual[0])

    class CvxpyLayer(torch.nn.Module):
        def __init__(self, problem, parameters, variables, solver=None, solver_args=None):
            super().__init__()
            self.ctx = pa.parse_args(problem, variables, parameters, solver, solver_args=solver_args)
            pp = problem["param_prob"]
            self._A, self._q = pp.reduced_A.reduced_mat, pp.q
            self._P = pp.reduced_P.reduced_mat if pp.reduced_P.problem_data_index is not None else None

        def forward(self, *params, solver_args=None, warm_start=False):
            batch = self.ctx.validate_params(list(params))
            p_stack = tl._flatten_and_batch_params(params, self.ctx, batch)
            P_eval = _Spmm.apply(self._P, p_stack) if self._P is not None else None
            q_eval, A_eval = _Spmm.apply(self._q, p_stack), _Spmm.apply(self._A, p_stack)
            layer = ifs.get_torch_cvxpylayer(self.ctx.solver)
            needs_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
            primal, dual, _, _ = layer.apply(P_eval, q_eval, A_eval, self.ctx, solver_args or {}, needs_grad, None)
            return tl._recover_results(primal, dual, self.ctx, batch)

    tl.CvxpyLayer, tl._apply_gp_log_transform, tl._flatten_and_batch_params, tl._recover_results = (
        CvxpyLayer, _apply_gp_log_transform, _flatten_and_batch_params, _recover_results)
    pkg.interfaces, pkg.utils, pkg.torch = ifs, utils, tpk
    utils.parse_args, tpk.cvxpylayer, tpk.CvxpyLayer = pa, tl, CvxpyLayer
    for name, mod in (("cvxpylayers", pkg), ("cvxpylayers.interfaces", ifs), ("cvxpylayers.utils", utils),
                      ("cvxpylayers.utils.parse_args", pa), ("cvxpylayers.torch", tpk), ("cvxpylayers.torch.cvxpylayer", tl)):
        monkeypatch.setitem(sys.modules, name, mod)
    import cvxpylayers_b200.interface as itf

    monkeypatch.setattr(itf, "_REGISTERED", False)
    return SimpleNamespace(pkg=pkg, ifs=ifs, pa=pa, tl=tl)


def fake_param_prob(bt, full_P: bool = True):
    """What cvxpy's canonicalisation would hand over for a layer whose parameters ARE the problem data of ``bt``
    (parameters, in order: A_cvx values in CSC order, b, c, P values of the FULL symmetric matrix in CSC order):
    ``reduced_A/P.problem_data_index`` (CSC structures), ``reduced_mat`` (parameter -> value maps, last column = constant)
    and ``q``.  Returns (problem dict, list of parameter arrays [B, size])."""
    import scipy.sparse as sp
    from types import SimpleNamespace

    from cvxpylayers_b200 import problems as pr

    st = bt.structure
    bd = pr.to_boundary(bt)
    n, m, B = st.n, st.m, bt.B
    na = bd.A_eval.shape[0]
    hasP = bt.P_vals is not None
    if hasP:
        Pd = np.stack([bt.P_dense(i) for i in range(B)])
        patt = sp.csc_matrix((np.abs(Pd).sum(0) != 0).astype(float)) if full_P else sp.csc_matrix(np.triu(np.abs(Pd).sum(0) != 0).astype(float))
        patt.sort_indices()
        prow, pcol = patt.indices, np.repeat(np.arange(n), np.diff(patt.indptr))
        Pvals = Pd[:, prow, pcol]
        nP = prow.size
    else:
        nP = 0
    P1 = na + n + nP + 1
    eye = lambda rows, off, tot: sp.csr_matrix((np.ones(rows), (np.arange(rows), off + np.arange(rows))), shape=(tot, P1))  # noqa: E731
    A_mat = eye(na, 0, na)
    q_mat = eye(n, na, n + 1)
    red_P = SimpleNamespace(problem_data_index=(patt.indices, patt.indptr, (n, n)) if hasP else None,
                            reduced_mat=eye(nP, na + n, nP) if hasP else None)
    pp = SimpleNamespace(reduced_A=SimpleNamespace(problem_data_index=(bd.con_indices, bd.con_ptr, bd.shape), reduced_mat=A_mat),
                         reduced_P=red_P, q=q_mat)
    dims = SimpleNamespace(zero=st.cones.z, nonneg=st.cones.l, soc=list(st.cones.q), psd=list(st.cones.s), exp=st.cones.ep, p3d=[])
    params = [bd.A_eval.T.copy(), bd.q_eval[:n].T.copy()] + ([Pvals] if hasP else [])
    return {"param_prob": pp, "dims": dims}, params
