"""Every shape the model accepts is computed by some kernel route; every other shape is refused up front.

`ScaMLGP` routes a call to the fused A_m path (`cond_prepare` / `predict_conditioned`), to the prediction kernel
plus the stand-alone cross-covariance kernel, or to the candidate-gradient and q-block kernels, by the number of
points per source task n, the input dimension d and the number of target points n_t.  For each cell of
n x d x n_t the model must either match the oracle or raise NotImplementedError naming the limit; a ScamlError (a
kernel refusing a launch the model sent it) fails the test."""
import pytest
import torch

from oracle import scaml_oracle as O
from tests.helpers import TOL_GRAD, TOL_MEAN_VAR, rel_err
from tests.test_qbatch import _fitted_model, _oracle_blocks

DT = torch.float64


def _refused(fn):
    """Run fn; None if it raised NotImplementedError naming a limit, else its result."""
    try:
        return fn(), None
    except NotImplementedError as e:
        msg = str(e)
        assert "<=" in msg or "outside" in msg, msg
        return None, msg


def _route_cell(eng, n, d, nt):
    got, msg = _refused(lambda: _fitted_model(eng, 2, n, d, nt, False, 0, 0, False))
    if got is None:
        assert nt > 0, msg  # building a model without target data launches nothing
        return "refused"
    model, args, g = got
    routes = []
    X1 = torch.rand(5, d, dtype=DT, generator=g)
    post, _ = _refused(lambda: model.posterior(X1))
    if post is not None:
        om, ov = O.scaml_posterior(*args, X1)
        assert rel_err(post.mean.reshape(-1).numpy(), om.numpy()) < TOL_MEAN_VAR
        assert float((post.variance.reshape(-1) - ov).abs().max()) < TOL_MEAN_VAR * float(ov.abs().max())
        routes.append("q1")
    X3 = torch.rand(2, 3, d, dtype=DT, generator=g)
    joint, _ = _refused(lambda: model.posterior(X3))
    if joint is not None:
        rm, rc = _oracle_blocks(args, X3)
        jm, jc = joint.mean.reshape(2, 3), joint.mvn.covariance_matrix
        assert float((jm - rm).abs().max()) < TOL_MEAN_VAR * max(1.0, float(rm.abs().max()))
        assert float((jc - rc).abs().max()) < TOL_MEAN_VAR * float(rc.abs().max())
        routes.append("joint")
    if model.supports_candidate_gradients:
        Xg = X1.clone().requires_grad_(True)
        mean, var, dm, dv = model.posterior_with_grad(X1)
        om, ov = O.scaml_posterior(*args, Xg)
        rdm, = torch.autograd.grad(om.sum(), Xg, retain_graph=True)
        rdv, = torch.autograd.grad(ov.sum(), Xg)
        assert rel_err(dm.numpy(), rdm.numpy()) < TOL_GRAD
        assert rel_err(dv.numpy(), rdv.numpy()) < TOL_GRAD
        bm, bc, vjp = model.posterior_blocks(X3)
        assert float((bc - rc).abs().max()) < TOL_MEAN_VAR * float(rc.abs().max())
        routes += ["grad", "blocks"]
    else:
        with pytest.raises(NotImplementedError):
            model.posterior_with_grad(X1)
        with pytest.raises(NotImplementedError):
            model.posterior_blocks(X3)
    # eval-mode prior (the joint prior blocks of forward)
    model.eval()
    prior, _ = _refused(lambda: model.forward(X1))
    if prior is not None:
        routes.append("forward")
    return routes


@pytest.fixture(scope="module")
def emu_engine(emu_lib):
    from tests.emu_engine import EmuEngine

    return EmuEngine(emu_lib)


# a few cells on the emulation: the fused path, d > 16 through the cross-covariance kernel, n > 256 without it
@pytest.mark.parametrize("n,d,nt", [(40, 6, 5), (40, 20, 5), (260, 3, 0), (260, 20, 3), (200, 32, 3)])
def test_emu_model_routes(emu_engine, n, d, nt):
    _route_cell(emu_engine, n, d, nt)


@pytest.mark.gpu
@pytest.mark.parametrize("nt", [0, 12, 140])
@pytest.mark.parametrize("d", [6, 20, 32])
@pytest.mark.parametrize("n", [200, 300, 512, 600])
def test_gpu_model_routes(engine, n, d, nt):
    routes = _route_cell(engine, n, d, nt)
    print(f"n={n} d={d} n_t={nt}: {routes}")
