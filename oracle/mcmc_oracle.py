"""numpy restatement of ``MCMC.model_mh`` of agarbuno/ces (ces/sample.py:121-196).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- the checker for the device chains of ces_b200/sample.py, never the
product.

Parity: PINNED.  tests/test_oracle_mcmc.py compares it with the chains of the REAL reference stored in
tests/golden/mcmc_cases.npz (ces/sample.py exec'd unmodified, tests/golden/make_golden_mcmc.py): same samples, same
acceptance rate, same state of numpy's global generator afterwards.

The restatement is functional where the reference is a method with state on ``self``: the forward model is a callable
``g = forward(theta)`` (the reference calls ``enka.G(theta, model)`` = ``model(theta)``, ces/calibrate.py:95-104), the
resume state (``self.samples``) is passed in and returned.  Random numbers come from numpy's global generator in the
reference's order: ``normal(0, 1, p)`` for the proposal (:198-202), whatever the model draws in its evaluation (the
reference's ``banana`` draws ``normal(0, 1, [2])`` even without noise, ces/utils.py:122 -- pass ``forward_draws=2``), then
``uniform()`` for the accept test (:182).  The device chains beside the reference's one are restated with ``start``, their
first state (also the point of the initial Phi), and ``noise``, their Philox draws (oracle/philox_oracle.py).
"""
import numpy as np


def model_mh(forward, n_mcmc, prior, Ustar, y_obs, Gamma, delta=1.0, enka_scaling=True, update=None, beta=0.5,
             samples=None, forward_draws=0, start=None, noise=None):
    """Returns ``(samples (p, n + 1 [+ previous]), accept_rate)``.  ``prior``: object with ``logpdf`` and ``cov``.
    ``start``: the first state and the point of the initial Phi (default: the ensemble mean).  ``noise``: a callable
    ``it -> (z (p), u)`` giving step it's normals and accept uniform (default: numpy's global generator, in the
    reference's order)."""
    Ustar = np.asarray(Ustar, dtype=float)
    p = Ustar.shape[0]
    if enka_scaling:                                                      # :123-126
        scales = delta * np.linalg.cholesky(np.cov(Ustar).reshape(p, p))
    else:
        scales = delta * np.eye(p)
    if update == "pCN":                                                   # :128-129
        scales = np.linalg.cholesky(prior.cov)

    def G(theta):
        if forward_draws:
            np.random.normal(0, 1, [forward_draws])                       # drawn inside the reference's model call
        return np.asarray(forward(theta), dtype=float)

    current = Ustar.mean(axis=1) if start is None else np.asarray(start, dtype=float)   # :131
    yg = G(current.flatten()) - y_obs                                     # :137-139
    phi_current = (yg * np.linalg.solve(2 * Gamma, yg)).sum()             # :140
    if update != "pCN":
        phi_current -= prior.logpdf(current.flatten())                    # :141-147
    if samples is not None:                                               # :156-160 (phi_current stays the mean's)
        chain = list(np.asarray(samples).T)
        current = chain[-1]
    else:
        chain = [current.flatten()]
    accept = 0.0
    for it in range(int(n_mcmc)):
        z, u = noise(it) if noise is not None else (np.random.normal(0, 1, p), None)
        if update is None:                                                # :167-168, :198-199
            proposal = current + np.matmul(scales, z)
        else:                                                             # :169-170, :201-202
            proposal = np.sqrt(1 - beta ** 2) * current + np.sqrt(beta) * np.matmul(scales, z)
        yg = G(proposal.flatten()) - y_obs                                # :172-178
        phi_proposal = (yg * np.linalg.solve(2 * Gamma, yg)).sum()
        if update != "pCN":
            phi_proposal -= prior.logpdf(proposal.flatten())              # :179-182
        if u is None:
            u = np.random.uniform()
        if np.log(u) < phi_current - phi_proposal:                        # :188-191
            current = np.copy(proposal)
            phi_current = np.copy(phi_proposal)
            accept += 1.0
        chain.append(current.flatten())                                   # :193
    return np.array(chain).T, accept / n_mcmc                             # :195-196
