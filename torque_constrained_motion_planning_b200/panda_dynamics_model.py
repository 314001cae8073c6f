"""Drop-in for ``panda_dynamics_model``, the module the reference's ``dyn`` torque test imports
(``import panda_dynamics_model as pdm``, panda_primitives.py:6, calls :86-91) but does not ship.

    get_mass_matrix(q)         -> ndarray (7, 7)   M(q), symmetric positive definite
    get_coriolis_matrix(q, dq) -> ndarray (7, 7)   C(q, dq), Christoffel-consistent: C dq + g == rne(q, dq, 0)
    get_gravity_vector(q)      -> ndarray (7,)     g(q)
    get_forward_dynamics(q, dq, tau) -> ndarray (7,)  ddq = M(q)^-1 (tau - C(q, dq) dq - g(q))
    get_inverse_mass_matrix(q) -> ndarray (7, 7)   M(q)^-1, exactly symmetric

The terms are those of the arm + hand the reference's rne.py models, without a payload (the ``dyn`` closure adds the
payload through the tool Jacobian).  Each call is a batch of one on the GPU and takes the first 7 entries of any
sequence, like ``rne.rne``.  The ``*_batch`` forms take ``[7][n]`` arrays (CUDA tensors or NumPy) and an optional
``engine.InertialModel``; ``engine.dynamics_batch`` returns several terms from one launch, and
``engine.forward_dynamics_batch`` both ddq and M^-1 (with a payload, in rne or dyn mode).
"""
from __future__ import annotations

import numpy as np

from . import engine


def _col(v) -> np.ndarray:
    return np.asarray(v, dtype=np.float64).reshape(-1)[:7].reshape(7, 1)


def get_mass_matrix(q) -> np.ndarray:
    return engine.dynamics_batch(_col(q))["M"][:, :, 0].copy()


def get_coriolis_matrix(q, dq) -> np.ndarray:
    return engine.dynamics_batch(_col(q), _col(dq), mass_matrix=False, coriolis=True, gravity=False)["C"][:, :, 0].copy()


def get_gravity_vector(q) -> np.ndarray:
    return engine.dynamics_batch(_col(q), mass_matrix=False)["g"][:, 0].copy()


def get_mass_matrix_batch(q, model=None):
    """[7][n] -> M [7][7][n]."""
    return engine.dynamics_batch(q, gravity=False, model=model)["M"]


def get_coriolis_matrix_batch(q, dq, model=None):
    """[7][n], [7][n] -> C [7][7][n]."""
    return engine.dynamics_batch(q, dq, mass_matrix=False, coriolis=True, gravity=False, model=model)["C"]


def get_gravity_vector_batch(q, model=None):
    """[7][n] -> g [7][n]."""
    return engine.dynamics_batch(q, mass_matrix=False, model=model)["g"]


def get_forward_dynamics(q, dq, tau) -> np.ndarray:
    return engine.forward_dynamics_batch(_col(q), _col(dq), _col(tau))["qdd"][:, 0].copy()


def get_inverse_mass_matrix(q) -> np.ndarray:
    return engine.forward_dynamics_batch(_col(q), qdd=False, minv=True)["Minv"][:, :, 0].copy()


def get_forward_dynamics_batch(q, dq, tau, model=None):
    """[7][n], [7][n], [7][n] -> ddq [7][n]."""
    return engine.forward_dynamics_batch(q, dq, tau, model=model)["qdd"]


def get_inverse_mass_matrix_batch(q, model=None):
    """[7][n] -> M^-1 [7][7][n]."""
    return engine.forward_dynamics_batch(q, qdd=False, minv=True, model=model)["Minv"]
