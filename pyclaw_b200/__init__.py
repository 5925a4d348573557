"""pyclaw_b200 -- PyClaw's finite-volume time-step hot path, native on B200 (sm_100a).

Keeps the reference's Python API (src/pyclaw/__init__.py:22-43): Controller, Solution,
State, Grid, Dimension, CFL, BC, ClawSolver1D/2D/3D, SharpClawSolver1D/2D/3D, limiters, riemann.
"""
from . import _lib, limiters, riemann, grid, state, solution, solver, clawpack, sharpclaw, controller, util
from . import plot
from .controller import Controller
from .data import Data
from .solution import Solution
from .grid import Dimension, Grid
from .state import State
from .cfl import CFL
from .clawpack import ClawSolver1D, ClawSolver2D, ClawSolver3D
from .sharpclaw import SharpClawSolver1D, SharpClawSolver2D, SharpClawSolver3D
from .solver import BC, CFLError
from .limiters import tvd

__all__ = ['Controller', 'Data', 'plot', 'Dimension', 'Grid', 'Solution', 'State', 'CFL', 'riemann',
           'ClawSolver1D', 'ClawSolver2D', 'ClawSolver3D', 'SharpClawSolver1D', 'SharpClawSolver2D', 'SharpClawSolver3D',
           'limiters', 'tvd', 'BC']
