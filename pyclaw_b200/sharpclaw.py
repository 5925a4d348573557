"""SharpClaw solvers (src/pyclaw/sharpclaw.py:28-563): WENO5 + SSP Runge-Kutta.

Each Runge-Kutta stage is ONE kernel launch that reconstructs, solves the interface and
in-cell Riemann problems, sums the fluctuations and applies the stage's linear
combination (clawb200_sharpclaw_stage), where the reference calls ``sharpclaw2.flux2``
and then combines full-field numpy temporaries (sharpclaw.py:172-206).  In 3-D a stage is
two launches (clawb200_sharpclaw_stage3: x and y plane by plane, then z).
"""
import ctypes

import torch

from . import _lib
from .solver import Solver, CFLError, _ptr, _stream


def _div(t, c):
    """t / c with one IEEE division per element (torch evaluates ``tensor / python_float``
    as a multiplication by the reciprocal on CUDA, which is not what numpy does)."""
    return torch.div(t, torch.full((), float(c), dtype=t.dtype, device=t.device))


def start_step(solver, solution):
    """Dummy routine called before each step (sharpclaw.py:19-25)."""
    pass


class SharpClawSolver(Solver):
    r"""
    Superclass for all SharpClawND solvers (sharpclaw.py:28-115).  Attributes: lim_type,
    weno_order, time_integrator ('Euler' | 'SSP33' | 'SSP104'), char_decomp,
    tfluct_solver, aux_time_dep, kernel_language, mbc, fwave, cfl_desired, cfl_max, dq_src.

    Extra attribute of this implementation: ``weno_literals`` ('f32' | 'f64').  The
    reference's generated weno.f90 writes its coefficients as kind-less literals, which
    gfortran reads as REAL(4); 'f32' (default) reproduces that, 'f64' uses doubles.
    """

    def __init__(self, data=None):
        self._required_attrs = list(Solver._base_required) + \
            ['limiters', 'start_step', 'lim_type', 'weno_order', 'time_integrator', 'char_decomp',
             'aux_time_dep', 'mwaves']
        d = dict(Solver._base_defaults)
        d.update({'limiters': [1], 'start_step': start_step, 'lim_type': 2, 'weno_order': 5,
                  'time_integrator': 'SSP104', 'char_decomp': 0, 'tfluct_solver': False,
                  'aux_time_dep': False, 'kernel_language': 'Fortran', 'mbc': 3, 'fwave': False,
                  'cfl_desired': 2.45, 'cfl_max': 2.5, 'dq_src': None, 'weno_literals': 'f32'})
        self._default_attr_values = d
        super(SharpClawSolver, self).__init__(data)

    def _needs_backup_copy(self):
        return self.start_step is not start_step

    # The table-driven WENO kernels (orders 7-17) read their coefficients from a device buffer
    # this solver owns; the problem struct points at it.  No table state lives in the library, so
    # solvers of different orders can be alive side by side.
    def _upload_weno_tables(self):
        tab = getattr(self, '_weno_tab', None)
        if tab is None:
            return
        import torch
        packed = _lib.pack_weno_tables(tab)
        self._weno_dev = torch.as_tensor(packed, device=self._cfl_dev.device)
        self._problem.weno_k = int(tab['k'])
        self._problem.weno_tab = self._weno_dev.data_ptr()

    # ---- one dq evaluation fused with a stage update ----
    def _stage(self, q_buf, qa_buf, out_buf, mode, ca, cb, div, slot, dq_buf=None):
        cfl = ctypes.c_void_p(self._cfl_dev.data_ptr() + 8 * slot)
        if self.ndim == 3:
            _lib.call("clawb200_sharpclaw_stage3", ctypes.byref(self._problem), int(self._mz), float(self._dz),
                      _ptr(q_buf), _ptr(qa_buf), _ptr(out_buf), _ptr(dq_buf), self._aux_ptr, float(self.dt), mode,
                      float(ca), float(cb), float(div), cfl, _stream())
            return
        _lib.call("clawb200_sharpclaw_stage", ctypes.byref(self._problem), _ptr(q_buf), _ptr(qa_buf),
                  _ptr(out_buf), _ptr(dq_buf), self._aux_ptr, float(self.dt), mode, float(ca), float(cb),
                  float(div), cfl, _stream())

    def _bcs_on(self, state, buf, t=None):
        """apply_q_bcs on an arbitrary padded buffer of this state's shape (the stage
        registers); ``t`` is the stage time seen by custom boundary conditions."""
        keep, tkeep = state._q.cur, state.t
        state._q.cur = buf
        if t is not None:
            state.t = t
        try:
            self.apply_q_bcs(state)
        finally:
            state._q.cur = keep
            state.t = tkeep

    def step(self, solution):
        """One Runge-Kutta step (sharpclaw.py:152-210).

        The stages are launched back to back and their Courant numbers are read once at
        the end; the result is committed only if no stage exceeded cfl_max, which is the
        state the reference is left in when CFLError interrupts it (q untouched)."""
        _lib.set_variant(getattr(self, '_variant', None) or self.arithmetic)
        state = solution.states[0]
        self.start_step(self, solution)
        if self.dq_src is not None:
            return self._step_unfused(solution)
        F = state._q
        q0 = F.cur
        self._cfl_dev.zero_()
        AX, CV, FIN = _lib.STAGE_AXPY, _lib.STAGE_CONVEX, _lib.STAGE_FINAL104
        self._bcs_on(state, q0)
        if self.time_integrator == 'Euler':
            new = F.get_spare()
            self._stage(q0, None, new, AX, 0, 0, 1.0, 0)
            nst, spares = 1, []
        elif self.time_integrator == 'SSP33':
            s = self._rk_stages[0]._q
            a, b, new = s.cur, s.get_spare(), F.get_spare()
            self._stage(q0, None, a, AX, 0, 0, 1.0, 0)              # s = q + dq(q)
            self._bcs_on(state, a, state.t + self.dt)
            self._stage(a, q0, b, CV, 0.75, 0.25, 1.0, 1)           # s = .75 q + .25 (s + dq(s))
            self._bcs_on(state, b, state.t + 0.5 * self.dt)
            self._stage(b, q0, new, CV, 1. / 3., 2. / 3., 1.0, 2)   # q = 1/3 q + 2/3 (s + dq(s))
            nst, spares = 3, [(s, b)]
        elif self.time_integrator == 'SSP104':
            s1f, s2f = self._rk_stages[0]._q, self._rk_stages[1]._q
            a, b, new = s1f.cur, s1f.get_spare(), F.get_spare()
            self._stage(q0, None, a, AX, 0, 0, 6., 0)               # s1 = q + dq(q)/6
            slot = 1
            ts = state.t + self.dt / 6.
            for i in range(4):
                self._bcs_on(state, a, ts)
                self._stage(a, None, b, AX, 0, 0, 6., slot)         # s1 = s1 + dq(s1)/6
                a, b = b, a
                slot += 1
                ts = ts + self.dt / 6.
            # s2 = q/25 + 9/25 s1 ; s1 = 15 s2 - 5 s1   (sharpclaw.py:195-196)
            s2 = s2f.cur
            _lib.call("clawb200_ssp104_combine", _ptr(q0), _ptr(a), _ptr(s2),
                      ctypes.c_longlong(q0.numel()), _stream())
            ts = state.t + self.dt / 3.
            for i in range(4):
                self._bcs_on(state, a, ts)
                self._stage(a, None, b, AX, 0, 0, 6., slot)
                a, b = b, a
                slot += 1
                ts = ts + self.dt / 6.
            self._bcs_on(state, a, ts)
            self._stage(a, s2, new, FIN, 0.6, 0.1, 1.0, slot)       # q = s2 + .6 s1 + .1 dq(s1)
            s1f.cur = a
            nst, spares = 10, [(s1f, b)]
        else:
            raise Exception('Unrecognized time integrator')
        for fld, buf in spares:
            fld.put_spare(buf)
        cfls = self._read_cfl(nst)
        for c in cfls:
            if c > self.cfl_max:
                # what the reference sees when dq() raises CFLError (sharpclaw.py:231-232)
                self.cfl.update_global_max(c)
                F.put_spare(new)
                return False
        self.cfl.update_global_max(cfls[-1])
        state._commit(new)

    # ---- path with a user dq_src hook: dq is materialised, combination done on tensors ----
    def dq(self, state):
        """Evaluate dq/dt * (delta t) (sharpclaw.py:221-237); returns the interior view."""
        deltaq = self.dq_hyperbolic(state)
        if self.cfl.get_cached_max() > self.cfl_max:
            raise CFLError('cfl_max exceeded')
        if self.dq_src is not None:
            deltaq += self.dq_src(self, state, self.dt)
        return deltaq

    def dq_hyperbolic(self, state):
        self.apply_q_bcs(state)
        if getattr(self, '_dq_field', None) is None:
            self._dq_field = state._q._alloc()
        self._cfl_dev.zero_()
        self._stage(state._q.cur, None, None, _lib.STAGE_DQ_ONLY, 0, 0, 1.0, 0, dq_buf=self._dq_field)
        self.cfl.update_global_max(self._read_cfl()[0])
        return state._q.interior(self._dq_field)

    def _step_unfused(self, solution):
        state = solution.states[0]
        try:
            if self.time_integrator == 'Euler':
                deltaq = self.dq(state)
                new = state.q + deltaq
            elif self.time_integrator == 'SSP33':
                s = self._rk_stages[0]
                s.q = state.q + self.dq(state)
                s.t = state.t + self.dt
                s.q = 0.75 * state.q + 0.25 * (s.q + self.dq(s))
                s.t = state.t + 0.5 * self.dt
                new = 1. / 3. * state.q + 2. / 3. * (s.q + self.dq(s))
            elif self.time_integrator == 'SSP104':
                s1, s2 = self._rk_stages[0], self._rk_stages[1]
                s1.q = state.q + _div(self.dq(state), 6.)
                s1.t = state.t + self.dt / 6.
                for i in range(4):
                    s1.q = s1.q + _div(self.dq(s1), 6.)
                    s1.t = s1.t + self.dt / 6.
                s2.q = _div(state.q, 25.) + 9. / 25 * s1.q
                s1.q = 15. * s2.q - 5. * s1.q
                s1.t = state.t + self.dt / 3.
                for i in range(4):
                    s1.q = s1.q + _div(self.dq(s1), 6.)
                    s1.t = s1.t + self.dt / 6.
                new = s2.q + 0.6 * s1.q + 0.1 * self.dq(s1)
            else:
                raise Exception('Unrecognized time integrator')
        except CFLError:
            return False
        buf = state._q.get_spare()
        state._q.interior(buf).copy_(new)
        state._commit(buf)

    def set_mthlim(self):
        self.mthlim = self.limiters
        if not isinstance(self.limiters, list):
            self.mthlim = [self.mthlim]
        if len(self.mthlim) == 1:
            self.mthlim = self.mthlim * self.mwaves
        if len(self.mthlim) != self.mwaves:
            raise Exception('Length of solver.limiters is not equal to 1 or to solver.mwaves')

    def setup(self, solution):
        """sharpclaw.py:303-326 / 475-498"""
        if self.kernel_language not in ('Fortran', 'CUDA'):
            raise NotImplementedError("only the CUDA kernels exist; there is no Python/CPU path")
        if self.weno_order not in (5, 7, 9, 11, 13, 15, 17):
            # reconstruct.f90:111-113
            raise Exception("weno_order must be an odd number between 5 and 17 (inclusive).")
        if self.ndim == 3:
            # the 3-D stage (clawb200_sharpclaw_stage3) is WENO5 / tvd2 on the components of q
            if self.weno_order != 5:
                raise NotImplementedError("SharpClawSolver3D: weno_order must be 5 (orders 7-17 are 1-D / 2-D only)")
            if self.char_decomp != 0:
                raise NotImplementedError("SharpClawSolver3D: char_decomp must be 0 (the reconstruction is "
                                          "component-wise in 3-D)")
            if solution.state.mcapa >= 0:
                raise NotImplementedError("SharpClawSolver3D: capacity functions (state.mcapa) are not supported "
                                          "in 3-D, as in ClawSolver3D")
        if self.weno_order != 5:
            # weno7 .. weno17 (weno.f90:104-2425): table-driven kernels, component-wise only
            if self.lim_type != 2 or self.char_decomp != 0:
                raise NotImplementedError("weno_order > 5 is implemented for lim_type=2, char_decomp=0")
            from .weno_tables import tables
            import numpy as np
            tab = tables((self.weno_order + 1) // 2, self.weno_literals)
            variant = _lib.WENO_TABLES
        elif self.lim_type == 2 and self.char_decomp == 0:
            variant = _lib.WENO_PYWENO_F32 if self.weno_literals == 'f32' else _lib.WENO_PYWENO_F64
        elif self.lim_type == 3:
            variant = _lib.WENO_OLD
        elif self.lim_type == 2 and self.char_decomp == 1:
            # wave-based WENO (flux1.f90:95-105; weno5_wave / weno5_fwave).  The reference's 2-D
            # flux1.f90:102-106 calls rpn2 without ixy and then BOTH reconstructions: it cannot run
            if self.ndim != 1:
                raise NotImplementedError("char_decomp=1 (wave-based reconstruction) exists in 1-D only: the "
                                          "reference's 2-D flux1.f90 cannot execute this branch")
            variant = _lib.RECON_WENO_FWAVE if self.fwave else _lib.RECON_WENO_WAVE
        elif self.lim_type == 1 and self.char_decomp == 0:
            # tvd2 (reconstruct.f90:568-625): second-order TVD reconstruction of the components of q
            variant = _lib.RECON_TVD2
        else:
            # char_decomp = 2 / 3 call evec(), which the reference ships as a stub that stops
            # (src/fortran/1d/sharpclaw/evec.f90:11-13: "subroutine evec() has not been provided")
            raise NotImplementedError("lim_type=%s char_decomp=%s is not implemented (char_decomp 2 and 3 need a "
                                      "user-supplied evec(); the reference's own evec.f90 stops)"
                                      % (self.lim_type, self.char_decomp))
        if self.tfluct_solver:
            # the reference's own tfluct is a stub that stops the interpreter
            # (src/fortran/1d/sharpclaw/tfluct.f90:11-13: "you have not defined a function tfluct")
            raise NotImplementedError("tfluct_solver=True: the reference ships no total-fluctuation solver "
                                      "(tfluct.f90 prints an error and stops); none is provided here either")
        # fwave = True with char_decomp = 0 (e.g. the stegoton script): flux1.f90 only uses the
        # solver's amdq / apdq, so an f-wave solver works unchanged
        self.mbc = (self.weno_order + 1) // 2
        state = solution.state
        state.set_mbc(self.mbc)
        self.allocate_rk_stages(solution)
        self.set_mthlim()
        if variant == _lib.RECON_TVD2 and state.meqn > len(self.mthlim):
            # tvd2 indexes mthlim (length mwaves, sharpclaw.py:213-218) with the COMPONENT number:
            # with meqn > mwaves the reference reads past the end of the array
            raise Exception("lim_type=1 reads limiters[m] for every component m: meqn = %d needs %d entries "
                            "but solver.limiters has mwaves = %d" % (state.meqn, state.meqn, len(self.mthlim)))
        # clawparams.mcapa = state.mcapa + 1 (sharpclaw.py:270)
        method = [int(self.dt_variable), 2, 0, 0, 0, state.mcapa + 1, state.maux]
        self._setup_device(state, method=method, mthlim=self.mthlim, weno_variant=variant)
        if self._rp.rp_id == _lib.RP_SHALLOW_BATHY_FWAVE:
            # WENO reconstructs h rather than the surface h + b: the in-cell solve is not balanced and a
            # lake at rest would move (that needs a surface / hydrostatic reconstruction)
            raise NotImplementedError("shallow_bathymetry_fwave runs with ClawSolver1D / ClawSolver2D only: "
                                      "SharpClaw's component-wise WENO reconstruction is not well balanced "
                                      "over bathymetry")
        self._weno_tab = tab if variant == _lib.WENO_TABLES else None
        self._upload_weno_tables()
        self.allocate_bc_arrays(state)
        self._aux_ptr = _ptr(state._aux.cur if state._aux is not None else None)
        self._dq_field = None

    def teardown(self):
        pass


class SharpClawSolver1D(SharpClawSolver):
    def __init__(self, data=None):
        self.ndim = 1
        super(SharpClawSolver1D, self).__init__(data)


class SharpClawSolver2D(SharpClawSolver):
    def __init__(self, data=None):
        self.ndim = 2
        super(SharpClawSolver2D, self).__init__(data)


class SharpClawSolver3D(SharpClawSolver):
    """SharpClaw in 3-D: dq is flux1 summed over the x-, y- and z-slices (DESIGN.md §1), with
    weno_order = 5 and lim_type 1 (tvd2), 2 (PyWENO weno5) or 3 (hand-written weno5), char_decomp = 0,
    no capacity function.  The Courant number is the largest over the three directions, not their sum."""

    def __init__(self, data=None):
        self.ndim = 3
        super(SharpClawSolver3D, self).__init__(data)
