"""Ray-transfer-matrix optics and detector images with the call shape of the reference's
``src/simulator/diagnostics.py`` (legacy twin: ``src/solvers-legacy/rtm_solver.py``).

Every ``*_solve`` is one pass of the fused optics kernel over the rays (``sp_optics_image``); ``histogram`` /
``interferogram`` / ``polarimetry`` is one binning pass.  ``spec()`` returns the same optical train as data so that
``propagator.solve_and_image`` can run it in the propagation kernel's epilogue instead.
Units: ``rf`` arrives in metres, is converted with ``m_to_mm`` (diagnostics.py:313), lengths L, R, Lx, Ly in mm.
"""
from dataclasses import dataclass, field as dc_field

import numpy as np
import torch

from . import engine


# ---- element functions (diagnostics.py:122-245): (4,N) in -> (4,N) out, NaN columns = rejected ----------
def _apply(r, ops):
    as_numpy = not isinstance(r, torch.Tensor)
    out, _ = engine.optics_image(engine.to_device(r), ops, input_mm=True)
    return out.cpu().numpy() if as_numpy else out


def m_to_mm(r):
    rr = r.clone() if isinstance(r, torch.Tensor) else np.array(r, copy=True)
    rr[0::2] = rr[0::2] * 1e3
    return rr


def mm_to_m(r):
    rr = r.clone() if isinstance(r, torch.Tensor) else np.array(r, copy=True)
    rr[0::2] = rr[0::2] * 1e-3
    return rr


def lens(r, f1, f2):
    return _apply(r, [("lens", f1, f2)])


def sym_lens(r, f):
    return lens(r, f, f)


def travel(r, d):
    return _apply(r, [("travel", d)])


distance = travel                                   # legacy name, rtm_solver.py:73


def circular_aperture(r, R, E=None):
    if E is None:
        return _apply(r, [("circ_ap", R)])
    as_numpy = not isinstance(r, torch.Tensor)
    ro, eo = engine.optics_image(engine.to_device(r), [("circ_ap", R)], jf=engine.to_device(E, torch.complex128),
                                 input_mm=True)
    return (ro.cpu().numpy(), eo.cpu().numpy()) if as_numpy else (ro, eo)


def circular_stop(r, R):
    return _apply(r, [("circ_stop", R)])


def annular_stop(r, R1, R2):                        # returns the mask only, as upstream (diagnostics.py:211-220)
    rr = r[0] ** 2 + r[2] ** 2
    return (rr > R1 ** 2) & (rr < R2 ** 2)


def rect_aperture(r, Lx, Ly):
    return _apply(r, [("rect_ap", Lx, Ly)])


def knife_edge(r, offset, axis, direction):
    if direction == 0:
        print("Direction must be < 0 or > 0")
        return r
    return _apply(r, [("knife", offset, {"x": 0, "y": 2}[axis], direction)])


def d2r(d):
    return d * np.pi / 180


# ---- optical trains as data -------------------------------------------------------------------------------
@dataclass
class DiagnosticSpec:
    ops: list
    image: object                  # engine.ImageBuffer
    wavelength: float = 0.0
    name: str = ""


def chain_ops(name, L=400, R=25, focal_plane=0, **kw):
    """Op lists of the reference's diagnostic layouts (diagnostics.py:388-524,614-638; rtm_solver.py:197-422)."""
    if name == "shadow_single":
        return [("travel", 3 * L / 4 - focal_plane), ("circ_ap", R), ("lens", L / 2, L / 2), ("travel", 3 * L / 2)]
    if name in ("shadow_two", "interf_two"):
        return [("travel", L - focal_plane), ("circ_ap", R), ("lens", L / 2, L / 2), ("travel", L * 2),
                ("circ_ap", R), ("lens", L / 2, L / 2), ("travel", L)]
    if name == "shadow_single_exp":
        return [("travel", L), ("circ_ap", R), ("lens", L / 2, L / 2), ("travel", kw.get("detL", 400))]
    if name in ("schlieren_DF", "schlieren_LF"):
        mid = ("circ_stop" if name.endswith("DF") else "circ_ap", kw.get("R_stop", 1))
        return [("travel", L - focal_plane), ("circ_ap", R), ("lens", L, L), ("travel", L), mid,
                ("travel", L), ("circ_ap", R), ("lens", L, L), ("travel", L)]
    if name == "refracto_incoherent":
        return [("travel", 3 * L / 4 - focal_plane), ("circ_ap", R), ("lens", L / 2, L / 2), ("travel", 3 * L / 2),
                ("rect_ap", 15, 30), ("circ_ap", R), ("lens", L / 3, L / 2), ("travel", L)]
    if name == "refracto_coherent":          # field not advanced across the middle travel (rtm_solver.py:308-314)
        return [("travel", 3 * L / 4 - focal_plane), ("circ_ap", R), ("lens", L / 2, L / 2), ("travel_noE", 3 * L / 2),
                ("circ_ap", R), ("lens", L / 3, L / 2), ("travel", L)]
    if name == "schlieren_knife":            # SURVEY.md 8d-C4: the dark-field layout with diagnostics.py:226-245's knife edge as the stop
        return [("travel", L), ("circ_ap", R), ("lens", L, L), ("travel", L),
                ("knife", kw.get("offset", 0.0), kw.get("axis", 2), kw.get("direction", 1)),
                ("travel", L), ("circ_ap", R), ("lens", L, L), ("travel", L)]
    # rtm_solver-louis.py:185-438 -- the older sympy-lambdified trains (lens * distance composites, apertures after the lenses;
    # the only diagnostic upstream that has a knife edge in it: fixed 0.1 mm threshold in the Fourier plane, :128-139,375-391)
    if name == "louis_refractometer":
        return [("travel", L), ("lens", L / 2, L / 2), ("circ_ap", R), ("travel", 3 * L / 2), ("lens", L / 3, L / 2),
                ("circ_ap", R), ("travel", L)]
    if name == "louis_shadowgraphy":
        return [("travel", kw.get("displacement", 0)), ("travel", L), ("lens", L / 2, L / 2), ("circ_ap", R), ("travel", 3 * L / 2),
                ("lens", L / 3, L / 3), ("circ_ap", R), ("travel", L)]
    if name == "louis_schlieren":
        return [("travel", L), ("lens", L / 2, L / 2), ("circ_ap", R), ("travel", L / 2), ("knife", 1e-1, 2, -1), ("travel", L),
                ("lens", L / 3, L / 3), ("circ_ap", R), ("travel", L)]
    if name == "louis_interferometer":       # no apertures; the field advances across every composite (:397-438)
        return [("travel", L), ("lens", L / 2, L / 2), ("travel", 3 * L / 2), ("lens", L / 3, L / 3), ("travel", L)]
    raise ValueError(name)


def spec(name, *, bin_scale=1, pix_x=3448, pix_y=2574, L=400, R=25, Lx=18, Ly=13.5, focal_plane=0, wavelength=0.0,
         interferogram=False, stokes=False, ref_beam=None, **kw):
    """A fused-path diagnostic: optical train ``name`` + a fresh detector image (a ray-count histogram, an interferogram,
    or with ``stokes=True`` the ray count and Stokes I, Q, U of a polarimeter, see ``Polarimetry``)."""
    if stokes and interferogram:
        raise ValueError("a channel records either an interferogram or a Stokes image, not both")
    if stokes and ref_beam is not None:
        raise ValueError("a reference beam has no polarimetric meaning: stokes=True takes no ref_beam")
    ops = chain_ops(name, L=L, R=R, focal_plane=focal_plane, **kw)
    if ref_beam is not None:
        ops = [("ref_beam", ref_beam[0], ref_beam[1])] + ops
    mk = (engine.ImageBuffer.for_interferogram if interferogram else
          engine.ImageBuffer.for_stokes if stokes else engine.ImageBuffer.for_histogram)
    return DiagnosticSpec(ops, mk(bin_scale, pix_x, pix_y, Lx, Ly), wavelength, name)


# ---- classes (diagnostics.py:269-640) ------------------------------------------------------------------------
class Diagnostic:
    def __init__(self, wavelength, rf, Jf=None, *, focal_plane=0, L=400, R=25, Lx=18, Ly=13.5, x=None, y=None,
                 x_l=None, y_l=None, amp=None, phase=None):
        self.wavelength, self.focal_plane, self.L, self.R, self.Lx, self.Ly = wavelength, focal_plane, L, R, Lx, Ly
        self.x, self.y, self.x_l, self.y_l, self.amp, self.phase = x, y, x_l, y_l, amp, phase
        if rf is None:
            raise ValueError("rf should not be None")
        self._numpy = not isinstance(rf, torch.Tensor)
        self._rf_m = engine.to_device(rf)                                  # metres, as returned by solve
        self._Jf = None if Jf is None else engine.to_device(Jf, torch.complex128)
        self._rf_det = None                                                # detector-plane rays (mm)
        self.H = None

    def _view(self, t):
        return t if (t is None or not self._numpy) else t.cpu().numpy()

    @property
    def rf(self):
        return self._view(self._rf_det if self._rf_det is not None else self._rf_m)

    @property
    def r0(self):
        return self._view(m_to_mm(self._rf_m))

    @property
    def Jf(self):
        return self._view(self._Jf)

    def _run(self, name, coherent=False, wl=None, ref_beam=None, **kw):
        ops = chain_ops(name, L=self.L, R=self.R, focal_plane=self.focal_plane, **kw)
        if ref_beam is not None:
            ops = [("ref_beam", ref_beam[0], ref_beam[1])] + ops
        self._ops = ops
        jf = self._Jf if coherent else None
        if coherent and jf is None:
            raise ValueError("This diagnostic requires a calculated Jf matrix.")
        self._rf_det, jo = engine.optics_image(self._rf_m, ops, jf=jf, wavelength=wl or self.wavelength)
        if coherent:
            self._Jf = jo

    def histogram(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False):
        """diagnostics.py:323-353: np.histogram2d of the non-NaN rays on [-Lx/2, Lx/2] x [-Ly/2, Ly/2]; H is (ny, nx)."""
        img = engine.ImageBuffer.for_histogram(bin_scale, pix_x, pix_y, self.Lx, self.Ly)
        src = self._rf_det if self._rf_det is not None else m_to_mm(self._rf_m)
        engine.optics_image(src, [], image=img, input_mm=True, want_rays=False)
        self.xedges = np.linspace(-self.Lx / 2, self.Lx / 2, img.nx + 1)
        self.yedges = np.linspace(-self.Ly / 2, self.Ly / 2, img.ny + 1)
        self.H = self._view(img.result())
        if clear_mem:
            clear_rays(self)

    def histogram_legacy(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False):
        """diagnostics.py:355-379: complex-amplitude binning on digitize edges; H = sqrt(Re(sum Ex)^2 + Re(sum Ey)^2)."""
        if self._Jf is None:
            raise ValueError("This diagnostic requires a calculated Jf matrix.")
        img = engine.ImageBuffer.for_interferogram(bin_scale, pix_x, pix_y, self.Lx, self.Ly)
        src = self._rf_det if self._rf_det is not None else m_to_mm(self._rf_m)
        engine.optics_image(src, [], jf=self._Jf, image=img, input_mm=True, want_rays=False)
        self.H = self._view(img.result())
        if clear_mem:
            clear_rays(self)


def clear_rays(self):                                # diagnostics.py:247-256
    self._rf_m = self._rf_det = self._Jf = None


class Shadowgraphy(Diagnostic):
    def single_lens_solve(self):                     # diagnostics.py:388-394
        self._run("shadow_single")

    def two_lens_solve(self):                        # diagnostics.py:396-405
        self._run("shadow_two")

    def single_exp_solve(self, detL=400):            # rtm_solver.py:216-222
        self._run("shadow_single_exp", detL=detL)


class Schlieren(Diagnostic):
    def DF_solve(self, R=1):                         # diagnostics.py:415-437
        self._run("schlieren_DF", R_stop=R)

    def LF_solve(self, R=1):                         # diagnostics.py:446-460
        self._run("schlieren_LF", R_stop=R)

    def knife_solve(self, offset=0.0, axis="y", direction=1):    # SURVEY.md 8d-C4 (upstream's own: chain_ops('louis_schlieren'))
        self._run("schlieren_knife", offset=offset, axis={"x": 0, "y": 2}[axis], direction=direction)


class Refractometry(Diagnostic):
    def incoherent_solve(self):                      # diagnostics.py:469-484
        self._run("refracto_incoherent")

    def coherent_solve(self, wl=None, generation="current"):
        """``generation='current'``: diagnostics.py:505-524 as upstream ships it -- the first aperture is applied to ``r0``
        (the rays never make the ``3L/4 - focal_plane`` leg to the first lens) while the field is advanced by the length of
        that leg (``propagate_E(r2, r1)``) and across every later element.  Two passes of the optics kernel: one whose
        only output is the advanced field, then the rest of the train on the unmoved rays.
        ``generation='legacy'``: rtm_solver.py:288-331 (rays carried to the lens; no field advance across the middle
        travel).  Both are pinned against the reference's own output (tests/golden g9 / g4)."""
        if generation == "legacy":
            return self._run("refracto_coherent", coherent=True, wl=wl)
        if generation != "current":
            raise ValueError("generation must be 'current' or 'legacy'")
        if self._Jf is None:
            raise ValueError("This diagnostic requires a calculated Jf matrix.")
        L_, wl = self.L, wl or self.wavelength
        _, jf = engine.optics_image(self._rf_m, [("travel", 3 * L_ / 4 - self.focal_plane)], jf=self._Jf, wavelength=wl)
        self._ops = [("circ_ap", self.R), ("lens", L_ / 2, L_ / 2), ("travel", 3 * L_ / 2), ("circ_ap", self.R),
                     ("lens", L_ / 3, L_ / 2), ("travel", L_)]
        self._rf_det, self._Jf = engine.optics_image(self._rf_m, self._ops, jf=jf, wavelength=wl)

    def refractogram(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False):   # diagnostics.py:526-527
        self.histogram_legacy(bin_scale=bin_scale, pix_x=pix_x, pix_y=pix_y, clear_mem=clear_mem)

    def fresnel_solve(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False, gridding="triangulation"):
        """diagnostics.py:529-552: the exit rays' amplitude and phase (constructor arguments ``amp``, ``phase``) are
        interpolated onto the grid ``x`` x ``y`` (lengths ``x_l``, ``y_l``) and carried over ``3L/4 - focal_plane`` by the
        Fresnel integral (``fresnel_integral.propagate``); ``self.Jf`` becomes that field, as upstream.  Upstream then
        indexes the (ny, nx) field with ray numbers while binning (``self.Jf[0, i]``), which JAX's clamped indexing turns
        into an image of two grid rows; here ``H`` is the field's magnitude on the grid instead."""
        from . import fresnel_integral
        if any(v is None for v in (self.x, self.y, self.x_l, self.y_l, self.amp, self.phase)):
            raise ValueError("fresnel_solve needs x, y, x_l, y_l, amp and phase (constructor keyword arguments)")
        U = fresnel_integral.propagate(self.wavelength, self.x, self.y, self.x_l, self.y_l, m_to_mm(self._rf_m), self.amp,
                                       self.phase, 3 * self.L / 4 - self.focal_plane, gridding=gridding)
        self._Jf = U
        self.H = self._view(U.abs())
        if clear_mem:
            clear_rays(self)


class Interferometry(Diagnostic):
    def interfere_ref_beam(self, n_fringes, deg):    # diagnostics.py:559-581 (evaluated on exit rays in METRES)
        if self._Jf is None:
            print("This diagnostic requires a calculated Jf matrix.")
            return None
        _, self._Jf = engine.optics_image(self._rf_m, [("ref_beam", n_fringes, deg)], jf=self._Jf)

    def two_lens_solve(self, wl=None, ref_beam=(10, 20)):
        """diagnostics.py:614-638 (reference beam n_fringes=10, deg=20 then two-lens telescope with E
        propagation); ``ref_beam=None`` gives the legacy rtm_solver.py:376-422 behaviour."""
        self._run("interf_two", coherent=True, wl=wl, ref_beam=ref_beam)

    def interferogram(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False):   # diagnostics.py:640
        self.histogram_legacy(bin_scale=bin_scale, pix_x=pix_x, pix_y=pix_y, clear_mem=clear_mem)


class Polarimetry(Diagnostic):
    """Faraday-rotation polarimetry (no upstream counterpart): per detector pixel the ray count ``N`` and the Stokes
    parameters ``I``, ``Q``, ``U`` of the rays' Jones vectors, summed incoherently, which is what a camera behind a
    polariser integrates.  For the reference's Jones vector ``E = amp e^{i phase} (-sin pol, cos pol)``
    (full_solver.py:883-890) a ray contributes ``I = amp^2``, ``Q = -amp^2 cos 2pol`` and ``U = -amp^2 sin 2pol``; Stokes V
    is identically 0.  ``pol`` is the Faraday rotation integrated by ``ScalarDomain(B_on=True)`` and ``amp`` the
    inverse-bremsstrahlung attenuation (``inv_brems=True``).  Needs ``Jf`` (``solve(..., return_E=True)``)."""

    def __init__(self, wavelength, rf, Jf=None, **kw):
        if Jf is None:
            raise ValueError("This diagnostic requires a calculated Jf matrix.")
        super().__init__(wavelength, rf, Jf, **kw)

    def single_lens_solve(self):                     # the shadowgraphy imaging trains
        self._run("shadow_single")

    def two_lens_solve(self):
        self._run("shadow_two")

    def polarimetry(self, bin_scale=1, pix_x=3448, pix_y=2574, clear_mem=False):
        """Bins the rays on the histogram's edges (np.histogram2d semantics); sets ``N``, ``I``, ``Q``, ``U`` (ny, nx) and
        ``H = I``, the attenuation-weighted shadowgram.  The Jones vectors are binned as they left the plasma: the optics
        multiply both components by the same phase factor, which the Stokes parameters do not see."""
        if self._Jf is None:
            raise ValueError("This diagnostic requires a calculated Jf matrix.")
        img = engine.ImageBuffer.for_stokes(bin_scale, pix_x, pix_y, self.Lx, self.Ly)
        src = self._rf_det if self._rf_det is not None else m_to_mm(self._rf_m)
        engine.optics_image(src, [], jf=self._Jf, image=img, input_mm=True, want_rays=False)
        self.xedges = np.linspace(-self.Lx / 2, self.Lx / 2, img.nx + 1)
        self.yedges = np.linspace(-self.Ly / 2, self.Ly / 2, img.ny + 1)
        S = img.stokes()
        self.N, self.I, self.Q, self.U = (self._view(S[k]) for k in "NIQU")
        self.H = self.I
        if clear_mem:
            clear_rays(self)

    def rotation_angle(self):
        """Intensity-weighted polarisation angle per pixel in the convention of ``pol``: ``0.5 atan2(-U, -Q)``, in
        (-pi/2, pi/2]; NaN where no ray landed."""
        if isinstance(self.I, torch.Tensor):
            a = 0.5 * torch.atan2(-self.U, -self.Q)
            return torch.where(self.N > 0, a, torch.full_like(a, float("nan")))
        with np.errstate(invalid="ignore"):
            return np.where(self.N > 0, 0.5 * np.arctan2(-self.U, -self.Q), np.nan)

    def analyser_image(self, angle):
        """What a camera behind a linear analyser at ``angle`` (radians, the convention of ``pol``) records:
        ``0.5 (I - Q cos 2 angle - U sin 2 angle)``; a ray of angle ``pol`` passes ``amp^2 cos^2(pol - angle)`` (Malus).
        Two calls at ``pi/2 +- delta`` give the two images of the usual two-camera polarimeter."""
        m = torch if isinstance(angle, torch.Tensor) else np          # angle: a number or a per-pixel array
        return 0.5 * (self.I - self.Q * m.cos(2 * angle) - self.U * m.sin(2 * angle))
