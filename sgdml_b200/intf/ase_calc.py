"""ASE calculator on the B200 engine -- the reference's ``sgdml.intf.ase_calc.SGDMLCalculator``
(intf/ase_calc.py:36-110): same constructor arguments, unit handling and ``results`` layout, float64 end to end
(the reference's torch path downcasts positions to float32, predict.py:1197-1201).

MD drivers call ``calculate`` with ONE geometry at a time: that call goes through the engine's small-batch path
(sweep over the training points split across CTAs, the launch sequence replayed from a CUDA graph,
``sgdml_b200_predict`` in csrc/predict.cu).

ASE itself is optional (as in the reference, which raises ImportError without it): ``SGDMLCalculatorCore`` holds
everything that does not need ASE and is what the tests exercise; ``SGDMLCalculator`` exists only when ASE imports.
"""

import logging

import numpy as np

from ..predict import GDMLPredict

# ase.units: kcal / mol in eV (CODATA 2014 values as ASE uses them): 4.184e3 J / (N_A e)
_KCAL_PER_MOL_IN_EV = 4.184e3 / (6.022140857e23 * 1.6021766208e-19)


class SGDMLCalculatorCore(object):
    """Unit conversion + prediction of intf/ase_calc.py:81-110, without the ASE base class."""

    implemented_properties = ['energy', 'forces']

    def _setup(self, model_path, E_to_eV, F_to_eV_Ang, use_torch=False):
        self.log = logging.getLogger(__name__)
        model = model_path if isinstance(model_path, dict) else np.load(model_path, allow_pickle=True)
        self.gdml_predict = GDMLPredict(model, use_torch=use_torch)
        self.gdml_predict.prepare_parallel(n_bulk=1)  # ase_calc.py:84 (a no-op tuning call on the engine)
        self.log.warning(
            "Please remember to specify the proper conversion factors, if your model does not use 'kcal/mol' and 'Ang' as units."
        )
        self.E_to_eV = E_to_eV  # energy unit of the model -> eV
        self.Ang_to_R = F_to_eV_Ang / E_to_eV  # Angstrom -> length unit of the model (ase_calc.py:93-94)
        self.F_to_eV_Ang = F_to_eV_Ang  # force unit of the model -> eV/Ang

    def compute(self, positions):
        """positions (N, 3) in Angstrom -> {'energy': eV, 'forces': (N, 3) eV/Ang} (ase_calc.py:98-110)."""
        r = np.array(positions, dtype=np.float64) * self.Ang_to_R
        e, f = self.gdml_predict.predict(r.ravel())
        e = e * self.E_to_eV
        f = f * self.F_to_eV_Ang
        return {'energy': e, 'forces': f.reshape(-1, 3)}

    def compute_hessian(self, positions):
        """positions (N, 3) in Angstrom -> analytic Hessian d^2 E / dR^2, (3N, 3N) in eV/Ang^2 (the model's
        Hessian times E_to_eV * Ang_to_R^2).  Rows and columns run over (atom, x/y/z)."""
        r = np.array(positions, dtype=np.float64) * self.Ang_to_R
        _, _, h = self.gdml_predict.predict_hessian(r.ravel())
        return h[0] * (self.E_to_eV * self.Ang_to_R**2)


try:
    from ase.calculators.calculator import Calculator
    from ase.units import kcal, mol

    class SGDMLCalculator(Calculator, SGDMLCalculatorCore):
        implemented_properties = ['energy', 'forces']

        def __init__(self, model_path, E_to_eV=kcal / mol, F_to_eV_Ang=kcal / mol, use_torch=False, *args, **kwargs):
            super(SGDMLCalculator, self).__init__(*args, **kwargs)
            self._setup(model_path, E_to_eV, F_to_eV_Ang, use_torch=use_torch)

        def calculate(self, atoms=None, *args, **kwargs):
            super(SGDMLCalculator, self).calculate(atoms, *args, **kwargs)
            self.results = self.compute(atoms.get_positions())

        def get_hessian(self, atoms=None):
            """Analytic Hessian (3N, 3N) in eV/Ang^2 at the positions of `atoms` (default: the attached atoms).
            'hessian' is not a standard ASE property, so it is not cached in ``results``.  Harmonic analysis::

                from ase.vibrations import VibrationsData
                vib = VibrationsData.from_2d(atoms, calc.get_hessian(atoms))
                vib.get_frequencies()
            """
            atoms = atoms if atoms is not None else self.atoms
            return self.compute_hessian(atoms.get_positions())

except ImportError:

    def __getattr__(name):
        if name == 'SGDMLCalculator':
            raise ImportError("Optional ASE dependency not found! Please run 'pip install sgdml[ase]' to install it.")
        raise AttributeError(name)
