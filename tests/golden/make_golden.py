"""Generates the golden fixtures under tests/golden/ by running the UNMODIFIED reference
(stefanch/sGDML v1.0.3, commit a6ae5e8) on seeded synthetic inputs.

The reference ships no tests or golden vectors of its own (SURVEY.md section 8c), so its
own outputs are the pin.  Run in the build container only (the reference is not on the
GPU box):

    cp -r /root/reference/sgdml baseline/_ref/          # writable copy (predict.py:1046-1074)
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py iterative
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py c60
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py n100
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py pbc_ecstr
    PYTHONPATH=baseline/_ref:. python tests/golden/make_golden.py dropin

Each fixture holds the inputs (geometries, labels, perms, sig, lam, query geometries) and
the reference outputs of every hot-path stage: tril_perms_lin (Desc.perm / train.py:897-904),
R_desc / R_d_desc (Desc.from_R), K (_assemble_kernel_mat, NumPy engine, 1 process), alphas_F,
R_d_desc_alpha, std, c (GDMLTrain.train, analytic solver) and E, F (GDMLPredict.predict,
NumPy engine) on query geometries and on the training geometries.
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'baseline', '_ref'))

import importlib.util  # noqa: E402

_spec = importlib.util.spec_from_file_location('synth', os.path.join(ROOT, 'sgdml_b200', 'synth.py'))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)

import sgdml  # noqa: E402  (the reference)
from sgdml.predict import GDMLPredict  # noqa: E402
from sgdml.train import GDMLTrain  # noqa: E402
from sgdml.utils.desc import Desc  # noqa: E402

assert sgdml.__version__ == '1.0.3'

CASES = {
    # name: (n_atoms, n_train, n_rotors, n_swaps, sig, n_query)
    'n9_m16_s6': (9, 16, 1, 1, 20, 12),  # ethanol-like (BASELINE config 1, reduced M)
    'n5_m10_s1': (5, 10, 0, 0, 10, 6),  # no symmetries
    'n12_m8_s12': (12, 8, 1, 2, 30, 5),  # larger group, D = 66
    'n21_m6_s6': (21, 6, 1, 1, 20, 4),  # aspirin-size descriptor (BASELINE config 2, reduced M)
}


def main():
    gdml_train = GDMLTrain(max_processes=1, use_torch=False)  # one instance per process (train.py:336-342)
    for name, (N, M, n_rot, n_swap, sig, n_query) in CASES.items():
        perms = synth.rotor_swap_group(N, n_rot, n_swap)
        task = synth.make_task(N, M, perms, sig)
        desc = Desc(N, max_processes=1)

        tril_perms = np.array([Desc.perm(p) for p in task['perms']])
        tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')

        R = task['R_train'].reshape(M, -1)
        R_desc, R_d_desc = desc.from_R(R, max_processes=1)
        K = gdml_train._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, sig, desc)

        model = gdml_train.train(task)
        assert np.array_equal(model['tril_perms_lin'], tril_perms_lin)

        predictor = GDMLPredict(model, max_processes=1, use_torch=False)
        R_query = synth.geometries(N, n_query, 1).reshape(n_query, -1)
        E_q, F_q = predictor.predict(R_query)
        E_t, F_t = predictor.predict(R)

        # K.v identity inputs: a fixed random vector through the reference's matrix
        rng = np.random.default_rng(5)
        v = rng.standard_normal(K.shape[0])
        Kv = K @ v

        out = os.path.join(HERE, name + '.npz')
        np.savez_compressed(
            out,
            reference_version=sgdml.__version__,
            n_atoms=N,
            perms=perms,
            sig=sig,
            lam=task['lam'],
            z=task['z'],
            R_train=task['R_train'],
            F_train=task['F_train'],
            E_train=task['E_train'],
            tril_perms_lin=tril_perms_lin,
            R_desc=R_desc,
            R_d_desc=R_d_desc,
            K=K,
            alphas_F=model['alphas_F'],
            R_d_desc_alpha=model['R_d_desc_alpha'],
            model_R_desc=model['R_desc'],
            std=model['std'],
            c=model['c'],
            R_query=R_query,
            E_query=E_q,
            F_query=F_q,
            E_train_pred=E_t,
            F_train_pred=F_t,
            v=v,
            Kv=Kv,
        )
        print(name, 'K', K.shape, 'size %.0f KB' % (os.path.getsize(out) / 1024))


def main_pbc_ecstr():
    """(f)4 rows: periodic boundary conditions (utils/desc.py:44-77: minimum-image pair differences; the
    lattice travels in the task and the model, train.py:524, 826-827, predict.py:332-334) and energy
    constraints in the kernel (train.py:234-300, 940-947, 1052-1086; predict.py:219-229).  Two fixtures:
    pbc_n6_m8 (lattice, no energy constraints) and ecstr_n6_m8 (use_E_cstr, no lattice)."""
    gdml_train = GDMLTrain(max_processes=1, use_torch=False)
    N, M, sig, n_query = 6, 8, 15, 5
    perms = synth.rotor_swap_group(N, 1, 1)
    for name in ('pbc_n6_m8', 'ecstr_n6_m8'):
        task = synth.make_task(N, M, perms, sig)
        lat = None
        if name.startswith('pbc'):
            # a cell smaller than the molecule's extent, so that the minimum-image convention is active for many pairs
            lat = np.array([[2.6, 0.3, 0.0], [0.0, 2.4, 0.2], [0.1, 0.0, 2.9]])  # columns = lattice vectors
            task['lattice'] = lat
        else:
            task['use_E_cstr'] = True
        desc = Desc(N, max_processes=1)
        lat_and_inv = None if lat is None else (lat, np.linalg.inv(lat))
        tril_perms = np.array([Desc.perm(p) for p in task['perms']])
        tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')
        R = task['R_train'].reshape(M, -1)
        R_desc, R_d_desc = desc.from_R(R, lat_and_inv=lat_and_inv, max_processes=1)
        use_E_cstr = bool(task['use_E_cstr'])
        K = gdml_train._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, sig, desc, use_E_cstr=use_E_cstr)
        model = gdml_train.train(task)
        predictor = GDMLPredict(model, max_processes=1, use_torch=False)
        R_query = synth.geometries(N, n_query, 1).reshape(n_query, -1)
        E_q, F_q = predictor.predict(R_query)
        E_t, F_t = predictor.predict(R)
        extra = {}
        if lat is not None:
            extra['lattice'] = lat
        if use_E_cstr:
            extra['alphas_E'] = model['alphas_E']
        out = os.path.join(HERE, name + '.npz')
        np.savez_compressed(
            out, reference_version=sgdml.__version__, n_atoms=N, perms=perms, sig=sig, lam=task['lam'], z=task['z'],
            R_train=task['R_train'], F_train=task['F_train'], E_train=task['E_train'], tril_perms_lin=tril_perms_lin,
            R_desc=R_desc, R_d_desc=R_d_desc, K=K, alphas_F=model['alphas_F'], R_d_desc_alpha=model['R_d_desc_alpha'],
            model_R_desc=model['R_desc'], std=model['std'], c=model['c'], R_query=R_query, E_query=E_q, F_query=F_q,
            E_train_pred=E_t, F_train_pred=F_t, use_E_cstr=use_E_cstr, **extra
        )
        print(name, 'K', K.shape, 'size %.0f KB' % (os.path.getsize(out) / 1024))


def main_iterative():
    """Nystroem-preconditioned CG (solvers/iterative.py) with the reference, forced by a tiny memory
    limit; np.random is seeded so that the leverage-score sampling is reproducible, and the sampled
    inducing columns are stored (the engine and the oracle then solve with the same columns)."""
    from sgdml.solvers.iterative import Iterative

    N, M, sig = 9, 40, 20
    perms = synth.rotor_swap_group(N, 1, 1)
    task = synth.make_task(N, M, perms, sig)
    max_memory = 0.004  # GB -> a handful of inducing points (iterative.py:826-843)
    gdml_train = GDMLTrain(max_memory=max_memory, max_processes=1, use_torch=False)
    np.random.seed(1234)
    model = gdml_train.train(task)
    assert model['solver_name'] == 'cg'
    desc = Desc(N, max_processes=1)
    R = task['R_train'].reshape(M, -1)
    R_desc, R_d_desc = desc.from_R(R, max_processes=1)

    # the preconditioner the reference builds for these inducing columns, applied to a fixed vector
    it = Iterative(gdml_train, desc, max_memory, 1, False)
    P_op, lev_scores = it._init_precon_operator(task, R_desc, R_d_desc, model['tril_perms_lin'], model['inducing_pts_idxs'])
    rng = np.random.default_rng(7)
    v = rng.standard_normal(3 * N * M)
    P_op @ v  # first call only "primes" the operator (iterative.py:122-125)
    Pv = P_op @ v

    predictor = GDMLPredict(model, max_processes=1, use_torch=False)
    R_query = synth.geometries(N, 10, 1).reshape(10, -1)
    E_q, F_q = predictor.predict(R_query)
    y = task['F_train'].ravel() / model['std']
    out = os.path.join(HERE, 'cg_n9_m40.npz')
    np.savez_compressed(
        out,
        reference_version=sgdml.__version__,
        n_atoms=N,
        n_train=M,
        perms=perms,
        sig=sig,
        lam=task['lam'],
        max_memory_gb=max_memory,
        inducing_pts_idxs=model['inducing_pts_idxs'],
        alphas_F=model['alphas_F'],
        solver_iters=model['solver_iters'],
        solver_resid=model['solver_resid'],
        solver_tol=model['solver_tol'],
        norm_y_train=model['norm_y_train'],
        std=model['std'],
        c=model['c'],
        lev_scores=lev_scores,
        v=v,
        Pv=Pv,
        R_query=R_query,
        E_query=E_q,
        F_query=F_q,
        y=y,
    )
    print('cg_n9_m40: %d inducing columns, %d iterations, resid %.3e (tol*|y| = %.3e), size %.0f KB'
          % (len(model['inducing_pts_idxs']), model['solver_iters'], model['solver_resid'],
             model['solver_tol'] * model['norm_y_train'], os.path.getsize(out) / 1024))


def main_c60():
    """BASELINE config 5 shape at reduced M: buckyball C60 (60 atoms, D = 1770) with the 120 permutations of
    I_h.  One block column of K and predictions of a model with random (not trained: K is numerically
    singular at this symmetry) coefficients -- pins the large-molecule assembly and the large-descriptor
    predictor to the reference."""
    N, M, sig = 60, 2, 50
    r0 = synth.c60_geometry()
    perms = synth.icosahedral_group(r0)
    task = synth.make_task(N, M, perms, sig, r0=r0)
    desc = Desc(N, max_processes=1)
    tril_perms = np.array([Desc.perm(p) for p in perms])
    tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')
    R = task['R_train'].reshape(M, -1)
    R_desc, R_d_desc = desc.from_R(R, max_processes=1)
    gdml_train = GDMLTrain(max_processes=1, use_torch=False)
    K_cols = gdml_train._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, sig, desc, col_idxs=np.arange(3 * N, 6 * N))  # index-list mode (train.py:1376-1407)
    rng = np.random.default_rng(11)
    alphas_F = rng.standard_normal(M * 3 * N)
    model = gdml_train.create_model(task, 'analytic', R_desc, R_d_desc, tril_perms_lin, 1.7, alphas_F)
    model['c'] = -3.25
    predictor = GDMLPredict(model, max_processes=1, use_torch=False)
    R_query = synth.geometries(N, 3, 1, r0=r0).reshape(3, -1)
    E_q, F_q = predictor.predict(R_query)
    out = os.path.join(HERE, 'big_c60_m2_s120.npz')
    np.savez_compressed(
        out,
        reference_version=sgdml.__version__,
        n_atoms=N,
        perms=perms,
        sig=sig,
        lam=task['lam'],
        z=task['z'],
        R_train=task['R_train'],
        tril_perms_lin=tril_perms_lin.astype(np.int64),
        R_desc=R_desc,
        R_d_desc=R_d_desc,
        K_cols=K_cols,
        col_start=3 * N,
        alphas_F=alphas_F,
        R_d_desc_alpha=model['R_d_desc_alpha'],
        model_R_desc=model['R_desc'],
        std=model['std'],
        c=model['c'],
        R_query=R_query,
        E_query=E_q,
        F_query=F_q,
    )
    print('big_c60_m2_s120: K_cols', K_cols.shape, 'size %.0f KB' % (os.path.getsize(out) / 1024))


def main_n100():
    """BASELINE config 4 shape at reduced M: synthetic 100-atom molecule (D = 4950), S = 12 (one rotor, two
    swaps).  Every 5th column of the second block column of K (index-list mode) and predictions of a
    random-coefficient model."""
    N, M, sig = 100, 2, 50
    perms = synth.rotor_swap_group(N, 1, 2)
    task = synth.make_task(N, M, perms, sig)
    desc = Desc(N, max_processes=1)
    tril_perms = np.array([Desc.perm(p) for p in perms])
    tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')
    R = task['R_train'].reshape(M, -1)
    R_desc, R_d_desc = desc.from_R(R, max_processes=1)
    gdml_train = GDMLTrain(max_processes=1, use_torch=False)
    cols = np.arange(3 * N, 6 * N, 5)
    K_cols = gdml_train._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, sig, desc, col_idxs=cols)
    rng = np.random.default_rng(12)
    alphas_F = rng.standard_normal(M * 3 * N)
    model = gdml_train.create_model(task, 'analytic', R_desc, R_d_desc, tril_perms_lin, 0.6, alphas_F)
    model['c'] = 12.5
    predictor = GDMLPredict(model, max_processes=1, use_torch=False)
    R_query = synth.geometries(N, 3, 1).reshape(3, -1)
    E_q, F_q = predictor.predict(R_query)
    out = os.path.join(HERE, 'big_n100_m2_s12.npz')
    np.savez_compressed(
        out,
        reference_version=sgdml.__version__,
        n_atoms=N,
        perms=perms,
        sig=sig,
        lam=task['lam'],
        z=task['z'],
        R_train=task['R_train'],
        tril_perms_lin=tril_perms_lin.astype(np.int64),
        R_desc=R_desc,
        R_d_desc=R_d_desc,
        K_cols=K_cols,
        cols=cols,
        alphas_F=alphas_F,
        R_d_desc_alpha=model['R_d_desc_alpha'],
        model_R_desc=model['R_desc'],
        std=model['std'],
        c=model['c'],
        R_query=R_query,
        E_query=E_q,
        F_query=F_q,
    )
    print('big_n100_m2_s12: K_cols', K_cols.shape, 'size %.0f KB' % (os.path.getsize(out) / 1024))


def main_dropin():
    """The reference's own command line (cli.py: create -> train -> test) on the synthetic dataset of
    tools/reference_cli_dropin.py, without the engine.  Stores the task the CLI created, the layout of the model
    file it wrote (keys, shapes, dtypes), c and std, the reference predictor's E / F from that file on the last 8
    dataset geometries and on every point outside the training and validation sets, and the parameter lists of
    the reference's GDMLTrain / GDMLPredict that the drop-in must reproduce."""
    import inspect
    import json
    import tempfile

    from sgdml import cli
    from sgdml.utils import io

    _tspec = importlib.util.spec_from_file_location('dropin', os.path.join(ROOT, 'tools', 'reference_cli_dropin.py'))
    dropin = importlib.util.module_from_spec(_tspec)
    _tspec.loader.exec_module(dropin)

    N, n_train, n_valid, n_test, sig = 9, 40, 20, 30, 20
    with tempfile.TemporaryDirectory() as wd:
        ds_path = os.path.join(wd, 'dataset.npz')
        dropin.make_dataset(ds_path, N, n_train + n_valid + n_test + 10)
        _, dataset = io.is_file_type(ds_path, 'dataset')
        np.random.seed(0)
        task_dir = os.path.join(wd, 'tasks')
        cli.create((ds_path, dataset), None, n_train, n_valid, [sig], False, True, False, True, task_dir=task_dir, command='create')
        task_files = sorted(f for f in os.listdir(task_dir) if f.startswith('task'))
        cli.train((task_dir, task_files), (ds_path, dataset), False, True, None, 1, False, command='train')
        model_files = sorted(f for f in os.listdir(task_dir) if f.startswith('model'))
        cli.test((task_dir, model_files), (ds_path, dataset), n_test, True, None, 1, False, command='test')
        with np.load(os.path.join(task_dir, task_files[0]), allow_pickle=True) as f:
            task = {k: f[k] for k in f.files}
        with np.load(os.path.join(task_dir, model_files[0]), allow_pickle=True) as f:
            model = {k: f[k] for k in f.files}

    predictor = GDMLPredict(model, max_processes=1, use_torch=False)
    n_data = dataset['R'].shape[0]
    R_query = dataset['R'][-8:].reshape(8, -1)
    E_q, F_q = predictor.predict(R_query)
    idxs_out = np.setdiff1d(np.arange(n_data), np.concatenate([task['idxs_train'], task['idxs_valid']]))
    R_out = dataset['R'][idxs_out].reshape(len(idxs_out), -1)
    E_out, F_out = predictor.predict(R_out)

    from sgdml.train import GDMLTrain as RefTrain

    sig_of = lambda f: list(inspect.signature(f).parameters)  # noqa: E731
    signatures = {
        'GDMLTrain.__init__': sig_of(RefTrain.__init__),
        'GDMLTrain.train': sig_of(RefTrain.train),
        'GDMLPredict.__init__': sig_of(GDMLPredict.__init__),
        'GDMLPredict.predict': sig_of(GDMLPredict.predict),
    }
    layout = {
        'keys': sorted(model.keys()),
        'shapes': {k: list(np.asarray(model[k]).shape) for k in ('R_desc', 'R_d_desc_alpha', 'alphas_F', 'perms', 'tril_perms_lin')},
        'dtypes': {k: str(np.asarray(model[k]).dtype) for k in ('R_desc', 'R_d_desc_alpha', 'alphas_F', 'perms', 'tril_perms_lin', 'sig', 'c', 'std')},
        'solver_name': str(model['solver_name']),
    }
    out = os.path.join(HERE, 'dropin_n9_m40.npz')
    np.savez_compressed(
        out,
        reference_version=sgdml.__version__,
        signatures=json.dumps(signatures),
        model_layout=json.dumps(layout),
        **{'task_' + k: v for k, v in task.items()},
        c=model['c'],
        std=model['std'],
        R_query=R_query,
        E_query=E_q,
        F_query=F_q,
        R_out=R_out,
        F_out_label=dataset['F'][idxs_out].reshape(len(idxs_out), -1),
        E_out=E_out,
        F_out=F_out,
    )
    print('dropin_n9_m40: %d training points, %d outside points, size %.0f KB' % (len(task['idxs_train']), len(idxs_out),
                                                                               os.path.getsize(out) / 1024))


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'dropin':
        main_dropin()  # separate process: the CLI's own GDMLTrain instances (train.py:336-342)
    elif len(sys.argv) > 1 and sys.argv[1] == 'n100':
        main_n100()
    elif len(sys.argv) > 1 and sys.argv[1] == 'c60':
        main_c60()
    elif len(sys.argv) > 1 and sys.argv[1] == 'pbc_ecstr':
        main_pbc_ecstr()
    elif len(sys.argv) > 1 and sys.argv[1] == 'iterative':
        main_iterative()   # separate process: the reference allows one GDMLTrain instance (train.py:336-342)
    else:
        main()
