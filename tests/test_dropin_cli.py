"""(f)1 -- the engine as a drop-in behind the reference's own CLI (north_star; INTEGRATION.md section 4).
The reference's side is frozen in tests/golden/dropin_n9_m40.npz (make_golden.py dropin): the task its CLI created
(`sgdml create`), the layout of the model file its `sgdml train` / `sgdml test` wrote, the predictions of that model
by its own GDMLPredict, and the parameter lists of its GDMLTrain / GDMLPredict."""

import inspect
import json
import sys
import types

import numpy as np
import pytest

from conftest import load_golden, rel_err


@pytest.fixture(scope='module')
def dropin():
    g = load_golden('dropin_n9_m40')
    g['signatures'] = json.loads(str(g['signatures']))
    g['model_layout'] = json.loads(str(g['model_layout']))
    return g


def _stand_in_reference(monkeypatch):
    """A package laid out like the reference (sgdml.cli, sgdml.train) with the host-side task functions the
    installed training class borrows."""

    class RefTrain(object):
        def create_task(self, *a, **k):
            pass

        def create_task_from_model(self, *a, **k):
            pass

        def draw_strat_sample(self, *a, **k):
            pass

    pkg = types.ModuleType('sgdml_stand_in')
    pkg.__path__ = []
    pkg.cli = types.ModuleType('sgdml_stand_in.cli')
    pkg.train = types.ModuleType('sgdml_stand_in.train')
    pkg.cli.GDMLTrain, pkg.cli.GDMLPredict = RefTrain, object
    pkg.train.GDMLTrain = RefTrain
    for mod in (pkg, pkg.cli, pkg.train):
        monkeypatch.setitem(sys.modules, mod.__name__, mod)
    return pkg, RefTrain


def test_install_rebinds_reference_cli_and_signatures_match(monkeypatch, dropin):
    """CPU: the two names the reference CLI instantiates are rebound; constructor / train / predict signatures of
    the engine classes equal the reference's (train.py:306, 836-841; predict.py:249-258, 1146)."""
    from sgdml_b200.integration import install_into_reference

    pkg, RefTrain = _stand_in_reference(monkeypatch)
    T, P = install_into_reference(pkg)
    assert pkg.cli.GDMLTrain is T and pkg.cli.GDMLPredict is P
    assert T.create_task is RefTrain.create_task and T.draw_strat_sample is RefTrain.draw_strat_sample
    assert T.create_task_from_model is RefTrain.create_task_from_model

    sig = lambda f: list(inspect.signature(f).parameters)  # noqa: E731
    ref = dropin['signatures']
    assert sig(T.__init__) == ref['GDMLTrain.__init__']
    assert sig(T.train) == ref['GDMLTrain.train']
    assert sig(P.__init__) == ref['GDMLPredict.__init__']
    assert sig(P.predict)[:3] == ref['GDMLPredict.predict'][:3]


@pytest.mark.gpu
def test_reference_cli_train_and_test_through_engine(tmp_path, dropin):
    """The task the reference's `sgdml create` wrote, trained by the engine: the model file has the keys / shapes /
    dtypes of the one the reference's `sgdml train` wrote, read back by a CPU predictor it predicts what the
    reference-trained model predicts (1e-6 rel, north_star), and its force error on the points outside the training
    and validation sets agrees with the reference model's."""
    import sgdml_b200
    from oracle import predict as opredict

    g = dropin
    task = {k[len('task_'):]: g[k] for k in g if k.startswith('task_')}
    model = sgdml_b200.GDMLTrain().train(task)
    path = tmp_path / 'model.npz'
    np.savez_compressed(path, **model)  # as cli.py:1098 writes it
    with np.load(path, allow_pickle=True) as f:
        model = {k: f[k] for k in f.files}

    ref = g['model_layout']
    assert sorted(model.keys()) == ref['keys']
    assert {k: list(np.asarray(model[k]).shape) for k in ref['shapes']} == ref['shapes']
    assert {k: str(np.asarray(model[k]).dtype) for k in ref['dtypes']} == ref['dtypes']
    assert str(model['solver_name']) == ref['solver_name'] == 'analytic'
    c, std = float(model['c']), float(model['std'])
    assert abs(c - float(g['c'])) < 1e-6 * abs(float(g['c'])) and abs(std - float(g['std'])) < 1e-12 * float(g['std'])

    E, F = opredict.Predictor(model).predict(g['R_query'])
    assert rel_err(E, g['E_query']) < 1e-6
    assert rel_err(F, g['F_query']) < 1e-6

    # force error on the held-out points, as `sgdml test` records it (cli.py:1502-1570), through the engine predictor
    _, F_out = sgdml_b200.GDMLPredict(model).predict(g['R_out'])
    assert rel_err(F_out, g['F_out']) < 1e-6
    rmse = np.sqrt(np.mean((F_out - g['F_out_label']) ** 2))
    rmse_ref = np.sqrt(np.mean((g['F_out'] - g['F_out_label']) ** 2))
    assert abs(rmse - rmse_ref) < 1e-6 + 0.05 * rmse_ref
