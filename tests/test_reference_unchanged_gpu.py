"""The reference's own training.py and model.py, UNMODIFIED, running on the drop-in modules
(north_star: "the existing training.py and model.py consume it unchanged"; reference training.py:12-14, 355-517).

The reference (kurtosis/mat_mul) is third-party code that this repository does not ship.  `scripts/install_ref.sh
<checkout>` copies its scripts into the git-ignored baseline/_ref/, and tests/golden/ref_sha256.json pins the contents
this project was tested against.  Without that copy both tests skip and say why; the drop-in's values are still checked
against vectors drawn from the reference (tests/golden/, test_dropin_gpu.py, test_buffers_gpu.py).  The test registers
mat_mul_b200.{utils,datasets,act} under the reference's module names (dropin.install), imports the reference's
training module and runs TensorGameTrainingApp for one tiny epoch: dataset construction (create_synthetic_demo,
TensorGameDataset, SyntheticDemoDataset), a train step and a validation step through DataLoader + model.fwd_train, an
act step through actor_prediction / MCTS (model.fwd_infer + get_child_states ...) and the replay buffers."""
import hashlib
import json
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
REF = ROOT / "baseline" / "_ref"
PINS = ROOT / "tests" / "golden" / "ref_sha256.json"
NOT_INSTALLED = ("needs the reference's own scripts in baseline/_ref/: third-party code (kurtosis/mat_mul) that this "
                 "repository does not ship; install a checkout with scripts/install_ref.sh <checkout>")


def _installed() -> bool:
    return (REF / "training.py").exists() and (REF / "model.py").exists()


def test_reference_copy_is_unmodified():
    if not _installed():
        pytest.skip(NOT_INSTALLED)
    pins = json.loads(PINS.read_text())
    for name in ("training.py", "model.py", "utils.py", "datasets.py", "act.py"):
        assert hashlib.sha256((REF / name).read_bytes()).hexdigest() == pins[name], f"{name} differs from the reference"


@pytest.mark.gpu
def test_reference_training_app_runs_on_the_dropin(tmp_path, monkeypatch):
    if not _installed():
        pytest.skip(NOT_INSTALLED)
    import numpy as np
    import torch

    import mat_mul_b200.dropin as dropin
    from mat_mul_b200 import _lib
    from mat_mul_b200 import datasets as tg_datasets

    monkeypatch.chdir(tmp_path)  # the reference writes data_unversioned/ and runs/ under the cwd
    # save_model mkdirs non-recursively (training.py:178): the parent has to exist, as in the author's checkout
    (tmp_path / "data_unversioned" / "models").mkdir(parents=True)
    monkeypatch.setattr(sys, "argv", ["training.py", "--len_data", "64", "--n_epochs", "1", "--n_games", "2", "--max_actions", "3",
                                      "--n_sim", "2", "--batch_size", "32", "--n_val", "1", "--n_act", "1", "--device", "cpu"])
    monkeypatch.syspath_prepend(str(REF))  # model.py and training.py come from the reference ...
    for name in ("training", "model", "utils", "datasets", "act"):
        monkeypatch.delitem(sys.modules, name, raising=False)
    dropin.install()  # ... utils / datasets / act from this package
    try:
        import training  # the reference's module, star-importing the drop-in

        assert Path(training.__file__).resolve().parent == REF.resolve()
        assert training.SyntheticDemoDataset is tg_datasets.SyntheticDemoDataset
        assert training.AlphaTensor.__module__ == "model"
        torch.manual_seed(0)
        np.random.seed(0)
        app = training.TensorGameTrainingApp()
        assert isinstance(app.dataset, tg_datasets.TensorGameDataset)
        assert app.dataset_val._slab.is_cuda  # the demo store lives in HBM
        before = [p.detach().clone() for p in app.model.parameters()]
        app.main()
        # one optimizer step happened, two games were played and stored, the best one was kept
        assert any(not torch.equal(a, b.detach()) for a, b in zip(before, app.model.parameters()))
        assert app.training_samples_count == 64
        assert len(app.dataset.buffer_played.game_lengths) == 2 and len(app.dataset.buffer_best.game_lengths) == 1
        st, sc, ac, rw = app.dataset.buffer_played[0]
        assert st.shape == (2, 4, 4, 4) and ac.shape == (12,) and rw.shape == (1,)
        assert list((tmp_path / "data_unversioned" / "models" / "tensor_game").glob("*.pt"))
        # and the kernels were what ran: the library is loaded from the tree
        assert _lib.LIB_PATH.exists() and _lib.lib().tg_version() == _lib.header_version()
    finally:
        dropin.uninstall()
        for name in ("training", "model"):
            sys.modules.pop(name, None)
