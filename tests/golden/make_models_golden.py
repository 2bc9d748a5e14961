"""Stores the values of the original project's model files (models/model_*_params.yaml: type, frequency and the flat Q, R, P
lists, as PyYAML parses them) in tests/golden/reference_models.npz, so that tests/test_models.py can check models/*.yaml against
them where the original project is not at hand.

    python tests/golden/make_models_golden.py <models directory of the original project>

The committed file was written from this repository's models/, whose files tests/test_models.py::
test_models_bit_identical_to_reference had found equal, value for value, to the original's (the files are unchanged since)."""
import os
import sys

import numpy as np
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
NAMES = ["uniform_velocity", "uniform_acceleration", "angular_velocities", "angular_rates"]

if __name__ == "__main__":
    src = sys.argv[1]
    out = {}
    for name in NAMES:
        with open(os.path.join(src, "model_%s_params.yaml" % name)) as f:
            doc = yaml.safe_load(f)
        out[name + "/type"] = np.array(doc["type"])
        out[name + "/frequency"] = np.array(float(doc["frequency"]))
        for k in "QRP":
            out[name + "/" + k] = np.array(doc[k], dtype=np.float64)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "reference_models.npz"), **out)
