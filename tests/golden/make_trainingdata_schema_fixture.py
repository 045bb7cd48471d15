"""tests/golden/trainingdata_schema.json: dtype and per-row shape of every array in the reference's own sample training file
(python/testdata/benchmark_data_1024.npz of the reference, whose directory $KATAGO_REF names)."""
import json, os
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
d = np.load(os.path.join(os.environ["KATAGO_REF"], "python", "testdata", "benchmark_data_1024.npz"))
with open(os.path.join(HERE, "trainingdata_schema.json"), "w") as f:
    f.write("{\n" + ",\n".join(f" {json.dumps(k)}: {json.dumps([d[k].dtype.str, list(d[k].shape[1:])])}" for k in sorted(d.files)) + "\n}\n")
