import sys, time, tempfile, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from recommender_tensorflow_b200.trainers import ml_100k
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.csv_reader import GpuCsvReader
fc = ml_100k.get_feature_columns(16)
eng = DeepFMEngine(fc["linear"], (), embedding_size=16, hidden_units=(256, 128), feature_dtypes=ml_100k.FEATURE_DTYPES, max_batch=65536)
path = os.path.join(tempfile.mkdtemp(), "t.csv")
ml_100k.write_synthetic_csv(path, 65536)
data = np.fromfile(path, dtype=np.uint8)
hdr = int(np.flatnonzero(data == 10)[0]) + 1
body = data[hdr:]
print("records 65536 bytes", body.size, "bytes/record", body.size / 65536)
rd = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, max_records=65536, max_bytes=body.size + 64)
pad = (body.size + 15) // 16 * 16
dev = torch.zeros(pad, dtype=torch.uint8, device="cuda")
dev[:body.size] = torch.from_numpy(body.copy()).cuda()
pinned = torch.from_numpy(body.copy()).pin_memory()
for name, src in (("device text", dev[:body.size]), ("pinned host text", pinned)):
    for _ in range(3):
        pb = rd.decode(src)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(20):
        pb = rd.decode(src)
    torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 20
    print("%s: %.3f ms/batch  %.1f M records/s  %.1f GB/s of text" % (name, dt * 1e3, 65536 / dt / 1e6, body.size / dt / 1e9))
