"""The Zstandard SST writer without a GPU: tests/test_gpu_zstd_writer.py on the emulated build of the library (see test_emu_engine.py),
files written under different thread orders compared byte for byte, and the storage layer's routing of `compression = Zstd`."""
import hashlib
import os
import subprocess
import sys

import pytest

from horaedb_b200.config import StorageConfig, WriteConfig
from horaedb_b200.storage import ObjectBasedStorage, Task, WriteRequest
from horaedb_b200.types import TimeRange

from helpers import arrow_schema, record_batch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def _env(order, guard=False):
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_engine_emu
    build_engine_emu.build()
    env = dict(os.environ)
    env["PYTHONPATH"] = os.path.join(ROOT, "tests", "emu") + os.pathsep + ROOT + os.pathsep + env.get("PYTHONPATH", "")
    env["HORAE_EMU_ORDER"] = str(order)
    env["HORAE_EMU_CRASH_REPORT"] = "1"
    if guard:
        env["HORAE_EMU_GUARD"] = "1"
    return env


@pytest.mark.parametrize("order,guard", [(0, True), (2, False)])
def test_gpu_zstd_writer_tests_on_the_emulated_library(order, guard):
    cmd = [sys.executable, "-m", "pytest", "-p", "emu_plugin", "-m", "gpu", "-q", "-p", "no:cacheprovider", "tests/test_gpu_zstd_writer.py"]
    r = subprocess.run(cmd, cwd=ROOT, env=_env(order, guard), capture_output=True, text=True, timeout=1500)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-40:])
    assert r.returncode == 0 and " passed" in tail and "failed" not in tail, tail


# writes a compaction and a write_batch with Zstd on the emulated library into argv[1] (same inputs every run)
_WRITE = r"""
import sys
import build_engine_emu
from horaedb_b200 import _ffi
_ffi.LIB_PATH = build_engine_emu.build(); _ffi._lib = None
import ctypes, os
ctypes.CDLL(_ffi.LIB_PATH).emu_set_order(int(os.environ["HORAE_EMU_ORDER"]))
from horaedb_b200 import sstgen
from horaedb_b200._ffi import Engine, SchemaHandle, SstInput
schema = sstgen.metric_storage_schema()
h = SchemaHandle(schema.arrow_schema, 2)
datas = [s[0] for s in sstgen.synth_overlapping_ssts(4, series=50, points=600, delta_ms=1000, keep_frac=0.5, compression="none")]
eng = Engine(device=0)
eng.compact_to_sst(h, [SstInput(id=i + 1, data=d, time_start=0, time_end=1, max_sequence=10 + i) for i, d in enumerate(datas)],
                   sys.argv[1] + "/c.sst", max_row_group_size=5000, compression="zstd")
import io
import pyarrow as pa, pyarrow.parquet as pq
t = pa.concat_tables([pq.read_table(io.BytesIO(d)) for d in datas])
user = pa.schema([f for f in t.schema if not f.name.startswith("__")])
b = pa.Table.from_arrays([t[n] for n in user.names], schema=user).combine_chunks().to_batches()[0]
eng.write_batch(h, b, 99, sys.argv[1] + "/w.sst", compression="zstd")
eng.close()
"""


def test_zstd_files_are_identical_under_every_thread_order(tmp_path):
    digests = []
    for order in (0, 2, 1):
        d = tmp_path / f"o{order}"
        d.mkdir()
        r = subprocess.run([sys.executable, "-c", _WRITE, str(d)], cwd=ROOT, env=_env(order), capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout + r.stderr
        digests.append([hashlib.sha256((d / f).read_bytes()).hexdigest() for f in ("c.sst", "w.sst")])
    assert digests[0] == digests[1] == digests[2]


class _Recorder:
    """an engine that records the writer calls storage.py makes (without write_batch: the host writes new files)"""
    def __init__(self):
        self.calls = []

    def compact_to_sst(self, handle, inputs, out_path, **kw):
        self.calls.append(("compact_to_sst", kw))
        raise RuntimeError("recorded")

    def compact(self, handle, inputs):
        self.calls.append(("compact", {}))
        raise RuntimeError("recorded")

    def unload_sst(self, id):
        pass


class _GpuWriteRecorder(_Recorder):
    def write_batch(self, handle, batch, file_id, path, **kw):
        self.calls.append(("write_batch", kw))
        raise RuntimeError("recorded")


def test_storage_sends_zstd_to_the_gpu_writer(tmp_path):
    user = arrow_schema([("pk1", "uint8"), ("pk2", "uint8"), ("value", "int64")])
    cfg = StorageConfig(write=WriteConfig(compression="zstd"))
    want = {"max_row_group_size": 8192, "compression": "zstd", "enable_sorting_columns": True}
    b = record_batch(user, {"pk1": [1], "pk2": [0], "value": [1]})
    eng = _GpuWriteRecorder()
    st = ObjectBasedStorage(str(tmp_path / "a"), 100, user, 2, cfg, engine=eng)
    with pytest.raises(RuntimeError, match="recorded"):
        st.write(WriteRequest(b, TimeRange(0, 10)))
    assert eng.calls == [("write_batch", want)]
    eng = _Recorder()
    st = ObjectBasedStorage(str(tmp_path / "b"), 100, user, 2, cfg, engine=eng)
    st.write(WriteRequest(b, TimeRange(0, 10)))
    st.write(WriteRequest(b, TimeRange(10, 20)))
    files = st.manifest.all_ssts()
    for f in files:
        f.mark_compaction()
    with pytest.raises(RuntimeError, match="recorded"):
        st.do_compaction(Task(files))
    assert eng.calls == [("compact_to_sst", want)]
    # Zstd with dictionary encoding stays on the host path
    st.config.write.enable_dict = True
    for f in files:
        f.mark_compaction()
    with pytest.raises(RuntimeError, match="recorded"):
        st.do_compaction(Task(files))
    assert eng.calls[-1][0] == "compact"
