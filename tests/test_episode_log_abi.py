"""CPU: the episode log's C ABI (ssd_episode_record, ssd_episode_log, ssd_set_episode_log) as the bindings declare it."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_fields(struct):
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.sub(r"\[.*\]|[\*\s]", "", d.strip().split()[-1]) for d in body.split(";") if d.strip()]


def test_episode_structs_match_header():
    """ctypes mirrors have the field order of the header; a record is 480 bytes with its metrics at byte 32."""
    from contracts_b200 import _lib
    assert _header_fields("ssd_episode_record") == [f[0] for f in _lib.ssd_episode_record._fields_]
    assert _header_fields("ssd_episode_log") == [f[0] for f in _lib.ssd_episode_log._fields_]
    assert ctypes.sizeof(_lib.ssd_episode_record) == 480
    assert _lib.ssd_episode_record.metrics.offset == 32 and _lib.ssd_episode_record.theta.offset == 16
    assert ctypes.sizeof(_lib.ssd_episode_log) == 24


def test_record_dtype_matches_struct():
    """The numpy view EpisodeLog.drain reads the records through has the struct's offsets."""
    from contracts_b200 import _lib
    from contracts_b200.episodes import RECORD_DTYPE
    assert RECORD_DTYPE.itemsize == ctypes.sizeof(_lib.ssd_episode_record)
    for name, _ in _lib.ssd_episode_record._fields_:
        assert RECORD_DTYPE.fields[name][1] == getattr(_lib.ssd_episode_record, name).offset, name


def test_set_episode_log_rejects_null_handle():
    """No device needed: a NULL handle is SSD_EINVAL, with or without a struct."""
    from contracts_b200 import _lib
    lib = _lib.load()
    log = _lib.ssd_episode_log(struct_size=ctypes.sizeof(_lib.ssd_episode_log), capacity=1, records_dev=None, count_dev=None)
    assert lib.ssd_set_episode_log(None, None) == -1
    assert lib.ssd_set_episode_log(None, ctypes.byref(log)) == -1
