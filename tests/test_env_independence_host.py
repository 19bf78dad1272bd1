"""CPU: the process environment selects no kernel, plan or launch attribute.

The routing of every kernel family -- ring, cluster-split (NFPB200_PATH_SPLIT), token (channels-last), planar band and
table, generic -- is queried through the C ABI in two fresh processes, one with a clean environment and one with every
former tuning variable set to a value other than its old default; the two answers must be identical.  A source check
keeps new environment reads out of the library and the Python layer."""
import ctypes
import itertools
import json
import os
import re
import subprocess
import sys

from neighbour_feature_pooling_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "neighbour_feature_pooling_b200")

# variables that used to pick plans, kernel variants or launch attributes, each with a value other than its old default
FORMER_SWITCHES = {
    "NFPB200_FUSED_IMPL": "split", "NFPB200_CHUNK_BYTES": "4096", "NFPB200_CTAS_PER_SM": "1",
    "NFPB200_NO_RESIDENT": "1", "NFPB200_PASSB_LANECH": "0", "NFPB200_RESIDENT_IMAGE": "0",
    "NFPB200_MAX_STAGES": "3", "NFPB200_BWD_DIRECT": "0", "NFPB200_Y_DELAY_NS": "1000", "NFPB200_Y_STAGES": "2",
    "NFPB200_PDL": "0", "NFPB200_UNIT_BYTES": "8192", "NFPB200_SUBCHUNKS": "2", "NFPB200_CLUSTER": "2",
    "NFPB200_MAX_CLUSTERS": "4", "NFPB200_PLANAR_SCALAR": "1", "NFPB200_PLANAR_TH": "4",
    "NFPB200_TOKEN_TWO_CTAS": "0", "NFPB200_X_STABLE_HINT": "1",
}

# (B, C, H, W, R, layout, inner_R, measure, padding_mode, stride): what each family takes for bf16 under path "auto"
SHAPES = [
    (256, 512, 7, 7, 1, 0, 0, "cosine", "reflect", 1),     # ring, more images than resident CTAs
    (4, 512, 7, 7, 1, 0, 0, "cosine", "zeros", 1),         # ring, one image per CTA (resident / per-lane tables)
    (8, 256, 14, 14, 1, 0, 0, "cosine", "replicate", 1),   # ring
    (4, 64, 2, 2, 1, 0, 0, "cosine", "reflect", 1),        # ring
    (3, 64, 4, 4, 1, 0, 0, "cosine", "reflect", 1),        # ring
    (4, 64, 7, 7, 2, 0, 0, "cosine", "reflect", 1),        # ring, 5x5
    (2, 32, 14, 14, 2, 0, 0, "cosine", "reflect", 1),      # ring, 5x5
    (3, 64, 7, 7, 2, 0, 1, "cosine", "reflect", 1),        # ring, multi-radius
    (256, 960, 7, 7, 1, 1, 0, "cosine", "reflect", 1),     # token
    (3, 64, 14, 14, 1, 1, 0, "cosine", "reflect", 1),      # token
    (3, 64, 7, 7, 2, 1, 1, "cosine", "reflect", 1),        # token, multi-radius
    (4, 64, 28, 28, 1, 0, 0, "cosine", "reflect", 1),      # band
    (2, 16, 112, 112, 1, 0, 0, "cosine", "reflect", 1),    # band
    (2, 16, 28, 28, 2, 0, 1, "cosine", "reflect", 1),      # band, multi-radius
    (2, 5, 3, 3, 1, 0, 0, "cosine", "reflect", 1),         # table
    (3, 20, 9, 6, 1, 0, 0, "cosine", "reflect", 1),        # table
    (2, 64, 7, 7, 1, 0, 0, "attention", "reflect", 1),     # generic
    (3, 5, 9, 11, 1, 0, 0, "cosine", "circular", 2),       # generic
]
DTYPES = (_capi.F32, _capi.BF16, _capi.F16)
PATHS = ("auto", "fused", "split", "generic")
OPS = (_capi.OP_FORWARD, _capi.OP_BACKWARD, _capi.OP_POOL_FORWARD, _capi.OP_POOL_BACKWARD,
       _capi.OP_POOLED_MAP_FORWARD, _capi.OP_POOLED_MAP_BACKWARD)


def _desc(shape, dtype, path):
    B, C, H, W, R, layout, inner, measure, mode, stride = shape
    return _capi.make_desc(dtype, B, C, H, W, R, stride, R, 1, mode, measure, True, False, 1e-6, 1, 1e-6, path,
                           layout=layout, inner_R=inner)


def _query(d, op):
    """[name, launch count, workspace bytes] of one op, or [status] where the op is refused."""
    lib = _capi.load()
    buf = ctypes.create_string_buffer(128)
    rc = lib.nfpb200_describe_path(ctypes.byref(d), op, buf, 128)
    if rc:
        return [rc]
    return [buf.value.decode(), _capi.launch_count(d, op), _capi.workspace_bytes(d, op)]


def routing_table():
    """{"shape/dtype/path": {"head": head_supported, op: query}} over the whole grid."""
    lib = _capi.load()
    out = {}
    for (si, s), dt, path in itertools.product(enumerate(SHAPES), DTYPES, PATHS):
        d = _desc(s, dt, path)
        cell = {"head": lib.nfpb200_head_supported(ctypes.byref(d))}
        cell.update({str(op): _query(d, op) for op in OPS})
        out[f"{si}/{dt}/{path}"] = cell
    return out


_CHILD = "import json, test_env_independence_host as T; print(json.dumps(T.routing_table(), sort_keys=True))"


def _table_in_subprocess(extra_env):
    env = {k: v for k, v in os.environ.items() if k not in FORMER_SWITCHES}
    env.update(extra_env, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    r = subprocess.run([sys.executable, "-c", _CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_grid_reaches_every_family():
    names = {q[0] for cell in routing_table().values() for k, q in cell.items() if k != "head" and len(q) == 3}
    for prefix in ("fused/stream_", "fused/split_", "fused/token_", "planar/band", "planar/table", "generic/pairs"):
        assert any(n.startswith(prefix) for n in names), (prefix, sorted(names))


def test_routing_ignores_former_tuning_variables():
    clean = _table_in_subprocess({})
    switched = _table_in_subprocess(FORMER_SWITCHES)
    diff = sorted(k for k in clean if clean[k] != switched.get(k))
    assert not diff and clean.keys() == switched.keys(), [(k, clean[k], switched.get(k)) for k in diff[:5]]


def test_no_environment_reads_in_sources():
    # the library: only the launch-failure diagnostics, which change no result
    csrc = os.path.join(PKG, "csrc")
    for name in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, name)) as f:
            src = f.read()
        calls = re.findall(r"\bgetenv\b\s*\(([^)]*)\)", src)
        assert len(calls) == len(re.findall(r"\bgetenv\b", src)), name
        assert all(c.strip() == '"NFPB200_VERBOSE"' for c in calls), (name, calls)
    # the Python layer: which library build to load (NFPB200_LIB), the compiler to build with (NVCC) and the torchrun
    # variables; no NFPB200_* variable besides NFPB200_LIB
    allowed = {"NFPB200_LIB", "NVCC", "RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR"}
    read = re.compile(r"\bos\.(?:environ\.get|environ\.setdefault|getenv)\(\s*\"(\w+)\"|\bos\.environ\[\s*\"(\w+)\"\s*\]")
    for name in sorted(f for f in os.listdir(PKG) if f.endswith(".py")):
        with open(os.path.join(PKG, name)) as f:
            src = f.read()
        keys = [a or b for a, b in read.findall(src)]
        assert len(keys) == len(re.findall(r"\b(?:environ|getenv)\b", src)), name
        assert set(keys) <= allowed, (name, sorted(set(keys) - allowed))
