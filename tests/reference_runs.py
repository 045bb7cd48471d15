"""Stored answers of the reference's own drivers, so that the tests that compare with the reference run from the repository alone.

The drivers under oracle/_ref/ (oracle/Makefile.ref, oracle/Makefile.drivers) link the unmodified reference and can only be built where
its sources are.  A test asks `reference_run(driver, args)` instead of running one.  Where oracle/_ref/<driver> is built, the driver
runs, as it always did.  Elsewhere the answer - the driver's stdout and every file it wrote at a path named in `args` - comes from
tests/golden/reference_runs/<driver>.json.xz, looked up by the driver's name, its arguments, the contents of the input files they and
its environment variables name (not their paths) and the contents of the repository sources oracle/Makefile.drivers compiles into it:
an answer recorded before one of those sources changed is not found, and the test fails asking for it to be recorded again.
libkgb200, which some drivers evaluate on, is the code under test and not part of the key.

To record, run the tests that call it with KGB_RECORD_REFERENCE=<directory> where the drivers are built (the GPU tests' drivers
evaluate on libkgb200 and need a B200): every query then runs the driver and is added to <directory>/<driver>.json.xz, which is
copied to tests/golden/reference_runs/.
"""
import base64
import hashlib
import json
import lzma
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STORE = os.path.join(ROOT, "tests", "golden", "reference_runs")
_cache = {}


def _load(store, driver):
    path = os.path.join(store, f"{driver}.json.xz")
    if path not in _cache:
        _cache[path] = json.loads(lzma.open(path).read()) if os.path.exists(path) else {}
    return path, _cache[path]


def _part(a):
    """An argument naming an existing file stands for its contents; a path the driver is to write stands for nothing but its place."""
    if os.path.isfile(a):
        return "file:" + hashlib.sha256(open(a, "rb").read()).hexdigest()
    return "path" if os.path.isabs(a) else a


def _sources(driver):
    """The repository files oracle/Makefile.drivers lists as prerequisites of oracle/_ref/<driver>, through the objects it links
    (libkgref.a, the reference itself, has its rule in oracle/Makefile.ref)."""
    rules = {}
    for ln in open(os.path.join(ROOT, "oracle", "Makefile.drivers")):
        m = re.match(r"\$\(OUT\)/(\S+):\s*(.*)$", ln)
        if m:
            rules[m.group(1)] = m.group(2).split()
    if driver not in rules:
        raise KeyError(f"oracle/Makefile.drivers has no rule for {driver}")
    found, todo = [], [driver]
    while todo:
        for dep in rules.get(todo.pop(), []):
            if dep.startswith("$(OUT)/"):
                todo.append(dep[len("$(OUT)/"):])
            elif not dep.endswith(".so") and dep not in found:
                found.append(dep)
    return sorted(found)


def _paths(args, env):
    """Where the driver may read or write files: its arguments and its environment variables, by name."""
    return [(str(i), a) for i, a in enumerate(args)] + [("env:" + k, v) for k, v in sorted(env.items())]


def reference_run(driver, args, env=None, timeout=600):
    """stdout of `oracle/_ref/<driver> args...` with `env` added to the environment; the files it wrote at paths named in `args` or `env`."""
    args, env = [str(a) for a in args], {k: str(v) for k, v in (env or {}).items()}
    sources = hashlib.sha256(b"".join(open(os.path.join(ROOT, f), "rb").read() for f in _sources(driver))).hexdigest()
    key = json.dumps([driver, "sources:" + sources, [_part(a) for _, a in _paths(args, env)]])
    where = dict(_paths(args, env))
    exe = os.path.join(ROOT, "oracle", "_ref", driver)
    record = os.environ.get("KGB_RECORD_REFERENCE")
    if not record and not os.path.exists(exe):
        _, runs = _load(STORE, driver)
        if key not in runs:
            raise KeyError(f"no stored reference answer for {driver} {' '.join(args)} with the present sources {_sources(driver)}: "
                           "record it (tests/reference_runs.py)")
        hit = runs[key]
        for name, data in hit["files"].items():
            with open(where[name], "wb") as f:
                f.write(data["text"].encode() if "text" in data else base64.b64decode(data["b64"]))
        return hit["stdout"]
    before = {name for name, a in where.items() if os.path.exists(a)}
    r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=timeout, env=dict(os.environ, **env))
    if r.returncode != 0:
        raise RuntimeError(f"{driver} failed: {r.stderr[-2000:]}")
    if record:
        files = {}
        for name, a in where.items():
            if name not in before and os.path.isfile(a):
                data = open(a, "rb").read()
                try:
                    files[name] = {"text": data.decode()}
                except UnicodeDecodeError:
                    files[name] = {"b64": base64.b64encode(data).decode()}
        path, runs = _load(record, driver)
        runs[key] = {"stdout": r.stdout, "files": files}
        os.makedirs(record, exist_ok=True)
        with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
            f.write(json.dumps(runs, sort_keys=True).encode())
    return r.stdout
