"""Records the calls the original project's ``examples/basic_example.py`` makes into ``neutts`` and ``soundfile``
and writes them to tests/golden/basic_example_calls.json, which tests/test_host_logic.py replays against this
package.  Run it with the original project's checkout (pure Python; nothing is downloaded):

    python oracle/record_example_calls.py <original project directory>

The example runs unmodified against stand-ins for the two modules that log every call.  Paths inside the scratch
directory are stored as ``{tmp}/<name>``; a value one call returned and a later call received is stored as
``{"$ret": <index of the call that returned it>}``.
"""
import importlib.util
import json
import os
import shutil
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "basic_example_calls.json")


def record(project_dir: str) -> dict:
    tmp = tempfile.mkdtemp()
    files = {"dave.txt": "hello there\n"}
    for name, text in files.items():
        with open(os.path.join(tmp, name), "w") as f:
            f.write(text)
    calls = []

    class Ret:
        def __init__(self, i):
            self.i = i

    def enc(v):
        if isinstance(v, Ret):
            return {"$ret": v.i}
        return v.replace(tmp, "{tmp}") if isinstance(v, str) else v

    def log(name, args, kwargs):
        calls.append({"call": name, "args": [enc(a) for a in args], "kwargs": {k: enc(v) for k, v in kwargs.items()}})
        return Ret(len(calls) - 1)

    class NeuTTS:
        def __init__(self, *args, **kwargs):
            log("neutts.NeuTTS", args, kwargs)

        def __getattr__(self, name):
            return lambda *args, **kwargs: log("NeuTTS." + name, args, kwargs)

    neutts = types.ModuleType("neutts")
    neutts.NeuTTS = NeuTTS
    sf = types.ModuleType("soundfile")
    sf.write = lambda *args, **kwargs: log("soundfile.write", args, kwargs)
    saved = {k: sys.modules.get(k) for k in ("neutts", "soundfile")}
    sys.modules.update(neutts=neutts, soundfile=sf)
    try:
        spec = importlib.util.spec_from_file_location("basic_example", os.path.join(project_dir, "examples", "basic_example.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        main_args = ["Testing.", f"{tmp}/dave.wav", f"{tmp}/dave.txt", "neuphonic/neutts-air"]
        main_kwargs = {"output_path": f"{tmp}/out.wav"}
        mod.main(*main_args, **main_kwargs)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        shutil.rmtree(tmp)
    return {"example": "examples/basic_example.py", "main": {"args": [enc(a) for a in main_args],
                                                              "kwargs": {k: enc(v) for k, v in main_kwargs.items()}},
            "files": files, "calls": calls}


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    with open(OUT, "w") as f:
        json.dump(record(sys.argv[1]), f, indent=1)
        f.write("\n")
    print("wrote", OUT)
