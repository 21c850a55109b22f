"""ORACLE recipe (test infrastructure, not product code): the REFERENCE ITSELF for the
memory-save path, compiled from where its sources lie under /root/reference into
oracle/_ref/pyref/ — byte code only (sourceless .pyc), git-ignored, not gpurun-ignored, so it
travels to the GPU box like oracle/_ref/libpack_oracle.so.  No reference source is copied.

    python oracle/build_ref.py            (also: make -C oracle pyref; __graft_entry__.build())

What gets compiled is found, not listed: a clean interpreter imports
dlrover/python/elastic_agent/torch/ckpt_saver.py from /root/reference, runs one tiny
SharedMemoryHandler.save_state_dict + load_state_dict (ckpt_saver.py:303-366) so that lazily
imported modules are loaded too, and reports every module it loaded from the source tree.
Then the reference's own agent (AsyncCheckpointSaver) and trainer (DdpCheckpointer) run one
session against each other in two more interpreters — a memory save, a load, a disk save and
the wait for its persist — and report theirs too.  Each module of the union is compiled with py_compile to the mirrored path under pyref/
(`x/y.py` -> `x/y.pyc`, `__init__.py` -> `__init__.pyc`), which Python imports without the
source.  MANIFEST.json records the files and the sha256 of the source each came from.

Used by oracle/ref_real.py (bench.py's `--impl reference` arm and `cpu_baseline`:
kind "reference"), by tests/test_oracle.py to pin ref_port.py / shm_layout.py to it, and by
tests/test_wire_compat.py, which runs the reference's agent and trainer from it against ours.
"""

from __future__ import annotations

import hashlib
import json
import os
import py_compile
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.environ.get("FC_REFERENCE_ROOT", "/root/reference")
OUT = os.path.join(HERE, "_ref", "pyref")

PROBE = r"""
import json, os, sys
sys.path.insert(0, sys.argv[1])
os.environ.setdefault("ROLE_NAME", "dlrover-trainer")
os.environ["TORCHELASTIC_RUN_ID"] = "fcbuildref%d" % os.getpid()
import logging
logging.disable(logging.CRITICAL)
import torch
from dlrover.python.elastic_agent.torch import ckpt_saver as ref
h = ref.SharedMemoryHandler(97, host=True)
sd = {"m": {"w": torch.arange(6, dtype=torch.float32).reshape(2, 3), "n": 3},
      ref.DLROVER_CKPT_CONFIG_KEY: ref.CheckpointConfig(step=1, paths={})}
h.save_state_dict(sd)
back = h.load_state_dict()
assert torch.equal(back["m"]["w"], sd["m"]["w"]) and back["m"]["n"] == 3
del back
h.unlink()
h.close()
"""

REPORT = r"""
root = os.path.realpath(sys.argv[1]) + os.sep
mods = sorted({os.path.realpath(m.__file__) for m in list(sys.modules.values())
               if getattr(m, "__file__", None)
               and os.path.realpath(m.__file__).startswith(root)
               and m.__file__.endswith(".py")})
print("FCREF " + json.dumps(mods), flush=True)
os._exit(0)
"""

SESSION_AGENT = r"""
import json, os, sys
from unittest import mock
sys.path.insert(0, sys.argv[1])
sys.modules.setdefault("kubernetes", mock.MagicMock())
import logging
logging.disable(logging.CRITICAL)
from dlrover.python.elastic_agent.torch.ckpt_saver import AsyncCheckpointSaver
AsyncCheckpointSaver.start_async_saving_ckpt()
print("AGENT_READY", flush=True)
sys.stdin.readline()                      # the trainer is done
""" + REPORT

SESSION_TRAINER = r"""
import json, os, sys
from unittest import mock
sys.path.insert(0, sys.argv[1])
sys.modules.setdefault("kubernetes", mock.MagicMock())
import logging
logging.disable(logging.CRITICAL)
import torch
from dlrover.trainer.torch.flash_checkpoint.ddp import DdpCheckpointer, StorageType
d = sys.argv[2]
ckpt = DdpCheckpointer(d)
sd = {"w": torch.arange(10, dtype=torch.float32), "step": 1}
ckpt.save_checkpoint(1, sd, storage_type=StorageType.MEMORY)
back = ckpt.load_checkpoint()
assert torch.equal(back["w"], sd["w"])
del back
ckpt.save_checkpoint(2, sd, storage_type=StorageType.DISK)
ckpt.wait_latest_checkpoint(timeout=60)
assert open(os.path.join(d, "dlrover_latest.txt")).read() == "2"
""" + REPORT


def _modules(out: str, what: str, rc: int, err: str):
    marker = [ln for ln in out.splitlines() if ln.startswith("FCREF ")]
    if rc != 0 or not marker:
        raise RuntimeError(f"reference {what} probe failed ({rc}):\n{err[-2000:]}")
    return json.loads(marker[-1][len("FCREF "):])


def _session(env) -> list:
    """Modules the reference's agent and trainer load in one session against each other."""
    import tempfile
    import uuid

    run_id = "fcbuildref" + uuid.uuid4().hex[:8]
    env = dict(env, TORCHELASTIC_RUN_ID=run_id, ROLE_NAME="dlrover-trainer")
    with tempfile.TemporaryDirectory() as ckpt_dir:
        agent = subprocess.Popen([sys.executable, "-c", SESSION_AGENT, REFERENCE],
                                 env=env, cwd="/tmp", stdin=subprocess.PIPE,
                                 stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        try:
            if "AGENT_READY" not in agent.stdout.readline():
                raise RuntimeError(f"reference agent probe failed:\n{agent.stderr.read()[-2000:]}")
            t = subprocess.run([sys.executable, "-c", SESSION_TRAINER, REFERENCE, ckpt_dir],
                               env=env, cwd="/tmp", capture_output=True, text=True, timeout=300)
            files = _modules(t.stdout, "trainer", t.returncode, t.stderr)
            out, err = agent.communicate("done\n", timeout=60)
            files += _modules(out, "agent", agent.returncode, err)
        finally:
            if agent.poll() is None:
                agent.kill()
                agent.wait()
            shutil.rmtree(os.path.join("/tmp/ckpt_sock", run_id), ignore_errors=True)
            for f in os.listdir("/dev/shm"):
                if f.startswith(run_id):
                    os.unlink(os.path.join("/dev/shm", f))
    return files


def build(verbose: bool = True) -> int:
    """Returns the number of modules compiled (0: no reference here, nothing done)."""
    if not os.path.isdir(os.path.join(REFERENCE, "dlrover")):
        if verbose:
            print(f"oracle/build_ref.py: no reference at {REFERENCE}; keeping what is in {OUT}")
        return 0
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    p = subprocess.run([sys.executable, "-c", PROBE + REPORT, REFERENCE], env=env, cwd="/tmp",
                       capture_output=True, text=True, timeout=600)
    files = _modules(p.stdout, "memory-save", p.returncode, p.stderr)
    files = sorted(set(files + _session(env)))
    root = os.path.realpath(REFERENCE) + os.sep
    tmp = OUT + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    manifest = {"python": sys.version.split()[0], "files": {}}
    for src in files:
        rel = src[len(root):]
        dst = os.path.join(tmp, rel + "c")          # x.py -> x.pyc, next to where x.py would be
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        py_compile.compile(src, cfile=dst, dfile=os.path.join("<reference>", rel), doraise=True,
                           invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
        with open(src, "rb") as f:
            manifest["files"][rel] = hashlib.sha256(f.read()).hexdigest()
    head = os.path.join(REFERENCE, ".git", "HEAD")
    if os.path.exists(head):
        try:
            ref = open(head).read().strip()
            if ref.startswith("ref: "):
                ref = open(os.path.join(REFERENCE, ".git", ref[5:])).read().strip()
            manifest["commit"] = ref
        except OSError:
            pass
    with open(os.path.join(tmp, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)
    shutil.rmtree(OUT, ignore_errors=True)
    os.replace(tmp, OUT)
    if verbose:
        print(f"oracle/build_ref.py: {len(files)} reference modules -> {OUT}")
    return len(files)


if __name__ == "__main__":
    build()
