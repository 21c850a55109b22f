"""Interoperability with the REFERENCE's agent and trainer halves: lock / queue / dict RPCs,
the meta tree, the saver ClassMeta and the SAVE event cross the process boundary as pickles.

  * live: the reference's own AsyncCheckpointSaver serves OUR DdpCheckpointer in wire-compat
    mode and persists our shared-memory bytes with its own code, and the reference's own
    DdpCheckpointer is served by OUR agent.  The reference runs from its byte code in
    oracle/_ref/pyref (oracle/build_ref.py), each half in a process of its own, as
    `dlrover-run` would host it.
  * recorded: tests/golden/wire_reference.json holds every distinct message the reference's
    agent and trainer sent each other in one session (tests/golden/make_wire_golden.py).  With
    this package in wire-compat mode, each must unpickle into this package's classes, and
    those must pickle the same content opcode for opcode as the reference's classes did."""

import json
import os
import subprocess
import sys
import uuid

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "wire_reference.json")
PYREF = os.path.join(ROOT, "oracle", "_ref", "pyref")

CHECK = r"""
import base64, importlib, io, json, pickle, pickletools, sys
sys.path.insert(0, sys.argv[1])
import dlrover_b200                       # DLROVER_B200_WIRE_COMPAT=1 -> enable_wire_compat()


def canonical(data):
    # the opcode stream with memo references resolved: whether two equal strings were one
    # object when pickled (an interned attribute name and a user dict key) is not content
    toks, memo, last, refs = [], [], None, 0
    for op, arg, _ in pickletools.genops(data):
        if op.name == "FRAME":
            continue
        if op.name == "MEMOIZE":
            if last[0] != "str":
                last, refs = ("ref", refs), refs + 1
            memo.append(last)
            continue
        if op.name in ("BINGET", "LONG_BINGET"):
            last = memo[arg]
        elif isinstance(arg, str) and "UNICODE" in op.name:
            last = ("str", arg)
        else:
            last = (op.name, repr(arg))
        toks.append(last)
    return toks


class Loader(pickle.Unpickler):
    # notes every reference class the message names that does not resolve to this package
    def find_class(self, mod, name):
        owner = importlib.import_module(mod)
        if mod.startswith("dlrover") and not owner.__name__.startswith("dlrover_b200"):
            self.foreign.append(f"{mod}.{name} -> {owner.__name__}")
        return super().find_class(mod, name)


out = []
for m in json.load(open(sys.argv[2]))["messages"]:
    if m["from"] != sys.argv[3]:
        continue
    want = base64.b64decode(m["pickle"])
    loader = Loader(io.BytesIO(want))
    loader.foreign = []
    obj = loader.load()
    foreign = loader.foreign
    out.append({"type": type(obj).__name__, "method": getattr(obj, "method", None),
                "foreign": foreign, "same_pickle": canonical(pickle.dumps(obj)) == canonical(want)})
print("FCWIRE " + json.dumps(out))
"""


def _replay(sender):
    env = dict(os.environ, DLROVER_B200_WIRE_COMPAT="1", PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    p = subprocess.run([sys.executable, "-c", CHECK, ROOT, GOLDEN, sender], env=env,
                       capture_output=True, text=True, timeout=180)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("FCWIRE ")]
    assert p.returncode == 0 and lines, p.stderr[-3000:]
    return json.loads(lines[-1][len("FCWIRE "):])


@pytest.mark.timeout(240)
def test_recorded_reference_agent_replies_load_into_our_classes():
    """The reference agent's replies (lock grants, dict snapshots with the meta tree) load
    into our classes, and pickle back unchanged."""
    got = _replay("agent")
    assert {r["type"] for r in got} >= {"SocketResponse", "LockAcquireResponse", "DictMessage"}
    for r in got:
        assert not r["foreign"] and r["same_pickle"], r


@pytest.mark.timeout(240)
def test_recorded_reference_trainer_requests_load_into_our_classes():
    """The reference trainer's requests (saver ClassMeta, SAVE events, lock acquire/release,
    meta-dict sets) load into our classes, and pickle back unchanged."""
    got = _replay("trainer")
    assert {r["method"] for r in got} >= {"put", "acquire", "release", "set", "get"}, got
    for r in got:
        assert r["type"] == "SocketRequest" and not r["foreign"] and r["same_pickle"], r


def _pyref():
    """The reference's byte code, built if its source tree is at hand."""
    from oracle import build_ref

    trainer = os.path.join(PYREF, "dlrover", "trainer", "torch", "flash_checkpoint", "ddp.pyc")
    if not os.path.exists(trainer):
        build_ref.build(verbose=False)
    if not os.path.exists(trainer):
        pytest.skip("oracle/_ref/pyref not built (oracle/build_ref.py needs the reference's source)")
    return PYREF


AGENT = r"""
import sys, time
from unittest import mock
sys.path.insert(0, %r)
sys.modules.setdefault("kubernetes", mock.MagicMock())
import dlrover.python.elastic_agent.torch.ckpt_saver as ref
assert ref.__file__.startswith(sys.path[0]), ref.__file__   # the reference's byte code
ref.AsyncCheckpointSaver.start_async_saving_ckpt()
print("AGENT_READY", flush=True)
time.sleep(120)
"""

TRAINER = r"""
import os, sys, time
sys.path.insert(0, %r)
import torch
import dlrover_b200                       # DLROVER_B200_WIRE_COMPAT=1 -> enable_wire_compat()
from dlrover_b200.flash_checkpoint.api import DdpCheckpointer, StorageType
from dlrover_b200.common.multi_process import SocketRequest
assert SocketRequest.__module__ == "dlrover.python.common.multi_process"
d = sys.argv[1]
ckpt = DdpCheckpointer(d)
sd = {"w": torch.arange(1000, dtype=torch.float32), "b": torch.ones(7, dtype=torch.bfloat16),
      "step": 12}
ckpt.save_checkpoint(12, sd, storage_type=StorageType.MEMORY)
back = ckpt.load_checkpoint()
assert torch.equal(back["w"], sd["w"]) and back["step"] == 12
del back
ckpt.save_checkpoint(13, sd, storage_type=StorageType.DISK)
ckpt.wait_latest_checkpoint(timeout=60)
print("TRACKER", open(os.path.join(d, "dlrover_latest.txt")).read())
print("FILES", sorted(os.listdir(os.path.join(d, "13"))))
on_disk = torch.load(os.path.join(d, "13", "rank_0.pt"))
assert torch.equal(on_disk["w"], sd["w"]) and torch.equal(on_disk["b"], sd["b"])
print("TRAINER_OK")
ckpt.engine.close()
"""


def test_our_trainer_against_the_reference_agent(tmp_path):
    ref = _pyref()
    run_id = "wire" + uuid.uuid4().hex[:8]
    env = dict(os.environ, TORCHELASTIC_RUN_ID=run_id, ROLE_NAME="dlrover-trainer",
               DLROVER_LOG_LEVEL="WARNING", PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    agent = subprocess.Popen([sys.executable, "-c", AGENT % ref], env=env,
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    try:
        line = agent.stdout.readline()
        assert "AGENT_READY" in line
        tenv = dict(env, DLROVER_B200_WIRE_COMPAT="1")
        out = subprocess.run([sys.executable, "-c", TRAINER % ROOT, str(tmp_path)], env=tenv,
                             capture_output=True, text=True, timeout=180)
        assert "TRAINER_OK" in out.stdout, out.stdout[-1500:] + out.stderr[-3000:]
        assert "TRACKER 13" in out.stdout and "FILES ['rank_0.pt']" in out.stdout
    finally:
        agent.kill()
        agent.wait()
        import glob
        import shutil

        shutil.rmtree(os.path.join("/tmp/ckpt_sock", run_id), ignore_errors=True)
        for f in glob.glob(f"/dev/shm/{run_id}_*"):
            os.unlink(f)


OUR_AGENT = r"""
import sys, time
sys.path.insert(0, %r)
import dlrover_b200                       # wire-compat: reference pickles resolve to our classes
from dlrover_b200.ckpt_saver import AsyncCheckpointSaver
AsyncCheckpointSaver.start_async_saving_ckpt()
print("AGENT_READY", flush=True)
time.sleep(120)
"""

REF_TRAINER = r"""
import os, sys, time
from unittest import mock
sys.path.insert(0, %r)
sys.modules.setdefault("kubernetes", mock.MagicMock())
import torch
import dlrover.trainer.torch.flash_checkpoint.ddp as ref
assert ref.__file__.startswith(sys.path[0]), ref.__file__   # the reference's byte code
DdpCheckpointer, StorageType = ref.DdpCheckpointer, ref.StorageType
d = sys.argv[1]
ckpt = DdpCheckpointer(d)
sd = {"w": torch.arange(1000, dtype=torch.float32), "step": 21}
ckpt.save_checkpoint(21, sd, storage_type=StorageType.DISK)
ckpt.wait_latest_checkpoint(timeout=60)
print("TRACKER", open(os.path.join(d, "dlrover_latest.txt")).read())
on_disk = torch.load(os.path.join(d, "21", "rank_0.pt"))
assert torch.equal(on_disk["w"], sd["w"]) and on_disk["step"] == 21
print("TRAINER_OK")
"""


def test_the_reference_trainer_against_our_agent(tmp_path):
    ref = _pyref()
    run_id = "wire" + uuid.uuid4().hex[:8]
    env = dict(os.environ, TORCHELASTIC_RUN_ID=run_id, ROLE_NAME="dlrover-trainer",
               DLROVER_LOG_LEVEL="WARNING", PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    agent = subprocess.Popen([sys.executable, "-c", OUR_AGENT % ROOT],
                             env=dict(env, DLROVER_B200_WIRE_COMPAT="1"),
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    try:
        assert "AGENT_READY" in agent.stdout.readline()
        out = subprocess.run([sys.executable, "-c", REF_TRAINER % ref, str(tmp_path)], env=env,
                             capture_output=True, text=True, timeout=180)
        assert "TRAINER_OK" in out.stdout, out.stdout[-1500:] + out.stderr[-3000:]
        assert "TRACKER 21" in out.stdout
    finally:
        agent.kill()
        agent.wait()
        import glob
        import shutil

        shutil.rmtree(os.path.join("/tmp/ckpt_sock", run_id), ignore_errors=True)
        for f in glob.glob(f"/dev/shm/{run_id}_*"):
            os.unlink(f)
