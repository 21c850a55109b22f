"""Generates tests/golden/wire_reference.json: every message the REFERENCE's own agent
(AsyncCheckpointSaver) and trainer (DdpCheckpointer) put on their local sockets during one
session — a memory save, a load, a disk save and the wait for it.  Each message is recorded
as the sender pickled it (length framing stripped), base64-encoded.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_wire_golden.py <reference checkout>

tests/test_wire_compat.py unpickles every recorded message with this package in wire-compat
mode and pickles it again: the opcodes must come out as the reference wrote them.
"""

import base64
import json
import os
import shutil
import subprocess
import sys
import tempfile
import uuid

HERE = os.path.dirname(os.path.abspath(__file__))

TAP = r"""
import base64, json, sys, threading
from unittest import mock
sys.path.insert(0, sys.argv[1])
sys.modules.setdefault("kubernetes", mock.MagicMock())
import dlrover.python.common.multi_process as mp
_lock, _orig, _log = threading.Lock(), mp._socket_send, open(sys.argv[2], "a")


def _tap(sock, message):
    with _lock:
        _log.write(json.dumps({"from": sys.argv[3], "pickle": base64.b64encode(message).decode()})
                   + "\n")
        _log.flush()
    _orig(sock, message)


mp._socket_send = _tap
"""

AGENT = TAP + r"""
import time
from dlrover.python.elastic_agent.torch.ckpt_saver import AsyncCheckpointSaver
AsyncCheckpointSaver.start_async_saving_ckpt()
print("AGENT_READY", flush=True)
time.sleep(120)
"""

TRAINER = TAP + r"""
import os
import torch
from dlrover.trainer.torch.flash_checkpoint.ddp import DdpCheckpointer, StorageType
d = sys.argv[4]
ckpt = DdpCheckpointer(d)
sd = {"w": torch.arange(1000, dtype=torch.float32), "b": torch.ones(7, dtype=torch.bfloat16),
      "step": 12}
ckpt.save_checkpoint(12, sd, storage_type=StorageType.MEMORY)
back = ckpt.load_checkpoint()
assert torch.equal(back["w"], sd["w"]) and back["step"] == 12
del back
ckpt.save_checkpoint(13, sd, storage_type=StorageType.DISK)
ckpt.wait_latest_checkpoint(timeout=60)
assert open(os.path.join(d, "dlrover_latest.txt")).read() == "13"
print("TRAINER_OK", flush=True)
"""


def main(reference: str) -> None:
    run_id = "wiregold" + uuid.uuid4().hex[:8]
    env = dict(os.environ, TORCHELASTIC_RUN_ID=run_id, ROLE_NAME="dlrover-trainer",
               DLROVER_LOG_LEVEL="WARNING", PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    with tempfile.TemporaryDirectory() as tmp:
        log = os.path.join(tmp, "wire.jsonl")
        # fixed on purpose: the checkpoint paths travel inside the messages, and a fixed
        # directory keeps the recording identical from run to run (so: one run at a time)
        ckpt_dir = "/tmp/wire_golden_ckpt"
        agent = subprocess.Popen([sys.executable, "-c", AGENT, reference, log, "agent"], env=env,
                                 stdout=subprocess.PIPE, text=True)
        try:
            assert "AGENT_READY" in agent.stdout.readline()
            out = subprocess.run([sys.executable, "-c", TRAINER, reference, log, "trainer",
                                  ckpt_dir], env=env, capture_output=True, text=True, timeout=180)
            assert "TRAINER_OK" in out.stdout, out.stderr[-3000:]
        finally:
            agent.kill()
            agent.wait()
            shutil.rmtree(ckpt_dir, ignore_errors=True)
            shutil.rmtree(os.path.join("/tmp/ckpt_sock", run_id), ignore_errors=True)
            for f in os.listdir("/dev/shm"):
                if f.startswith(run_id):
                    os.unlink(os.path.join("/dev/shm", f))
        messages = [json.loads(ln) for ln in open(log)]
    seen, unique = set(), []
    for m in messages:  # polling repeats the same request; one copy of each is enough
        if m["pickle"] not in seen:
            seen.add(m["pickle"])
            unique.append(m)
    with open(os.path.join(HERE, "wire_reference.json"), "w") as f:
        json.dump({"session": "DdpCheckpointer: save(MEMORY), load, save(DISK), wait",
                   "python": sys.version.split()[0], "messages": unique}, f, indent=1)
    print(f"{len(messages)} messages, {len(unique)} distinct")


if __name__ == "__main__":
    main(sys.argv[1])
