"""`python -m torch.distributed.run` for tests that must not leave a rank behind.

torchrun starts every worker in a session of its own, so killing torchrun (what subprocess.run does
on a timeout) orphans ranks that wait in a collective, holding their GPU.  Here a timeout sends
SIGTERM to torchrun instead: its agent then stops its workers (SIGTERM, SIGKILL after its grace
period) before it exits.  Only if torchrun itself does not exit is its own process group killed."""
import os
import signal
import subprocess
import sys


def torchrun(args, world, port, cwd, timeout, env=None):
    """torchrun --nproc-per-node world <args> -> CompletedProcess (text); raises TimeoutExpired after
    `timeout` seconds, once the launch and its ranks are gone."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port)] + list(args)
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=cwd, env=env,
                         start_new_session=True)
    try:
        out, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        p.terminate()
        try:
            p.communicate(timeout=120)
        except subprocess.TimeoutExpired:
            os.killpg(p.pid, signal.SIGKILL)
            p.communicate()
        raise
    return subprocess.CompletedProcess(cmd, p.returncode, out, err)
