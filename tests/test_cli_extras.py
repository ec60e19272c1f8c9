"""arap_deform's 8-token lines (backward flow + occlusion outputs) without a GPU: the thin client (ARAP_SERVER) hands
6- and 8-token lines to the worker unchanged, drops nothing and keeps 6-token lines as they were; tokens after the
eighth are still ignored.  The worker side is played by the test."""
import os
import subprocess
import time

from arap_flow_b200 import driver

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "arap_flow_b200", "bin")


def _handoff(tmp_path, argv):
    """Run the client against a fake worker; returns (client result, the job file's lines)."""
    spool = tmp_path / "spool"
    spool.mkdir()
    (spool / "ready").write_text("0\n")
    env = dict(os.environ, ARAP_PLAN=driver.PLAN, ARAP_SERVER=str(spool))
    p = subprocess.Popen([os.path.join(BIN, "arap_deform")] + argv, env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True)
    t0 = time.time()
    jobs = []
    while not jobs and time.time() - t0 < 60:
        jobs = [f for f in os.listdir(spool) if f.endswith(".job")]
        time.sleep(0.01)
    assert jobs, "the client wrote no job"
    job = spool / jobs[0]
    lines = [ln.split() for ln in job.read_text().splitlines()]
    job.unlink()
    (spool / (jobs[0][:-4] + ".done")).write_text("0\n%d\n" % len(lines))
    out, err = p.communicate(timeout=60)
    return p.returncode, out, lines


def test_client_carries_mixed_lines(tmp_path):
    six = ["r.png", "m.png", "c.txt", "f.flo", "w.png", "wm.png"]
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join([" ".join(six + ["b.flo", "o.png"]), " ".join(six), " ".join(six + ["x"]),
                              " ".join(six + ["b2.flo", "o2.png", "ignored"]), "too short"]) + "\n")
    rc, out, lines = _handoff(tmp_path, [str(lst)])
    assert rc == 0 and out.count("Saved") == 4
    assert lines == [six + ["b.flo", "o.png"], six, six, six + ["b2.flo", "o2.png"]]


def test_client_carries_eight_argv(tmp_path):
    argv = ["r.png", "m.png", "c.txt", "f.flo", "w.png", "wm.png", "b.flo", "o.png"]
    rc, out, lines = _handoff(tmp_path, argv)
    assert rc == 0 and out.count("Saved") == 1 and lines == [argv]


def test_seven_or_nine_argv_are_rejected():
    for n in (7, 9):
        r = subprocess.run([os.path.join(BIN, "arap_deform")] + ["a"] * n, capture_output=True, text=True)
        assert r.returncode == 1 and "Invalid Input!" in r.stdout
