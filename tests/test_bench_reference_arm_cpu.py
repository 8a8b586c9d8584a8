"""``bench.py --impl reference`` (the driver's reference arm) on the "tiny" configuration: runs the UNMODIFIED reference's
``gen_image`` on the host cores, prints ONE JSON line with the contract keys, and bounds its sample (calibration step +
deadline: the host arm runs in a killable subprocess and the number is derived from whatever finished) whatever
--steps / --warmup are passed. The tests that run the arm need the reference (oracle/ref_harness.py); the others do not."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*extra):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--height", "256",
                        "--width", "256", *extra], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


@pytest.mark.reference
def test_reference_arm_line():
    line = run("--steps", "2", "--warmup", "1")
    assert "unavailable" not in line, line
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    assert line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == line["value"] and "gen_image" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["ar_steps_run"] == {"warmup": 1, "timed": 2}


@pytest.mark.reference
def test_reference_arm_deadline_is_reported_not_fatal():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", BD_REF_DEADLINE_S="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][0])
    assert p.returncode == 0 and line["impl"] == "reference" and "not built within 1 s" in line["unavailable"]


def test_reference_arm_other_ranks_do_nothing():
    """under torchrun (N > 1) rank 0 alone runs the arm; the other ranks exit 0 without work or output"""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--model", "tiny"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert p.returncode == 0 and p.stdout.strip() == ""


def _log(n_steps_done, n_evals_extra=0, done=False, S=3):
    """a worker event log: build, gen_start, 4 prefill passes, then per AR step S+1 evaluations + 2 block passes"""
    ev, t = [dict(ev="start", t=0.0, threads=4), dict(ev="built", t=5.0, s=5.0, pn=16), dict(ev="gen_start", t=5.0)], 5.0
    for rows in (66, 16, 5, 16):
        t += 2.0
        ev.append(dict(ev="llm", t=t, s=2.0, rows=rows))
    for k in range(n_steps_done + 1):
        ev.append(dict(ev="step", t=t))
        n_ev = (S + 1) if k < n_steps_done else n_evals_extra
        for _ in range(n_ev):
            t += 1.0
            ev.append(dict(ev="eval", t=t, s=1.0, rows=32))
        if k < n_steps_done:
            for _ in range(2):
                t += 3.0
                ev.append(dict(ev="llm", t=t, s=3.0, rows=16))
    if done:
        ev = [e for e in ev[:-1]] if ev[-1]["ev"] == "step" else ev
        ev.append(dict(ev="gen_done", t=t, prefill_s=8.0, ar_s=[10.0] * n_steps_done, total_s=t - 5.0))
    return ev


def test_derive_reference_sample_from_partial_logs():
    sys.path.insert(0, ROOT)
    import bench
    kw = dict(wall=60.0, threads=4, model="tiny", n_warm=1, S=3, bs=1, deadline_s=60.0)
    # (a) finished: 1 warm-up + 2 timed steps of 10 s; prefill 8 s -> image = 8 + 64 * 10
    r = bench.derive_reference_sample(_log(3, done=True), killed=False, **kw)
    assert r["ar_step_s"] == 10.0 and abs(r["prefill_s"] - 8.0) < 1e-9 and abs(1 / r["images_per_s"] - 648.0) < 1e-6
    assert (r["n_warm"], r["n_timed"]) == (1, 2) and "1 warm-up + 2 timed" in r["sample"]
    # (b) killed during the 2nd step: one complete step (4 evaluations + 2 block passes = 10 s)
    r = bench.derive_reference_sample(_log(1, n_evals_extra=2), killed=True, **kw)
    assert abs(r["ar_step_s"] - 10.0) < 1e-9 and "1 complete AR step" in r["sample"] and "killed" in r["sample"]
    # (c) killed inside the first step after 3 evaluations: (S + 1) * 1 s + 2 * 2 s (the prefill's first-block passes)
    r = bench.derive_reference_sample(_log(0, n_evals_extra=3), killed=True, **kw)
    assert abs(r["ar_step_s"] - (4 * 1.0 + 2 * 2.0)) < 1e-9 and "NO complete AR step" in r["sample"]
    assert abs(r["prefill_s"] - 8.0) < 1e-9
    # nothing usable: killed during the prefill
    with pytest.raises(RuntimeError):
        bench.derive_reference_sample(_log(0)[:5], killed=True, **kw)
    with pytest.raises(RuntimeError):
        bench.derive_reference_sample(_log(0)[:1], killed=True, **kw)


def test_usable_cpus_honours_the_cgroup_quota(tmp_path):
    """profiles/r02_host_probe.txt: a GPU box shows 128 CPUs and grants ``cpu.max = 1600000 100000`` (16 CPUs)"""
    sys.path.insert(0, ROOT)
    from bitdance_b200.hostinfo import usable_cpus
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    (tmp_path / "cpu.max").write_text("200000 100000\n")
    assert usable_cpus(str(tmp_path)) == min(n, 2)
    (tmp_path / "cpu.max").write_text("max 100000\n")
    assert usable_cpus(str(tmp_path)) == n
    (tmp_path / "cpu.max").write_text("50000 100000\n")          # half a CPU still means one thread
    assert usable_cpus(str(tmp_path)) == 1
    (tmp_path / "cpu.max").unlink()
    (tmp_path / "cpu").mkdir()
    (tmp_path / "cpu" / "cpu.cfs_quota_us").write_text("300000\n")     # cgroup v1
    (tmp_path / "cpu" / "cpu.cfs_period_us").write_text("100000\n")
    assert usable_cpus(str(tmp_path)) == min(n, 3)
    (tmp_path / "cpu" / "cpu.cfs_quota_us").write_text("-1\n")
    assert usable_cpus(str(tmp_path)) == n
    assert usable_cpus(str(tmp_path / "missing")) == n
