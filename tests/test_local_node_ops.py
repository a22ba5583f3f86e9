"""The node-side operations run ON the node (cro_local_node_op, csrc/gpus_local.cpp): the same restated flows
as tests/test_node_side_entries.py, but with the Exec seam answered locally — native /proc scans, spawned
read-only commands, mutating commands only on request.  CPU tests use a fake /proc; the GPU tests run the real
read-only checks against the box."""
import os

import pytest

DEV = "GPU-7cc45b7b-2a6d-f0ac-1b02-6f8de09e1a6c"


def fake_proc(tmp_path, gpus, procs=()):
    root = tmp_path / "proc"
    for bus, (minor, uuid) in gpus.items():
        d = root / "driver" / "nvidia" / "gpus" / bus
        d.mkdir(parents=True)
        (d / "information").write_text("Model: \t NVIDIA B200\nGPU UUID: \t %s\nDevice Minor: \t %s\nBus Location: \t %s\n" % (uuid, minor, bus))
    for pid, cmdline in procs:
        p = root / str(pid)
        p.mkdir(parents=True)
        (p / "cmdline").write_bytes(b"\0".join(a.encode() for a in cmdline) + b"\0")
        (p / "comm").write_text(cmdline[0].rsplit("/", 1)[-1] + "\n")
        (p / "fd").mkdir()
    root.mkdir(exist_ok=True)
    return str(root)


def test_cmdline_scan(cro, tmp_path):
    target = "/sys/bus/pci/devices/0000:1f:00.0/remove"
    root = fake_proc(tmp_path, {}, [(100, ["/bin/sh", "-c", "/usr/bin/echo 1 | /usr/bin/tee %s > /dev/null" % target]), (101, ["/usr/bin/sleep", "9"])])
    assert cro.scan_cmdline_for(root, target) is True
    assert cro.scan_cmdline_for(root, "/sys/bus/pci/devices/0000:2f:00.0/remove") is False
    assert cro.scan_cmdline_for(str(tmp_path / "nowhere"), target) is False


def test_rke2_flavour_with_a_fake_proc(cro, tmp_path):
    req = {"node": "worker-0", "device_id": DEV, "device_resource_type": "DRA", "driver_container": False}
    # the GPU is not under /proc/driver/nvidia/gpus any more: nothing to check, nothing to drain (gpus.go:109-121, :227-230)
    root = fake_proc(tmp_path / "a", {"0000:2f:00.0": ("1", "GPU-other")})
    for op in ("check_no_gpu_loads", "drain"):
        out = cro.local_node_op(None, dict(req, op=op, proc_root=root))
        assert out["error"] == "" and [(x["kind"], x["how"]) for x in out["exec_log"]] == [("proc_scan", "native")], out
    # it is there: the next step needs nvidia-smi, which this container does not have — the spawn error is the exec error
    # (native_nvml off: where libnvidia-ml is loadable the query would otherwise be answered in process)
    root = fake_proc(tmp_path / "b", {"0000:1f:00.0": ("0", DEV)})
    out = cro.local_node_op(None, dict(req, op="drain", proc_root=root, native_nvml=False))
    assert [(x["kind"], x["how"]) for x in out["exec_log"]] == [("proc_scan", "native"), ("command", "spawned")]
    assert out["exec_log"][1]["argv"] == ["/bin/chroot", "/host-root", "/usr/bin/nvidia-smi", "drain", "-p", "0000:1F:00.0", "-q"]
    if not os.path.exists("/usr/bin/nvidia-smi"):
        assert out["error"].startswith("check gpu drain status command failed: 'exec: \"/usr/bin/nvidia-smi\": No such file or directory'")
    with pytest.raises(cro.ProbeError):
        cro.local_node_op(None, dict(req, op="reboot"))


@pytest.mark.gpu
def test_local_checks_on_the_box(cro):
    """Real read-only checks: this very process holds a CUDA context on GPU 0, so the load check finds a compute app
    and the open-file scan finds a holder of /dev/nvidia<minor> — both are the reference's refusals, spelled its way."""
    with cro.ProbeContext(sweep_bytes=64 << 20, devices=[0], read_sweeps=1, copy_sweeps=1) as ctx:
        info = ctx.own_devices()[0]
        uuid = info.gpu_uuid.decode()
        ctx.probe_device(0)
        base = {"node": "worker-0", "device_id": uuid, "driver_container": True}
        out = cro.local_node_op(ctx, dict(base, op="run_nvidia_smi"))
        assert out["error"] == "" and out["exec_log"][0]["how"] == "native"          # answered from the enumeration
        out = cro.local_node_op(ctx, dict(base, op="check_gpu_visible", device_resource_type="DEVICE_PLUGIN"))
        assert out["error"] == "" and out["visible"] is True
        out = cro.local_node_op(ctx, dict(base, op="check_gpu_visible", device_resource_type="DEVICE_PLUGIN", device_id="GPU-nope"))
        assert out["visible"] is False
        out = cro.local_node_op(ctx, dict(base, op="check_no_gpu_loads", device_resource_type="DEVICE_PLUGIN"))
        # the compute-apps query goes through this process's NVML session, no child process (csrc/nvml_ops.cpp)
        assert out["exec_log"][0]["how"] == "native" and out["exec_log"][0]["argv"][1] == "--query-compute-apps=gpu_uuid,process_name"
        assert out["error"] == "" or out["error"].startswith("found gpu loads on node 'worker-0': '[GPUUUID: '")
        # dry run of the drain: enumeration (with device_minor, which driver 580's nvidia-smi refuses to print) is native,
        # persistence mode is skipped, and the open-file scan stops the drain because WE hold the device node
        out = cro.local_node_op(ctx, dict(base, op="drain", device_resource_type="DEVICE_PLUGIN"))
        hows = [(x["kind"], x["how"]) for x in out["exec_log"]]
        assert hows[:3] == [("command", "native"), ("command", "skipped (dry run)"), ("fd_scan", "native")], out
        assert out["exec_log"][2]["argv"][2].startswith('TARGET_FILE="/dev/nvidia%d"' % info.device_minor)
        assert out["error"].startswith("check /dev/nvidiaX command failed: there is a process ") and "occupied the nvidiaX file" in out["error"]
        print("local drain dry run:", out["error"].strip(), hows)


def test_dry_run_gate_is_an_allow_list(cro):
    """ADVICE r1: a deny-list lets any command nobody classified run for real.  Only known READ shapes are executed."""
    skipped = [["/usr/bin/nvidia-smi", "-i", DEV, "-pm", "0"], ["/usr/bin/nvidia-smi", "drain", "-p", "0000:1F:00.0", "-m", "1"],
               ["/usr/bin/nvidia-smi", "drain", "-p", "0000:1F:00.0", "-r"], ["/usr/bin/rm", "-f", "/dev/nvidia0"],
               ["/usr/sbin/modprobe", "-r", "nvidia_uvm"], ["/bin/sh", "-c", "echo 1 > /sys/bus/pci/devices/0000:1f:00.0/remove"],
               ["/usr/bin/nvidia-smi", "--gpu-reset"],                       # never classified by anyone: must NOT run
               ["/usr/bin/touch", "/tmp/cro-should-not-exist"], ["/usr/sbin/lsmod", "--extra"],
               ["/bin/chroot", "/host-root", "/usr/bin/rm", "-f", "/dev/nvidia0"]]
    for argv in skipped:
        out = cro.local_exec(argv)
        assert out["how"] == "skipped (dry run)" and not out["failed"], (argv, out)
    assert not os.path.exists("/tmp/cro-should-not-exist")
    for argv in (["/usr/bin/nvidia-smi", "--query-gpu=gpu_uuid", "--format=csv,noheader,nounits"],
                 ["/bin/chroot", "/host-root", "/usr/bin/nvidia-smi", "--query-compute-apps=gpu_uuid,process_name", "--format=csv,noheader,nounits"],
                 ["/bin/chroot", "/host-root", "/usr/bin/nvidia-smi", "drain", "-p", "0000:1F:00.0", "-q"], ["/usr/sbin/lsmod"]):
        out = cro.local_exec(argv, native_nvml=False)
        assert out["how"] == "spawned", (argv, out)      # (fails to exec here: no such binary — but it WAS attempted)
    # with mutation allowed the same unknown command is executed
    out = cro.local_exec(["/bin/sh", "-c", "echo hello; echo oops >&2; exit 3"], allow_mutation=True)
    assert out["how"] == "spawned" and out["failed"] and out["exec_err"] == "command terminated with exit code 3"
    assert out["stdout"] == "hello\n" and out["stderr"] == "oops\n"


def test_wedged_command_is_killed_at_the_deadline(cro):
    """A nvidia-smi stuck on a GPU that is mid-drain must not hang the agent: deadline, SIGKILL, reap."""
    import time
    t0 = time.monotonic()
    out = cro.local_exec(["/bin/sh", "-c", "echo started; sleep 30"], allow_mutation=True, exec_deadline_ms=300)
    assert time.monotonic() - t0 < 5
    assert out["failed"] and out["exec_err"] == "context deadline exceeded" and out["stdout"] == "started\n"
    # a child that closes its pipes and lingers is reaped by the same deadline
    t0 = time.monotonic()
    out = cro.local_exec(["/bin/sh", "-c", "exec >/dev/null 2>&1; sleep 30"], allow_mutation=True, exec_deadline_ms=300)
    assert time.monotonic() - t0 < 5 and out["exec_err"] == "context deadline exceeded"


def test_small_error_buffer_gets_a_truncated_message_not_stale_bytes(cro):
    import ctypes
    err = ctypes.create_string_buffer(b"STALE-STALE-STALE-STALE", 24)
    rc = cro.lib.cro_fm_parse_scale_up_response(b'{"data":{"machines":[]}}', b"cr", b"gpu", b"m", ctypes.create_string_buffer(64), 64,
                                                ctypes.create_string_buffer(64), 64, err, 24)
    assert rc == cro.ERR_PARSE
    assert err.value == b"can not find the added "           # 23 bytes of the reference's sentence + NUL
