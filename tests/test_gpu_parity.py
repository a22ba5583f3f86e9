"""Parity tests proper: the CUDA path (through the C ABI) against the oracle.

Bit-exact bar: the kernels compute 64-bit integer checksums; identity strings
are compared byte for byte with what `nvidia-smi` prints on the same box."""
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu

MASK = (1 << 64) - 1
VARIANTS = [1, 2, 3]          # READ_LDG, READ_TMA, READ_LDG256
COPY_VARIANTS = [1, 2, 3]     # COPY_LDG, COPY_TMA, COPY_TMA_FUSED


@pytest.fixture(scope="module")
def ctx_small(cro):
    with cro.ProbeContext(sweep_bytes=64 << 20, devices=[0], flags=cro.F_VERIFY_COPY, read_sweeps=3, copy_sweeps=2) as c:
        yield c


def test_pattern_words_match_oracle(cro, coracle, ctx_small):
    ctx_small.hbm_fill(0)
    seed = ctx_small.seed(0)
    n_words = (64 << 20) // 8
    for first, n in ((0, 4096), (n_words - 1024, 1024), (123457, 999)):
        got = ctx_small.read_words(0, first, n)
        assert got == [coracle.pattern_word(seed, first + i) for i in range(n)]


@pytest.mark.parametrize("variant", VARIANTS)
def test_read_checksum_matches_oracle(cro, coracle, ctx_small, variant):
    s = ctx_small.hbm_read_checksum(0, variant)
    assert s.checksum == coracle.checksum(ctx_small.seed(0), 0, (64 << 20) // 8)
    assert s.variant == variant and s.bytes == 64 << 20 and s.ns > 0 and s.timer_ns > 0


def test_expected_kernel_matches_oracle(coracle, ctx_small):
    s = ctx_small.hbm_expected_checksum(0)
    assert s.checksum == coracle.checksum(ctx_small.seed(0), 0, (64 << 20) // 8)


@pytest.mark.parametrize("cv", COPY_VARIANTS)
def test_copy_round_trip(cro, coracle, ctx_small, cv):
    want = coracle.checksum(ctx_small.seed(0), 0, (64 << 20) // 8)
    ctx_small.hbm_fill(0)
    c = ctx_small.hbm_copy(0, cv)
    assert c.bytes == 2 * (64 << 20) and c.variant == cv
    if cv == 3:
        assert c.checksum == want          # the checksumming copy folds its source as it moves it
    for rv in VARIANTS:
        d = ctx_small.hbm_read_checksum(0, rv, dst=True)
        assert d.checksum == want, (cv, rv)
    # destination words themselves, not only their checksum
    n_words = (64 << 20) // 8
    assert ctx_small.read_words(0, n_words + 77, 64) == ctx_small.read_words(0, 77, 64)


# ragged and tiny sizes: not a multiple of any tile; the smallest legal sweep is 16 bytes
@pytest.mark.parametrize("nbytes", [16, 32, 4096 + 16, 65536 - 16, 1 << 20, (1 << 20) + 48, 3 * (1 << 20) + 16 * 7,
                                    (32 << 20) + 32784])
def test_ragged_sizes(cro, coracle, nbytes):
    with cro.ProbeContext(sweep_bytes=nbytes, devices=[0], flags=cro.F_VERIFY_COPY, read_sweeps=1, copy_sweeps=1,
                          seed_base=0x1234500000000000) as c:
        want = coracle.checksum(c.seed(0), 0, nbytes // 8)
        for rv in VARIANTS:
            s = c.hbm_read_checksum(0, rv)
            assert s.checksum == want, (nbytes, rv)
        for cv in COPY_VARIANTS:
            c.inject_fault(0, nbytes // 8, 0xFFFF)     # dirty the destination first: the copy must overwrite it
            k = c.hbm_copy(0, cv)
            if cv == 3:
                assert k.checksum == want, (nbytes, cv)
            d = c.hbm_read_checksum(0, 1, dst=True)
            assert d.checksum == want, (nbytes, cv)
        e = c.hbm_expected_checksum(0)
        assert e.checksum == want
        # the whole probe at this size (graph, ping-pong copies, device-written verdict)
        r = c.probe_device(0)
        assert r.status == 0 and r.checksum == r.expect == coracle.checksum(r.seed, 0, nbytes // 8) and r.copy_verified == 1


def test_fault_is_detected_and_located(cro, coracle, ctx_small):
    """A single flipped bit anywhere must change the checksum by exactly that bit; the probe reports it."""
    ctx_small.hbm_fill(0)
    seed, n_words = ctx_small.seed(0), (64 << 20) // 8
    clean = coracle.checksum(seed, 0, n_words)
    for word, bit in ((0, 0), (n_words - 1, 63), (n_words // 3, 17)):
        ctx_small.inject_fault(0, word, 1 << bit)
        for rv in VARIANTS:
            s = ctx_small.hbm_read_checksum(0, rv)
            assert s.checksum_xor == clean[0] ^ (1 << bit), (word, bit, rv)
            assert s.checksum_sum != clean[1]
            # the weighted component moves by exactly (flipped value - clean value) * (2*word + 1)
            w = coracle.pattern_word(seed, word)
            assert s.checksum_wsum == (clean[2] + ((w ^ (1 << bit)) - w) * (2 * word + 1)) & MASK
        k = ctx_small.hbm_copy(0, 3)                        # the checksumming copy sees it in its source stream too
        assert k.checksum_xor == clean[0] ^ (1 << bit)
        ctx_small.inject_fault(0, word, 1 << bit)          # undo
    s = ctx_small.hbm_read_checksum(0, 1)
    assert s.checksum == clean
    # two words swapping places: XOR and sum cannot see it, the position-weighted sum does
    a, b = 12345, n_words - 777
    wa, wb = coracle.pattern_word(seed, a), coracle.pattern_word(seed, b)
    ctx_small.inject_fault(0, a, wa ^ wb)
    ctx_small.inject_fault(0, b, wa ^ wb)
    for rv in VARIANTS:
        s = ctx_small.hbm_read_checksum(0, rv)
        assert (s.checksum_xor, s.checksum_sum) == clean[:2] and s.checksum_wsum != clean[2], rv
    assert ctx_small.hbm_copy(0, 3).checksum_wsum != clean[2]
    ctx_small.inject_fault(0, a, wa ^ wb)
    ctx_small.inject_fault(0, b, wa ^ wb)
    # the full probe refills (with the NEXT nonce's pattern), so it passes
    r = ctx_small.probe_device(0)
    assert r.status == 0 and r.checksum == r.expect == r.copy_checksum == coracle.checksum(r.seed, 0, n_words)


def test_every_probe_writes_a_fresh_pattern(cro, coracle, ctx_small):
    """A fill or copy that silently did nothing must not pass on the previous probe's bytes: each probe takes the next
    nonce, so its pattern (and closed form) differs from whatever is still in HBM."""
    d = ctx_small.own_devices()[0]
    r1 = ctx_small.probe_device(0)
    r2 = ctx_small.probe_device(0)
    assert r2.nonce == r1.nonce + 1 and r1.seed != r2.seed and r1.checksum != r2.checksum
    for r in (r1, r2):
        assert r.seed == coracle.probe_seed(0x00C0FFEE00000000, max(d.device_minor, 0), r.nonce)
        assert r.status == 0 and r.checksum == r.expect == coracle.checksum(r.seed, 0, (64 << 20) // 8)
    assert ctx_small.seed(0) == r2.seed                    # what the region holds now
    assert ctx_small.read_words(0, 5, 3) == [coracle.pattern_word(r2.seed, 5 + i) for i in range(3)]


def test_probe_catches_corruption_in_either_half(cro, coracle):
    """Fault injection THROUGH a probe: an asynchronous probe is begun, and while it cannot be touched a fresh context is
    used instead — corrupt half B (a copy destination) between two single sweeps and the ping-pong must report it."""
    S = 32 << 20
    n = S // 8
    with cro.ProbeContext(sweep_bytes=S, devices=[0], read_sweeps=2, copy_sweeps=2) as c:
        r = c.probe_device(0)
        assert r.status == 0 and r.copy_verified == 2 and r.fail_code == cro.FAIL_NONE
        want = coracle.checksum(c.seed(0), 0, n)
        # source half: the checksumming copy reads A, sees the flipped word, still copies it faithfully
        c.inject_fault(0, 99, 1 << 5)
        k = c.hbm_copy(0, 3)
        assert k.checksum_xor == want[0] ^ (1 << 5)
        assert c.hbm_read_checksum(0, 1, dst=True).checksum_xor == want[0] ^ (1 << 5)
        c.inject_fault(0, 99, 1 << 5)
        # destination half: corrupt B after a clean copy; the re-read (what the next ping-pong sweep does) catches it
        c.hbm_copy(0, 3)
        c.inject_fault(0, n + 4242, 1 << 40)
        d = c.hbm_read_checksum(0, 2, dst=True)
        assert d.checksum_xor == want[0] ^ (1 << 40) and d.checksum_wsum != want[2]


def test_probe_result_fields(cro, coracle, ctx_small):
    r = ctx_small.probe_device(0)
    d = ctx_small.own_devices()[0]
    assert r.abi_version == 2 and r.status == 0 and r.world == 1 and r.rank == 0
    assert r.gpu_uuid == d.gpu_uuid and r.pci_bus_id == d.pci_bus_id and r.device_minor == d.device_minor
    assert r.sweep_bytes == 64 << 20 and r.read_sweeps == 3 and r.copy_sweeps == 2
    assert r.seed == coracle.probe_seed(0x00C0FFEE00000000, max(d.device_minor, 0), r.nonce)
    assert 0 < r.read_best_ns <= r.read_median_ns and 0 < r.copy_best_ns <= r.copy_median_ns and r.fill_ns > 0
    assert r.sm_count == 148 and r.copy_verified == 2 and r.fail_code == 0 and r.copy_variant == cro.COPY_TMA_FUSED
    assert r.total_ns >= r.fill_ns + 3 * r.read_best_ns + 2 * r.copy_best_ns


def test_device_written_struct_equals_host_assembly(cro, coracle, ctx_small):
    """The 512-byte struct is written by the finalize kernel.  Rebuild it on the host from the same raw material —
    identity from the enumeration, checksums from the oracle, times from the per-sweep %globaltimer windows — and
    compare field by field; the CUDA-event times of the same sweeps must agree with the device's own timers."""
    r = ctx_small.probe_device(0)
    d = ctx_small.own_devices()[0]
    times = ctx_small.sweep_times(0)
    assert [t.kind for t in times] == [0] + [1] * r.copy_sweeps + [2] * r.read_sweeps
    want = coracle.checksum(r.seed, 0, r.sweep_bytes // 8)
    reads = sorted(t.timer_ns for t in times if t.kind == 2)
    copies = sorted(t.timer_ns for t in times if t.kind == 1)
    host = {
        "abi_version": 2, "status": 0, "cuda_ordinal": d.cuda_ordinal, "device_minor": d.device_minor,
        "gpu_uuid": d.gpu_uuid, "pci_bus_id": d.pci_bus_id, "hbm_bytes_total": d.hbm_bytes_total,
        "sweep_bytes": 64 << 20, "checksum_xor": want[0], "checksum_sum": want[1], "checksum_wsum": want[2],
        "expect_xor": want[0], "expect_sum": want[1], "expect_wsum": want[2],
        "copy_checksum_xor": want[0], "copy_checksum_sum": want[1], "copy_checksum_wsum": want[2],
        "fill_ns": times[0].timer_ns, "read_best_ns": reads[0], "read_median_ns": reads[len(reads) // 2],
        "copy_best_ns": copies[0], "copy_median_ns": copies[len(copies) // 2],
        "sm_count": d.sm_count, "read_sweeps": 3, "copy_sweeps": 2, "copy_verified": 2, "fail_code": 0, "fail_index": 0,
        "rank": 0, "world": 1, "read_variant": cro.READ_LDG256, "copy_variant": cro.COPY_TMA_FUSED, "p2p_ok": 0,
    }
    for k, v in host.items():
        assert getattr(r, k) == v, (k, getattr(r, k), v)
    assert list(r.p2p_read_ns) == [0] * 8 and list(r.p2p_write_ns) == [0] * 8
    for t in times:       # the two clocks watch the same kernels: events add launch latency, never lose time
        assert t.timer_ns <= t.event_ns * 1.02 + 2000 and t.event_ns <= t.timer_ns * 1.25 + 20000, (t.kind, t.index, t.timer_ns, t.event_ns)


def test_full_size_probe_matches_oracle(cro, coracle):
    """BASELINE config 2: S = 4 GiB.  The C oracle recomputes the closed form with all host threads."""
    S = 4 << 30
    with cro.ProbeContext(sweep_bytes=S, devices=[0], flags=cro.F_VERIFY_COPY) as c:
        r = c.probe_device(0)
        want = coracle.checksum(r.seed, 0, S // 8, threads=os.cpu_count() or 1)
        assert r.status == 0 and r.copy_verified == 5 and r.read_sweeps == 5 and r.copy_sweeps == 5
        assert r.checksum == want
        assert r.copy_checksum == want
        assert r.expect == want
        # size-independent property: checksum of the whole == combination of the halves' closed forms
        a = coracle.checksum(r.seed, 0, S // 16, threads=os.cpu_count() or 1)
        x2, s2, w2 = want[0] ^ a[0], (want[1] - a[1]) & MASK, (want[2] - a[2]) & MASK
        assert (x2, s2, w2) == coracle.checksum(r.seed, S // 16, S // 16)
        for rv in VARIANTS:
            s = c.hbm_read_checksum(0, rv)
            assert s.checksum == want
            s = c.hbm_read_checksum(0, rv, dst=True)       # after 5 ping-pong copies both halves hold the pattern
            assert s.checksum == want
        assert c.hbm_copy(0, cro.COPY_TMA_FUSED).checksum == want
        # a second probe: next nonce, fresh pattern, again bit-exact
        r2 = c.probe_device(0)
        assert r2.nonce == r.nonce + 1 and r2.status == 0
        assert r2.checksum == r2.expect == coracle.checksum(r2.seed, 0, S // 8, threads=os.cpu_count() or 1)


@pytest.mark.parametrize("mib", [256, 1024, 16384])
def test_the_other_sweep_sizes_of_config_2(cro, coracle, mib):
    """SURVEY.md §8d config 2 also names S = 256 MiB, 1 GiB and 16 GiB (word indices beyond 2^31 at the last one):
    whole probe, every sweep and every copy destination, bit-exact against the C oracle's closed form."""
    S = mib << 20
    with cro.ProbeContext(sweep_bytes=S, devices=[0]) as c:
        r = c.probe_device(0)
        want = coracle.checksum(r.seed, 0, S // 8, threads=os.cpu_count() or 1)
        assert r.status == 0 and r.sweep_bytes == S and r.copy_verified == 5
        assert r.checksum == r.copy_checksum == r.expect == want
        for rv in VARIANTS:
            assert c.hbm_read_checksum(0, rv).checksum == want
            assert c.hbm_read_checksum(0, rv, dst=True).checksum == want


def test_deadline_is_honoured_and_the_context_survives(cro, coracle):
    """cro_opts.deadline_ms stands in for the Go context that cannot cross cgo (SURVEY.md §8b, threading): a probe that
    outlasts it returns CRO_ERR_DEADLINE at once — the kernels cannot be recalled and finish on the device — and the
    context stays usable: the next sweep queues behind them and finds the pattern the timed-out probe wrote."""
    import time
    S = 4 << 30                                   # 9.7 ms of sweeps against a 2 ms deadline
    with cro.ProbeContext(sweep_bytes=S, devices=[0], deadline_ms=2) as c:
        c.hbm_fill(0)                             # module load, first launches: not what the deadline is about
        time.sleep(0.05)
        t0 = time.monotonic()
        with pytest.raises(cro.ProbeError) as e:
            c.probe_device(0)
        waited = time.monotonic() - t0
        assert e.value.code == cro.ERR_DEADLINE and "deadline of 2 ms exceeded" in str(e.value)
        assert waited < 1.0                       # (the first probe also captures its graph)
        time.sleep(0.1)                           # the device finishes what was enqueued
        want = coracle.checksum(c.seed(0), 0, S // 8, threads=os.cpu_count() or 1)
        assert c.hbm_read_checksum(0, cro.READ_TMA).checksum == want
        assert c.hbm_read_checksum(0, cro.READ_TMA, dst=True).checksum == want
    with cro.ProbeContext(sweep_bytes=S, devices=[0], deadline_ms=2000) as c:
        assert c.probe_device(0).status == 0


def test_identity_strings_match_nvidia_smi(cro):
    """cro_emit_csv must print what the reference's exec of nvidia-smi prints (gpus.go:886)."""
    smi = shutil.which("nvidia-smi")
    if not smi:
        pytest.skip("nvidia-smi not on this box")
    with cro.ProbeContext(sweep_bytes=1 << 20, flags=cro.F_LAZY_ALLOC) as c:
        devs = c.enumerate()
        def smi_csv(q):
            return subprocess.run([smi, "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True)
        for q in ("gpu_uuid", "gpu_uuid,pci.bus_id", "index,gpu_uuid,pci.bus_id,name"):
            want = smi_csv(q)
            assert want.returncode == 0, want.stdout + want.stderr
            assert cro.emit_csv(devs, q) == want.stdout, q
        # The reference's 3-field query (gpus.go:216-218).  Some nvidia-smi builds (driver 580 here) reject
        # `device_minor` ("not a valid field to query") — then the minor is pinned through NVML's
        # minor_number spelling if the build has it, and through /proc below.
        want = smi_csv("device_minor,gpu_uuid,pci.bus_id")
        if want.returncode == 0:
            assert cro.emit_csv(devs, "device_minor,gpu_uuid,pci.bus_id") == want.stdout
        else:
            assert "not a valid field" in want.stdout + want.stderr
            alt = smi_csv("minor_number,gpu_uuid,pci.bus_id")
            if alt.returncode == 0:
                assert cro.emit_csv(devs, "minor_number,gpu_uuid,pci.bus_id") == alt.stdout
        # /proc flavour (gpus.go:1017-1037), when the driver exposes it in this container (a container may mount the
        # registry empty; the enumeration above then came from NVML)
        base = "/proc/driver/nvidia/gpus"
        if os.path.isdir(base) and os.listdir(base):
            lines = ""
            for name in sorted(os.listdir(base)):
                p = os.path.join(base, name, "information")
                if os.path.isfile(p):
                    lines += cro.proc_information_to_line(open(p).read())
            rc, js = cro.getGPUInfoFromProcOutput(lines, "", None, "device_minor,gpu_uuid,pci.bus_id")
            assert rc == 0
            import json
            by_uuid = {m["gpu_uuid"]: m for m in json.loads(js)}
            for d in devs:
                m = by_uuid[d.gpu_uuid.decode()]
                assert m["device_minor"] == str(d.device_minor)
                assert cro.normalize(0, m["pci.bus_id"]).endswith(cro.normalize(2, d.pci_bus_id.decode()))


def test_reconcile_attach_live(cro, oracle):
    import __graft_entry__ as g
    with cro.ProbeContext(sweep_bytes=32 << 20, devices=[0], read_sweeps=1, copy_sweeps=1) as c:
        uuid = c.own_devices()[0].gpu_uuid.decode()
        base = {"name": "cr-0", "spec": {"type": "gpu", "model": "NVIDIA-B200", "target_node": "worker-0"},
                "status": {"state": "Attaching"}, "device_resource_type": "DEVICE_PLUGIN", "probe": True}
        out = cro.reconcile_attach(c, dict(base, provider={"device_id": uuid, "cdi_device_id": "res-0-0"}))
        assert g.json_status(out) == oracle.emit_status("Online", "", uuid, "res-0-0")
        assert out["probe"]["cohdi.io/probe-status"] == "ok" and out["probe"]["cohdi.io/probe-device-id"] == uuid
        # a device the fabric promised but the node does not have: stays Attaching, 30 s requeue
        out = cro.reconcile_attach(c, dict(base, provider={"device_id": "GPU-00000000-dead-beef-0000-000000000000", "cdi_device_id": "r"}))
        assert g.json_status(out) == oracle.emit_status("Attaching", "", "GPU-00000000-dead-beef-0000-000000000000", "r")
        assert out["requeue_after_s"] == 30 and "probe" not in out


def test_launch_count_is_kernels(cro):
    with cro.ProbeContext(sweep_bytes=16 << 20, devices=[0], read_sweeps=4, copy_sweeps=3) as c:
        c.probe_device(0)
        first = c.launch_count()
        assert first == 1 + 1 + 4 + 3 + 1      # fill + closed form + reads + copies + finalize
        c.probe_device(0)
        assert c.launch_count() - first == 1 + 1 + 4 + 3 + 1   # every probe has its own pattern, hence its own closed form


def test_probe_all_on_a_single_device(cro, coracle):
    """A one-GPU node: no NVLink rounds, no NCCL (nothing to gather from), same result as the per-device probe."""
    S = 64 << 20
    with cro.ProbeContext(sweep_bytes=S, devices=[0], read_sweeps=2, copy_sweeps=1) as c:
        res = c.probe_all()
        assert len(res) == 1
        r = res[0]
        assert r.status == 0 and r.rank == 0 and r.world == 1
        assert r.checksum == coracle.checksum(r.seed, 0, S // 8)
        assert all(x == 0 for x in r.p2p_read_ns) and all(x == 0 for x in r.p2p_write_ns)
        one = c.probe_device(0)
        assert one.gpu_uuid == r.gpu_uuid and one.nonce == r.nonce + 1
        assert one.checksum == coracle.checksum(one.seed, 0, S // 8)
        assert c.fullbox_times().host_syncs == 1


def test_multi_device_probe_all(cro, coracle):
    S, P, HOPS = 256 << 20, 64 << 20, 2048
    with cro.ProbeContext(sweep_bytes=S, p2p_bytes=P, read_sweeps=2, copy_sweeps=1, latency_hops=HOPS) as c:
        n = c.device_count()
        if n < 2:
            pytest.skip("single-GPU box")
        devs = c.enumerate()
        for rep in range(2):                     # the second call is the steady state: nothing is set up again
            res = c.probe_all()
            assert len(res) == n
            for i, r in enumerate(res):
                assert r.status == 0 and r.rank == i and r.world == n and r.fail_code == 0 and r.nonce == rep
                assert r.checksum == coracle.checksum(r.seed, 0, S // 8)
                for j in range(min(n, 8)):
                    if j == i or not r.p2p_access[j]:
                        continue
                    assert r.p2p_read_ns[j] > 0 and r.p2p_latency_ns_x16[j] > 0 and r.p2p_write_ns[j] > 0
                    assert r.p2p_ok & (1 << j)
                    prefix = coracle.checksum(res[j].seed, 0, P // 8)
                    assert r.p2p_checksum_xor[j] == prefix[0]
                    d = c.p2p_detail(i, j)
                    assert (d.read_xor, d.read_sum, d.read_wsum) == prefix == (d.expect_xor, d.expect_sum, d.expect_wsum)
                    # what i pushed into j landed intact: j found i's own prefix in its scratch half
                    assert (d.landed_xor, d.landed_sum, d.landed_wsum) == coracle.checksum(r.seed, 0, P // 8)
                    # the chase ended where the oracle's restatement of the permutation says it must
                    mi, mj = max(devs[i].device_minor, 0), max(devs[j].device_minor, 0)
                    assert d.chase_end == d.chase_expect == coracle.chase_end(mi, mj, HOPS) and d.hops == HOPS
                    assert d.read_ns == r.p2p_read_ns[j] and d.push_ns == r.p2p_write_ns[j]
            t = c.fullbox_times()
            assert t.host_syncs == n and t.rounds == (n - 1 if n % 2 == 0 else n) and t.gather_ns > 0
            assert t.p2p_ns > 0 and t.chase_ns > 0 and t.hbm_ns > 0 and t.gather == cro.GATHER_NCCL


def test_without_nccl_the_full_box_probe_degrades_to_a_host_gather(cro, coracle, monkeypatch):
    """SURVEY.md §8e, "If NCCL unavailable": host-side gather over pinned memory, reported as such — not a failed attach."""
    monkeypatch.setenv("CRO_NCCL_PATH", "off")
    S, P = 64 << 20, 16 << 20
    with cro.ProbeContext(sweep_bytes=S, p2p_bytes=P, read_sweeps=1, copy_sweeps=1, latency_hops=256) as c:
        n = c.device_count()
        if n < 2:
            pytest.skip("needs two devices")
        res = c.probe_all()
        t = c.fullbox_times()
        assert t.gather == cro.GATHER_DEGRADED and t.gather_ns == 0 and t.host_syncs == n
        assert "CRO_NCCL_PATH=off" in c.last_error()
        for i, r in enumerate(res):
            assert r.status == 0 and r.rank == i and r.checksum == coracle.checksum(r.seed, 0, S // 8)
            assert all(r.p2p_ok & (1 << j) for j in range(n) if j != i)
    monkeypatch.delenv("CRO_NCCL_PATH")
    with cro.ProbeContext(sweep_bytes=S, p2p_bytes=P, read_sweeps=1, copy_sweeps=1, latency_hops=256, flags=cro.F_SKIP_NCCL) as c:
        c.probe_all()
        assert c.fullbox_times().gather == cro.GATHER_HOST


def test_peer_push_lands_the_pushers_pattern(cro, coracle):
    """The push leg writes a's pattern prefix into the scratch half of b over NVLink; afterwards that half
    must hold exactly a's words (read back through the C ABI and compared with the oracle's generator)."""
    S, P = 64 << 20, 16 << 20
    with cro.ProbeContext(sweep_bytes=S, p2p_bytes=P, read_sweeps=1, copy_sweeps=1, latency_hops=256, flags=cro.F_SKIP_COPY) as c:
        n = c.device_count()
        if n < 2:
            pytest.skip("single-GPU box")
        res = c.probe_all()
        assert all(r.status == 0 for r in res)
        # the LAST round of the 1-factorisation pairs each device with a known partner: find it by content
        seeds = [r.seed for r in res]
        for b in range(n):
            words = c.read_words(b, S // 8, 4)                  # first words of b's scratch half
            owners = [a for a in range(n) if a != b and list(words) == [coracle.pattern_word(seeds[a], i) for i in range(4)]]
            assert len(owners) == 1, (b, words)
            tail = c.read_words(b, S // 8 + P // 8 - 4, 4)       # ...and the last words of the pushed prefix
            assert list(tail) == [coracle.pattern_word(seeds[owners[0]], P // 8 - 4 + i) for i in range(4)]


def test_oom_fails_loudly_or_degrades(cro, coracle):
    """A sweep region that does not fit (2*S = 192 GiB > 180 GB): CRO_ERR_OOM by default; with
    CRO_F_DEGRADE_ON_OOM the probe halves S until it fits and says so in the result."""
    S = 96 << 30
    import pynvml                                      # not torch: a host that loads torch AFTER libcroprobe has loaded the
    pynvml.nvmlInit()                                  # system NCCL would trip over the older libnccl.so.2 (see load_nccl)
    uuid0 = None
    with cro.ProbeContext(sweep_bytes=1 << 20, devices=[0], flags=cro.F_LAZY_ALLOC) as c0:
        uuid0 = c0.own_devices()[0].gpu_uuid.decode()
    try:
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid0)
    except TypeError:
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid0.encode())
    used_before = pynvml.nvmlDeviceGetMemoryInfo(h).used
    for _ in range(3):                                   # a failed init must release what it had already built
        with pytest.raises(cro.ProbeError) as e:
            cro.ProbeContext(sweep_bytes=S, devices=[0])
        assert e.value.code == cro.ERR_OOM
        assert "cudaMalloc" in str(e.value) and "asked for" in str(e.value)      # cro_last_error(NULL) carries the reason
    assert pynvml.nvmlDeviceGetMemoryInfo(h).used - used_before < (768 << 20)   # the CUDA context itself stays; no region leaked
    with cro.ProbeContext(sweep_bytes=S, devices=[0], flags=cro.F_DEGRADE_ON_OOM, read_sweeps=1, copy_sweeps=1) as c:
        r = c.probe_device(0)
        assert r.status == 0 and r.sweep_bytes == 48 << 30
        assert r.checksum == coracle.checksum(r.seed, 0, r.sweep_bytes // 8, threads=os.cpu_count() or 1)


def test_concurrent_callers_are_serialised_per_device(cro, coracle):
    """Reconciles for different CRs may probe the same GPU from different OS threads (cgo migrates
    goroutines): every entry point takes the device mutex and calls cudaSetDevice itself."""
    import threading
    with cro.ProbeContext(sweep_bytes=32 << 20, devices=[0], read_sweeps=2, copy_sweeps=1) as c:
        errors, results = [], []
        n_words = (32 << 20) // 8

        def worker(k):
            try:
                for i in range(4):
                    if (k + i) % 3 == 0:
                        # another thread's probe may land between two calls and move the pattern on: a read is judged
                        # against the closed form of whichever pattern was there (expected-kernel under the same lock? no —
                        # against every seed this device has had so far)
                        s = c.hbm_read_checksum(0, 1 + (k + i) % 3)
                        results.append(("read", s.checksum))
                    elif (k + i) % 3 == 1:
                        r = c.probe_device(0)
                        assert r.status == 0 and r.checksum == r.expect
                        results.append(("probe", r.seed, r.checksum))
                    else:
                        out = cro.reconcile_attach(c, {"status": {"state": "Attaching"}, "probe": True, "spec": {"type": "gpu", "model": "m", "target_node": "n"},
                                                       "provider": {"device_id": c.own_devices()[0].gpu_uuid.decode(), "cdi_device_id": "r"}})
                        assert out["status"]["state"] == "Online"
            except Exception as e:   # noqa: BLE001
                errors.append(repr(e))
        ts = [threading.Thread(target=worker, args=(k,)) for k in range(6)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert errors == [] and results
        seeds = {}
        for r in results:
            if r[0] == "probe":
                seeds[r[1]] = r[2]
                assert r[2] == coracle.checksum(r[1], 0, n_words)
        d = c.own_devices()[0]
        legal = {coracle.checksum(coracle.probe_seed(0x00C0FFEE00000000, max(d.device_minor, 0), k), 0, n_words) for k in range(64)}
        assert all(r[1] in legal for r in results if r[0] == "read")
        assert len(seeds) == sum(1 for r in results if r[0] == "probe")      # no two probes shared a nonce


def test_cli_helper_process(cro):
    """croprobe-cli: the fresh-process form (a hot-plugged GPU is invisible to an already initialised CUDA process)."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "composable-resource-operator_b200", "croprobe-cli")
    smi = shutil.which("nvidia-smi")
    if smi:
        want = subprocess.run([smi, "--query-gpu=gpu_uuid,pci.bus_id", "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
        got = subprocess.run([cli, "csv", "gpu_uuid,pci.bus_id"], capture_output=True, text=True)
        assert got.returncode == 0 and got.stdout == want
    devs = json.loads(subprocess.run([cli, "enumerate"], capture_output=True, text=True).stdout)
    uuid = devs[0]["gpu_uuid"]
    out = subprocess.run([cli, "probe", uuid, "256"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    ann = json.loads(out.stdout)
    assert ann["cohdi.io/probe-status"] == "ok" and ann["cohdi.io/probe-device-id"] == uuid
    assert subprocess.run([cli, "probe", "GPU-00000000-dead-beef-0000-000000000000"], capture_output=True).returncode == 3
    cold = json.loads(subprocess.run([cli, "cold", "0", "4096"], capture_output=True, text=True).stdout)
    assert cold["status"] == 0 and cold["cold_total_s"] > cold["warm_probe_s"] > 0
    print("cold vs warm:", cold)


def test_c_harness_on_gpu(cro):
    """The plain-C caller (what cgo compiles to) runs a probe + emit through the same ABI."""
    from test_abi import build_c_harness
    out = subprocess.run([build_c_harness(), "gpu"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "gpu ok: GPU-" in out.stdout and "cohdi.io/probe-status" in out.stdout


def test_async_probe_begin_end(cro, coracle):
    """cro_probe_begin / cro_probe_end: same result as the synchronous probe; a sweep in between drains it."""
    with cro.ProbeContext(sweep_bytes=32 << 20, devices=[0], read_sweeps=2, copy_sweeps=1) as c:
        n_words = (32 << 20) // 8
        c.probe_begin(0)
        c.probe_begin(0)                       # second begin: a second probe, queued on the device behind the first
        c.probe_begin(0)                       # third begin is a no-op (two lanes)
        r = c.probe_end(0)                     # results come out oldest first
        assert r.status == 0 and r.nonce == 0 and r.checksum == coracle.checksum(r.seed, 0, n_words)
        r2 = c.probe_end(0)
        assert r2.status == 0 and r2.nonce == 1 and r2.checksum == coracle.checksum(r2.seed, 0, n_words)
        assert r2.t_start_ns >= r.t_start_ns + r.total_ns          # back to back on the device, never interleaved
        assert c.launch_count() == 2 * (3 + 2 + 1)                 # exactly two probes ran
        rs = c.probe_end(0)                    # end without begin probes synchronously
        assert rs.status == 0 and rs.nonce == 2
        c.probe_begin(0)
        s = c.hbm_read_checksum(0, 1)          # another op first drains the in-flight probe
        assert s.checksum == coracle.checksum(c.seed(0), 0, n_words)
        r3 = c.probe_end(0)
        assert r3.status == 0 and r3.read_best_ns > 0 and r3.nonce == 3 and r3.seed == c.seed(0)


def test_storm_and_churn_with_live_probe(cro):
    """BASELINE configs 4 / 5 in miniature with the CUDA probe in the attach slot (all GPUs of the box)."""
    import random
    with cro.ProbeContext(sweep_bytes=64 << 20, read_sweeps=2, copy_sweeps=1) as ctx:
        n = ctx.device_count()
        uuids = [d.gpu_uuid.decode() for d in ctx.enumerate()]
        with cro.Cluster({"nodes": ["worker-%d" % i for i in range(n)], "probe": True}, ctx) as c:
            rng = random.Random(1)
            sizes = {}
            for i in range(24):
                sizes["req-%02d" % i] = rng.randint(1, 3)
                assert c.apply("req-%02d" % i, {"type": "gpu", "model": "NVIDIA-B200-%d" % (i // n), "size": sizes["req-%02d" % i],
                                                "target_node": "worker-%d" % (i % n)}) == ""
            st = c.run()
            assert st["requests_running"] == 24 and st["reconcile_errors"] == 0 and st["probe_failures"] == 0
            assert st["probes"] == sum(sizes.values())          # every attach was probed exactly once
            d = c.dump()
            for name, req in d["requests"].items():
                node = int(req["spec"]["target_node"].split("-")[1])
                assert all(cs["state"] == "Online" and cs["device_id"] == uuids[node] for cs in req["status"]["resources"].values())
            for name in sizes:
                c.delete(name)
            c.run()
            d = c.dump()
            assert d["requests"] == {} and d["resources"] == {}


def test_probe_by_uuid_in_process_and_through_the_helper(cro, coracle):
    """cro_probe_uuid: a device the context holds is probed in process; a device it does NOT hold — the position a GPU
    composed after cuInit is in — is probed by the helper process (fresh cuInit, CUDA_VISIBLE_DEVICES=<uuid>), and its
    512-byte verdict comes back over a pipe.  With no context at all every device goes through the helper."""
    with cro.ProbeContext(sweep_bytes=64 << 20, devices=[0], read_sweeps=2, copy_sweeps=1) as c:
        mine = c.own_devices()[0]
        node = c.enumerate()                          # the whole node, fresh
        assert any(d.gpu_uuid == mine.gpu_uuid and d.flags & cro.DEV_IN_PROCESS for d in node)
        r = cro.probe_uuid(c, mine.gpu_uuid.decode())
        assert r.status == 0 and r.gpu_uuid == mine.gpu_uuid and r.sweep_bytes == 64 << 20
        assert r.checksum == coracle.checksum(r.seed, 0, r.sweep_bytes // 8)
        others = [d for d in node if d.flags & cro.DEV_NEEDS_HELPER]
        if others:                                    # multi-GPU box: a GPU this context cannot touch
            o = others[0]
            assert o.dev_index == -1 and o.cuda_ordinal == -1
            rh = cro.probe_uuid(c, o.gpu_uuid.decode())
            assert rh.status == 0 and rh.gpu_uuid == o.gpu_uuid and rh.nonce == 0 and rh.copy_verified == rh.copy_sweeps
            assert rh.checksum == rh.expect == coracle.checksum(rh.seed, 0, rh.sweep_bytes // 8, threads=os.cpu_count() or 1)
            out = cro.reconcile_attach(c, {"status": {"state": "Attaching"}, "probe": True, "spec": {"type": "gpu", "model": "m", "target_node": "n"},
                                           "provider": {"device_id": o.gpu_uuid.decode(), "cdi_device_id": "r"}})
            assert out["status"]["state"] == "Online" and out["probe"]["cohdi.io/probe-device-id"] == o.gpu_uuid.decode()
        with pytest.raises(cro.ProbeError) as e:
            cro.probe_uuid(c, "GPU-00000000-dead-beef-0000-000000000000")
        assert e.value.code == cro.ERR_NO_DEVICE
    # no context: the helper does everything (1 GiB first sweep)
    rh = cro.probe_uuid(None, mine.gpu_uuid.decode())
    assert rh.status == 0 and rh.gpu_uuid == mine.gpu_uuid and rh.sweep_bytes == 1 << 30
    assert rh.checksum == coracle.checksum(rh.seed, 0, rh.sweep_bytes // 8, threads=os.cpu_count() or 1)


def test_illegal_knob_fails_the_init_with_the_references_wording(cro, monkeypatch):
    """composableresource_adapter.go:44: "the env variable X has an invalid value: 'v'" — same sentence, same refusal."""
    monkeypatch.setenv("CRO_TMA_READ_TILE", "12345")          # not a multiple of 16
    with pytest.raises(cro.ProbeError) as e:
        cro.ProbeContext(sweep_bytes=1 << 20, devices=[0])
    assert e.value.code == cro.ERR_INVALID_ARG and "the env variable CRO_TMA_READ_TILE has an invalid value: '12345'" in str(e.value)
    monkeypatch.setenv("CRO_TMA_READ_TILE", "16384")
    monkeypatch.setenv("CRO_TMA_READ_STAGES", "8")
    with cro.ProbeContext(sweep_bytes=256 << 20, devices=[0], read_sweeps=1, copy_sweeps=1, read_variant=cro.READ_TMA) as c:
        assert c.probe_device(0).status == 0


def test_fill_that_did_not_happen_is_caught(cro, coracle):
    """ADVICE r1: with a constant seed a fill that silently does nothing passes on the previous probe's bytes.  Here the
    region is left holding probe k's pattern and is then read against probe k+1's closed form: every component differs."""
    S = 32 << 20
    with cro.ProbeContext(sweep_bytes=S, devices=[0], read_sweeps=1, copy_sweeps=1) as c:
        r1 = c.probe_device(0)
        stale = c.hbm_read_checksum(0, 1).checksum            # what is in HBM now: probe 1's pattern
        assert stale == r1.checksum
        r2 = c.probe_device(0)
        assert r2.expect != stale and all(a != b for a, b in zip(r2.expect, stale))
        assert r2.status == 0 and r2.checksum == r2.expect


def test_live_context_follows_a_changing_node(cro, tmp_path, monkeypatch):
    """ADVICE r1 (high): the device list must not be the init-time snapshot.  A real context (device 0) is pointed at a
    fake driver registry (CRO_PROC_ROOT) holding its own GPU; GPUs are then added to and removed from that registry
    between calls and cro_enumerate / the attach reconcile must follow at once."""
    from test_inventory import put, drop, U, BUS, INFO
    with cro.ProbeContext(sweep_bytes=1 << 20, devices=[0], flags=cro.F_LAZY_ALLOC) as c0:
        me = c0.own_devices()[0]
    root = str(tmp_path)
    d = os.path.join(root, "driver", "nvidia", "gpus", "0000:1b:00.0")
    os.makedirs(d)
    with open(os.path.join(d, "information"), "w") as f:
        f.write(INFO % (7, me.gpu_uuid.decode(), "0000:1b:00.0", max(me.device_minor, 0)))
    monkeypatch.setenv("CRO_PROC_ROOT", root)
    with cro.ProbeContext(sweep_bytes=16 << 20, devices=[0], flags=cro.F_NO_NVML, read_sweeps=1, copy_sweeps=1) as c:
        assert [(x.gpu_uuid, x.flags) for x in c.enumerate()] == [(me.gpu_uuid, cro.DEV_IN_PROCESS)]
        put(root, 2)                                               # hot-plug: a GPU the CUDA context has never seen
        got = {x.gpu_uuid.decode(): x for x in c.enumerate()}
        assert set(got) == {me.gpu_uuid.decode(), U[2]} and got[U[2]].flags == cro.DEV_NEEDS_HELPER and got[U[2]].dev_index == -1
        base = {"status": {"state": "Attaching"}, "probe": False, "spec": {"type": "gpu", "model": "m", "target_node": "n"},
                "device_resource_type": "DEVICE_PLUGIN"}
        out = cro.reconcile_attach(c, dict(base, provider={"device_id": U[2], "cdi_device_id": "r"}))
        assert out["status"]["state"] == "Online"                  # the reference's membership rule sees the new GPU
        drop(root, 2)                                              # ... and it is drained off the bus again
        assert [x.gpu_uuid for x in c.enumerate()] == [me.gpu_uuid]
        out = cro.reconcile_attach(c, dict(base, provider={"device_id": U[2], "cdi_device_id": "r"}))
        assert out["status"]["state"] == "Attaching" and out["requeue_after_s"] == 30
        # the context's OWN device leaves the bus: it stops being listed (Detaching then sees visible=false)
        os.remove(os.path.join(d, "information")); os.rmdir(d)
        assert c.enumerate() == []
        out = cro.reconcile_attach(c, dict(base, provider={"device_id": me.gpu_uuid.decode(), "cdi_device_id": "r"}))
        assert out["status"]["state"] == "Attaching"


def test_metrics_text_is_prometheus_exposition(cro):
    with cro.ProbeContext(sweep_bytes=64 << 20, devices=[0], read_sweeps=1, copy_sweeps=1) as c:
        c.probe_device(0)
        c.probe_device(0)
        c.enumerate()
        text = c.metrics_text()
        uuid = c.own_devices()[0].gpu_uuid.decode()
        lines = [ln for ln in text.splitlines() if ln and not ln.startswith("#")]
        vals = {ln.rsplit(" ", 1)[0]: int(ln.rsplit(" ", 1)[1]) for ln in lines}
        assert vals["cro_probe_total"] == 2 and vals["cro_probe_failures_total"] == 0 and vals["cro_kernel_launches_total"] == 10
        key = 'cro_probe_status{gpu_uuid="%s",minor="%d"}' % (uuid, c.own_devices()[0].device_minor)
        assert vals[key] == 0 and vals[key.replace("cro_probe_status", "cro_probe_nonce")] == 1
        assert vals[key.replace("cro_probe_status", "cro_probe_copies_verified")] == 1
        assert vals[key.replace("cro_probe_status", "cro_probe_hbm_read_bytes_per_second")] > 10**11
        families = {ln.split(" ")[2] for ln in text.splitlines() if ln.startswith("# TYPE ")}
        assert all(k.split("{")[0] in families for k in vals)      # every sample belongs to a declared family


@pytest.mark.parametrize("after,half,code,index,verified", [
    (0, 0, "FAIL_COPY_SRC", 0, 0),     # the fill is corrupted: copy 0 reads something else than the pattern
    (1, 1, "FAIL_COPY_SRC", 1, 0),     # copy 0's destination (B) is corrupted: copy 1, which reads it, says so
    (2, 0, "FAIL_COPY_SRC", 2, 1),     # copy 1's destination (A): copy 0's was fine (1 verified), copy 2 trips
    (3, 1, "FAIL_READ", 0, 2),         # the last copy's destination (B): read sweep 0 re-reads it
    (4, 0, "FAIL_READ", 1, 3),         # after read 0: half A, read by read sweep 1
    (5, 0, "FAIL_NONE", 0, 3),         # after the last sweep that reads half A: nobody looks again — and nothing was written
])
def test_device_side_verdict_names_the_sweep_that_caught_it(cro, coracle, after, half, code, index, verified):
    """Fault injection INSIDE the probe (a one-word XOR kernel behind a chosen sweep of the captured graph): the finalize
    kernel's verdict must name the first sweep that read the corrupted half, and count the copies verified before it.
    Probe shape: fill, 3 copies (A->B, B->A, A->B), 2 reads (B, A)."""
    S = 32 << 20
    n = S // 8
    word = half * n + 123457
    with cro.ProbeContext(sweep_bytes=S, devices=[0], read_sweeps=2, copy_sweeps=3, inject=(after, word, 1 << 33)) as c:
        r = c.probe_device(0, allow_checksum_error=True)
        want = coracle.checksum(r.seed, 0, n)
        assert r.expect == want
        assert r.fail_code == getattr(cro, code) and (r.fail_code == 0 or r.fail_index == index), (r.fail_code, r.fail_index)
        assert r.status == (0 if code == "FAIL_NONE" else cro.ERR_CHECKSUM)
        assert r.copy_verified == verified
        if code == "FAIL_READ":
            # the struct shows the checksum of the sweep that failed: exactly one bit off in xor, the weighted sum moved by that word's weight
            w = coracle.pattern_word(r.seed, 123457)
            assert r.checksum_xor == want[0] ^ (1 << 33)
            assert r.checksum_wsum == (want[2] + ((w ^ (1 << 33)) - w) * (2 * 123457 + 1)) & MASK
        if code != "FAIL_NONE":
            assert "sweep" in cro_last_error(cro, c)


def cro_last_error(cro, c):
    import ctypes
    buf = ctypes.create_string_buffer(1024)
    cro.lib.cro_last_error(c.handle, buf, 1024)
    return buf.value.decode()


def test_probe_all_over_an_odd_number_of_devices(cro, coracle):
    """K_3: the 1-factorisation has a bye in every round (one GPU sits a round out and publishes no round events);
    every directed pair must still be read, pushed, chased and verified exactly once."""
    S, P, HOPS = 64 << 20, 16 << 20, 512
    with cro.ProbeContext(sweep_bytes=1 << 20, flags=cro.F_LAZY_ALLOC) as c0:
        total = c0.device_count()
    if total < 3:
        pytest.skip("needs three GPUs")
    with cro.ProbeContext(sweep_bytes=S, p2p_bytes=P, devices=[0, 1, 2], read_sweeps=1, copy_sweeps=1, latency_hops=HOPS) as c:
        devs = c.own_devices()
        for rep in range(2):
            res = c.probe_all()
            assert len(res) == 3 and c.fullbox_times().rounds == 3 and c.fullbox_times().host_syncs == 3
            for i, r in enumerate(res):
                assert r.status == 0 and r.world == 3 and r.p2p_ok == (7 & ~(1 << i)), (i, r.status, r.fail_code, r.fail_index, r.p2p_ok)
                for j in range(3):
                    if j == i:
                        continue
                    d = c.p2p_detail(i, j)
                    assert (d.read_xor, d.read_sum, d.read_wsum) == coracle.checksum(res[j].seed, 0, P // 8)
                    assert (d.landed_xor, d.landed_sum, d.landed_wsum) == coracle.checksum(r.seed, 0, P // 8)
                    assert d.chase_end == coracle.chase_end(max(devs[i].device_minor, 0), max(devs[j].device_minor, 0), HOPS)
