"""A fake kubelet (grpcio client) drives GetDevicePluginOptions / GetPreferredAllocation over a unix
socket, with messages laid out as vendor/k8s.io/kubelet/pkg/apis/deviceplugin/v1beta1/api.proto:28-33,
133-150 has them, against the plugin-side mirror in elastic-gpu-agent_b200/kubelet_plugin.py
(reference handlers: pkg/plugins/base.go:72-76, 94-96).

CPU: the handler calls a harness build of csrc/egpu_plugin.cc whose stand-in for the device call asks
the ORACLE (tests may link it) - this checks the message plumbing, the ID selection rule and the error
mapping.  GPU: the same conversation against the product library and a real context."""
import ctypes as C
import os
import subprocess
from concurrent import futures

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "_build", "plugin_host_harness.so")
CORE, MEM = 0, 1


def ids(gpu, units):
    return ["%d-%02d" % (gpu, u) for u in units]


def expected_ids(available, must, size, gpu):
    """the documented selection rule: must-include first, then the chosen GPU's lowest unit numbers"""
    rest = sorted((int(s.split("-")[1]), i) for i, s in enumerate(available) if s.startswith("%d-" % gpu) and s not in must)
    return list(must) + [available[i] for _, i in rest][:size - len(must)]


def oracle_choice(oracle_c, counts, size, resource, pinned=None):
    """best fit over the availability table the plugin builds (egpu_plugin.cc step 3)"""
    D = max(counts) + 1
    cap = 100 if resource == CORE else (1 << 18) - 1
    fc = np.zeros(D, np.int32)
    fm = np.zeros(D, np.int32)
    for d in range(D):
        usable = pinned is None or d == pinned
        c = min(counts.get(d, 0), cap)
        fc[d] = (c if usable else 0) if resource == CORE else (100 if usable else 0)
        fm[d] = (c if usable else 0) if resource == MEM else ((1 << 18) - 1 if usable else 0)
    rc_, rm_ = (size, 1) if resource == CORE else (1, size)
    return oracle_c.load().oracle_pick_one(C.c_void_p(fc.ctypes.data), C.c_void_p(fm.ctypes.data), D, rc_, rm_)


def conversation(stub, T, oracle_c, resource):
    opts = stub.get_options(T["Empty"]())
    assert opts.pre_start_required and opts.get_preferred_allocation_available
    # one pod, two containers: GPU 0 has 60 units left, GPU 1 30, GPU 2 25 (units shuffled on purpose)
    available = ids(0, range(40, 100)) + ids(2, range(75, 100))[::-1] + ids(1, range(0, 30))
    counts = {0: 60, 1: 30, 2: 25}
    req = T["PreferredAllocationRequest"]()
    for size, must in ((25, []), (26, []), (31, []), (20, ["0-55", "0-41"]), (61, []), (10, [])):
        c = req.container_requests.add()
        c.available_deviceIDs.extend(available)
        c.must_include_deviceIDs.extend(must)
        c.allocation_size = size
    resp = stub.get_preferred(req)
    assert len(resp.container_responses) == 6
    for cresp, creq in zip(resp.container_responses, req.container_requests):
        must = list(creq.must_include_deviceIDs)
        pinned = int(must[0].split("-")[0]) if must else None
        gpu = oracle_choice(oracle_c, counts, creq.allocation_size, resource, pinned)
        if gpu < 0:
            assert list(cresp.deviceIDs) == []          # unsatisfiable: empty preference, kubelet decides
        else:
            assert list(cresp.deviceIDs) == expected_ids(available, must, creq.allocation_size, gpu)
    # hand-checked anchors (tightest leftover, then lowest index): 25 -> GPU 2 exactly, 26 -> GPU 1, 31 -> GPU 0
    got = [list(r.deviceIDs) for r in resp.container_responses]
    assert got[0] == ids(2, range(75, 100)) and got[1] == ids(1, range(0, 26)) and got[2] == ids(0, range(40, 71))
    assert got[3][:2] == ["0-55", "0-41"] and len(got[3]) == 20 and got[4] == []
    assert got[5] == ids(2, range(75, 85))                      # a part of a GPU offered in descending order: lowest units first
    # whole-card requests: > 100 gpu-core units = allocation_size / 100 whole GPUs (pkg/plugins/gpushare.go:62-69);
    # cards 0, 2, 3 are completely available, card 1 is not
    whole = ids(0, range(100)) + ids(1, range(60)) + ids(3, range(100))[::-1] + ids(2, range(100))
    wcounts = {0: 100, 1: 60, 2: 100, 3: 100}
    wreq = T["PreferredAllocationRequest"]()
    cases = [(200, []), (300, []), (400, []), (250, []), (200, ["2-05"]), (200, ["3-99", "0-00"]), (200, ["1-07"])]
    for size, must in cases:
        c = wreq.container_requests.add()
        c.available_deviceIDs.extend(whole)
        c.must_include_deviceIDs.extend(must)
        c.allocation_size = size
    wresp = stub.get_preferred(wreq)
    for (size, must), cresp in zip(cases, wresp.container_responses):
        # expected: pinned cards first, then sequential best-fit picks of a full card among the cards left
        pins = []
        for m_ in must:
            g = int(m_.split("-")[0])
            if g not in pins:
                pins.append(g)
        chosen, ok = [], size % 100 == 0 and len(pins) <= size // 100
        for pick in range(size // 100 if ok else 0):
            left = {g: (n if g not in chosen and (pick < len(pins) and g == pins[pick] or pick >= len(pins) and g not in pins) else 0)
                    for g, n in wcounts.items()}
            g = oracle_choice(oracle_c, left, 100, resource)
            if g < 0:
                ok = False
                break
            chosen.append(g)
        if not ok:
            assert list(cresp.deviceIDs) == [], (size, must)
            continue
        exp = list(must)
        for g in chosen:
            exp += [s_ for s_ in ids(g, range(100)) if s_ not in must]
        assert list(cresp.deviceIDs) == exp, (size, must)
    got_w = [list(r.deviceIDs) for r in wresp.container_responses]
    assert got_w[0] == ids(0, range(100)) + ids(2, range(100))                 # ties among full cards: lowest index first
    assert got_w[1][200:] == ids(3, range(100)) and got_w[2] == [] and got_w[3] == [] and got_w[6] == []
    assert got_w[4][0] == "2-05" and got_w[4][100:] == ids(0, range(100))      # the pinned card first, then the best of the rest
    # a malformed ID is an RPC error, as a Go handler returning (nil, err) is
    import grpc
    bad = T["PreferredAllocationRequest"]()
    c = bad.container_requests.add()
    c.available_deviceIDs.extend(["0-00", "zz"])
    c.allocation_size = 1
    with pytest.raises(grpc.RpcError) as ei:
        stub.get_preferred(bad)
    assert ei.value.code() == grpc.StatusCode.UNKNOWN


def serve_and_talk(tmp_path, monkeypatch, handle, lib, oracle_c, resource=CORE):
    import grpc
    from elastic_gpu_agent_b200 import kubelet_plugin as kp
    T = kp.messages()
    # the socket is named relative to tmp_path: a unix socket path holds at most 107 bytes, and a deep
    # temporary directory alone can be longer than that
    monkeypatch.chdir(tmp_path)
    sock = "unix:elastic-gpushare-core.sock"      # pkg/plugins/base.go:226
    server = grpc.server(futures.ThreadPoolExecutor(max_workers=4))
    kp.add_to_server(kp.BestFitDevicePlugin(handle, resource, lib), server)
    server.add_insecure_port(sock)
    server.start()
    try:
        with grpc.insecure_channel(sock) as ch:
            conversation(kp.KubeletStub(ch), T, oracle_c, resource)
    finally:
        server.stop(0)


def test_wire_format_matches_the_v1beta1_field_numbers():
    """Serialised bytes, checked by hand against api.proto:133-150: field 1 (LEN) available_deviceIDs,
    field 2 (LEN) must_include_deviceIDs, field 3 (VARINT) allocation_size; response field 1 (LEN) deviceIDs."""
    from elastic_gpu_agent_b200 import kubelet_plugin as kp
    T = kp.messages()
    c = T["ContainerPreferredAllocationRequest"](available_deviceIDs=["0-07"], must_include_deviceIDs=["1-00"], allocation_size=25)
    assert c.SerializeToString() == b"\x0a\x040-07" + b"\x12\x041-00" + b"\x18\x19"
    r = T["PreferredAllocationRequest"](container_requests=[c])
    assert r.SerializeToString() == b"\x0a\x0e" + c.SerializeToString()
    o = T["DevicePluginOptions"](pre_start_required=True, get_preferred_allocation_available=True)
    assert o.SerializeToString() == b"\x08\x01\x10\x01"
    resp = T["ContainerPreferredAllocationResponse"](deviceIDs=["2-75"])
    assert resp.SerializeToString() == b"\x0a\x042-75"


def test_fake_kubelet_round_trip_on_cpu_harness(tmp_path, monkeypatch, oracle_c):
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "elastic-gpu-agent_b200", "csrc", "egpu_plugin.cc"), os.path.join(HERE, "plugin_host_harness.cc"), "-o", SO]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(SO)
    pick = oracle_c.load().oracle_pick_one
    cb_t = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32)
    cb = cb_t(lambda fc, fm, D, core, mem: pick(C.c_void_p(fc), C.c_void_p(fm), D, core, mem))
    lib.stub_use_callback(cb)
    try:
        serve_and_talk(tmp_path, monkeypatch, C.c_void_p(1), lib, oracle_c)
    finally:
        lib.stub_use_callback(cb_t())


@pytest.mark.gpu
def test_fake_kubelet_round_trip_on_gpu(tmp_path, monkeypatch, alloc, oracle_c, egpu):
    # the context also tracks a committed table: the RPCs must leave it alone
    alloc.set_table([100, 40, 75], [183359, 9000, 50000])
    serve_and_talk(tmp_path, monkeypatch, alloc.handle, egpu.load(), oracle_c)
    fc, fm, ov = alloc.table()
    assert fc.tolist() == [100, 40, 75] and fm.tolist() == [183359, 9000, 50000] and not ov.any()
