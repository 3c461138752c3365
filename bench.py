#!/usr/bin/env python
"""bench.py - TensorProto encode+decode throughput on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c5] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic requests: ONE ``b200tfs_encode_requests`` call
over the batch's PredictRequests (device tensors -> wire arena) and ONE decode call over the batch's
PredictResponses (wire -> device tensors).  Workloads (BASELINE.json ``configs``):

    c2  (default)  fp32 [1024,1024], one tensor per request; a batch of 256 request/response pairs     weak
    c3             256 requests {image fp32[3,224,224], label int64[1]} -> 256 responses fp32[1000]     weak
    c4             fp16 (or bf16) [8,512,1024] cast to DT_FLOAT on encode, decoded back to fp16; 32     weak
    c5             ONE batch of 8192 requests of fp32[3,224,224], request r on GPU r // ceil(8192/N)    strong

``value`` = tensor payload bytes (encode sources + decoded tensors) per second, inputs resident in HBM, device
timed, max over ranks; ``e2e`` = the same through the host-buffer C-ABI entry points on pinned host memory with the
H2D / D2H copies inside the timed region; ``roofline`` = algorithmic bytes (SURVEY 8d: 2P+H per direction) of the
two launches of a step / their measured durations / the measured HBM copy peak; ``cpu_baseline`` = the unmodified
reference (baseline/ref_loader.py) on one host core over a bounded sample.  Every batch is larger than the 126 MB
L2 (or rotates through a ring that is), and every run ends with a bit-exact comparison of the device's wire bytes
and decoded tensors against the oracle - AFTER the timed region, on the buffers the timed steps wrote.

Multi-GPU (torchrun, one rank per GPU): requests shard by index, no collective on the data path; NCCL carries
only the barrier and the MAX (time) / SUM (bytes) reductions.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(REPO, "min-tfs-client_b200"), REPO]

L2_BYTES = 126 * 1024 * 1024
METRIC = "TensorProto encode+decode GB/s"


# ------------------------------------------------------------------------------------------------
# small wire helpers (bench-local; used to fabricate the responses the decode leg consumes - pinned to
# the oracle by tests/test_bench_cpu.py.  The oracle itself is only touched by verify / the CPU legs)
# ------------------------------------------------------------------------------------------------
def _uv(x):
    out = bytearray()
    while True:
        b = x & 0x7F
        x >>= 7
        out.append(b | (0x80 if x else 0))
        if not x:
            return bytes(out)


def _ld(tag, body):
    return bytes([tag]) + _uv(len(body)) + body


def _f32_tensor_header(shape, nbytes):
    dims = b"".join(_ld(0x12, b"\x08" + _uv(d)) for d in shape)
    return b"\x08\x01" + _ld(0x12, dims) + b"\x2a" + _uv(nbytes)


def response_wire_parts(key, shape, nbytes, model=b"default", version=1, sig=b"serving_default"):
    """(prefix, suffix) such that prefix + payload + suffix is a canonical PredictResponse."""
    th = _f32_tensor_header(shape, nbytes)
    tp_len = len(th) + nbytes
    entry_len = 1 + len(_uv(len(key))) + len(key) + 1 + len(_uv(tp_len)) + tp_len
    prefix = b"\x0a" + _uv(entry_len) + _ld(0x0A, key) + b"\x12" + _uv(tp_len) + th
    spec = _ld(0x0A, model) + _ld(0x12, b"\x08" + _uv(version)) + _ld(0x1A, sig)
    return prefix, _ld(0x12, spec)


def request_wire_parts(key, shape, nbytes, model=b"default", version=1):
    th = _f32_tensor_header(shape, nbytes)
    tp_len = len(th) + nbytes
    entry_len = 1 + len(_uv(len(key))) + len(key) + 1 + len(_uv(tp_len)) + tp_len
    spec = _ld(0x0A, model) + _ld(0x12, b"\x08" + _uv(version))
    return _ld(0x0A, spec) + b"\x12" + _uv(entry_len) + _ld(0x0A, key) + b"\x12" + _uv(tp_len) + th


def quiet_f32(a):
    """What the reference's float32 -> Python double -> float32 trip does to signalling NaNs (SURVEY Q3)."""
    u = np.ascontiguousarray(a).view(np.uint32).copy()
    u[(u & 0x7FFFFFFF) > 0x7F800000] |= 0x00400000
    return u.view(np.float32).reshape(a.shape)


SNAN_PROBE = np.array([0x7F800001, 0xFF800001, 0x7FC00001, 0x80000000], dtype=np.uint32).view(np.float32)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = str(gpu_index)
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 9 and parts[0] == self.gpu:
                self.rows.append((time.time(), parts))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [p for (t, p) in self.rows if t0 <= t <= t1 + 0.1] or [p for (_, p) in self.rows[-3:]]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sample"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# distributed plumbing (control plane only)
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(gpu_index):
    """Run this process on the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the e2e leg are
    first-touched there and the PCIe copies do not cross the socket interconnect (what `numactl --cpunodebind` would do
    per rank).  Returns a description for the bench line; does nothing when the topology cannot be read
    (B200TFS_BENCH_NUMA=0 turns it off)."""
    if os.environ.get("B200TFS_BENCH_NUMA", "1") == "0":
        return "off"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bdf = out[-12:] if len(out) >= 12 else out            # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return "unknown node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no cpus allowed on node"
        os.sched_setaffinity(0, cpus)
        return f"node {node} ({len(cpus)} cpus)"
    except Exception as e:  # noqa: BLE001 - best effort
        return f"unavailable ({type(e).__name__})"


class World:
    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.size = int(os.environ.get("WORLD_SIZE", "1"))
        self.numa = bind_to_gpu_numa_node(self.local_rank)
        self.dist = None
        self.torch = None
        if self.size > 1:
            import torch
            import torch.distributed as dist

            self.torch = torch
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def _reduce(self, x, op):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX) if self.dist else x

    def sum(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM) if self.dist else x

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# workloads: what a request / response of each BASELINE config is (pure numpy; shared by the GPU arm,
# the verification and the CPU legs)
# ------------------------------------------------------------------------------------------------
def _with_probe(a):
    """Plant three NaN encodings and a negative zero at the front of a float32 tensor: the sNaN-quieting path (Q3) is then
    checked by every verification, not only timed."""
    flat = a.reshape(-1)
    if flat.dtype == np.float32 and flat.size >= 4:
        flat[:4] = SNAN_PROBE
    return a


class Workload:
    name = ""
    title = ""
    scaling = "weak"
    sharded = False          # True: ONE global batch cut across the ranks; False: every rank runs the whole batch
    default_batch = 0        # requests per global batch
    out_dtype = None         # decode-side cast (DT_* enum) or None
    wire_dtype = None        # encode-side cast or None
    unique = 0               # distinct inputs generated (request i uses input i % unique); 0: every request its own

    def __init__(self, batch=None):
        self.batch = int(batch or self.default_batch)

    # one request: (model_name, version, [(key, ndarray), ...]) and its response
    def inputs(self, i):
        raise NotImplementedError

    def response_tensor(self, i):
        """(key, float32 ndarray) the response of request i carries."""
        raise NotImplementedError

    def seed_of(self, i):
        return i % self.unique if self.unique else i

    def unit(self, i):
        """(model, version, inputs, response key, response tensor) of request i."""
        model, version, ins = self.inputs(i)
        rk, rx = self.response_tensor(i)
        return model, version, ins, rk, rx

    def expected_decoded(self, i, rx=None):
        if rx is None:
            rx = self.response_tensor(i)[1]
        return quiet_f32(rx)


class C2(Workload):
    name, default_batch, unique = "c2", 256, 4
    title = "C2 fp32[1024,1024] single-tensor PredictRequest encode + PredictResponse decode (BASELINE.json configs[1])"
    SHAPE = (1024, 1024)

    def _x(self, i):
        return _with_probe(np.random.default_rng(self.seed_of(i)).standard_normal(self.SHAPE, dtype=np.float32))

    def inputs(self, i):
        return "default", 1, [("x", self._x(i))]

    def response_tensor(self, i):
        return "y", self._x(i)

    def unit(self, i):           # the response carries the same tensor back: generate it once
        x = self._x(i)
        return "default", 1, [("x", x)], "y", x


class C3(Workload):
    name, default_batch = "c3", 256
    title = ("C3 batch of 256 PredictRequests, inputs {image fp32[3,224,224], label int64[1]}, responses {scores fp32[1000]} "
             "(BASELINE.json configs[2])")

    def inputs(self, i):
        img = _with_probe(np.random.default_rng(i).standard_normal((3, 224, 224), dtype=np.float32))
        return "default", 1, [("image", img), ("label", np.array([i % 1000], dtype=np.int64))]

    def response_tensor(self, i):
        return "scores", _with_probe(np.random.default_rng(10000 + i).standard_normal((1000,), dtype=np.float32))


class C4(Workload):
    name, default_batch, unique = "c4", 32, 4
    title = "C4 fp16[8,512,1024] cast to DT_FLOAT on encode, DT_FLOAT response decoded back to fp16 (BASELINE.json configs[3])"
    SHAPE = (8, 512, 1024)
    wire_dtype, out_dtype = 1, 19    # DT_FLOAT on the wire, DT_HALF in memory on the way back
    np_dtype = np.float16

    def _x(self, i):
        return np.random.default_rng(self.seed_of(i)).standard_normal(self.SHAPE).astype(self.np_dtype)

    def inputs(self, i):
        return "default", 1, [("x", self._x(i))]

    def response_tensor(self, i):
        return "y", self._x(i).astype(np.float32)

    def unit(self, i):
        x = self._x(i)
        return "default", 1, [("x", x)], "y", x.astype(np.float32)

    def expected_decoded(self, i, rx=None):
        # fp16 -> fp32 -> fp16 is the identity: the tolerance is zero for a wire that carries widened fp16 / bf16 values
        return self._x(i) if rx is None else rx.astype(self.np_dtype)


class C4BF(C4):
    name = "c4bf"
    title = C4.title.replace("fp16", "bf16")
    out_dtype = 14

    def __init__(self, batch=None):
        super().__init__(batch)
        import ml_dtypes

        self.np_dtype = ml_dtypes.bfloat16


class C5(Workload):
    name, default_batch, scaling, sharded = "c5", 8192, "strong", True
    title = "C5 ONE batch of 8192 PredictRequests of fp32[3,224,224], request r on GPU r // ceil(8192/N) (BASELINE.json configs[4])"

    def _x(self, i):
        return _with_probe(np.random.default_rng(i).standard_normal((3, 224, 224), dtype=np.float32))

    def inputs(self, i):
        return "default", 1, [("image", self._x(i))]

    def response_tensor(self, i):
        return "image", self._x(i)

    def unit(self, i):
        x = self._x(i)
        return "default", 1, [("image", x)], "image", x


WORKLOADS = {"c2": C2, "c3": C3, "c4": C4, "c4bf": C4BF, "c5": C5}


# ------------------------------------------------------------------------------------------------
# the GPU arm: one rank's share of a batch, resident in HBM, through the C ABI
# ------------------------------------------------------------------------------------------------
def _parallel_map(fn, items, threads=8):
    if len(items) < 4:
        return [fn(i) for i in items]
    from concurrent.futures import ThreadPoolExecutor

    with ThreadPoolExecutor(threads) as ex:
        return list(ex.map(fn, items))


class Timer:
    """CUDA events on a context's stream (b200tfs_event_*: the stream every call of that context is ordered on)."""

    def __init__(self, N, lib, ctx):
        self.N, self.lib, self.ctx = N, lib, ctx
        self.e0, self.e1 = C.c_void_p(), C.c_void_p()
        N.check(lib.b200tfs_event_create(C.byref(self.e0)))
        N.check(lib.b200tfs_event_create(C.byref(self.e1)))

    def run(self, fn, reps):
        N, lib = self.N, self.lib
        N.check(lib.b200tfs_sync(self.ctx))
        N.check(lib.b200tfs_event_record(self.ctx, self.e0))
        for k in range(reps):
            fn(k)
        N.check(lib.b200tfs_event_record(self.ctx, self.e1))
        N.check(lib.b200tfs_event_sync(self.e1))
        N.check(lib.b200tfs_sync(self.ctx))
        ms = C.c_float(0)
        N.check(lib.b200tfs_event_elapsed_ms(self.e0, self.e1, C.byref(ms)))
        return float(ms.value)


class DeviceBatch:
    """This rank's share [lo, hi) of a workload's batch: device tensors, request structs, wire arena, response wires and
    destination slots, `slots` independent buffer sets (the timed steps rotate through them)."""

    def __init__(self, wl: Workload, device, world_size, rank, slots=None):
        from min_tfs_client import _native as N
        from min_tfs_client.codec import _Prepared
        from min_tfs_client.sharding import shard

        self.N, self.lib, self.wl = N, N.load(), wl
        lib = self.lib
        ctx = C.c_void_p()
        N.check(lib.b200tfs_create(device, C.byref(ctx)))
        if wl.out_dtype is not None:
            N.check(lib.b200tfs_set_decode_cast(ctx, wl.out_dtype))
        self.ctx = ctx
        self.device = device
        share = shard(wl.batch, world_size, rank) if wl.sharded else range(wl.batch)
        self.lo, self.hi = share.start, share.stop
        self.n = n = len(share)
        self.timer = Timer(N, lib, ctx)
        # ---- host side: generate the distinct inputs / responses of the share ----
        ids = list(share)
        uniq = sorted({wl.seed_of(i) for i in ids})
        units = _parallel_map(lambda u: wl.unit(u), uniq)
        self.host_in = {u: t[:3] for u, t in zip(uniq, units)}            # seed -> (model, version, [(key, arr)])
        self.host_resp = {u: t[3:] for u, t in zip(uniq, units)}          # seed -> (key, f32 arr)
        first = self.host_in[uniq[0]] if uniq else None
        # ---- sizes ----
        self.src_bytes = sum(a.nbytes for _, a in first[2]) if first else 0          # per request, in memory
        k0, r0 = self.host_resp[uniq[0]] if uniq else ("", np.zeros(0, np.float32))
        self.resp_prefix, self.resp_suffix = response_wire_parts(k0.encode(), r0.shape, r0.nbytes)
        self.resp_len = len(self.resp_prefix) + r0.nbytes + len(self.resp_suffix)
        self.resp_payload = r0.nbytes
        out_size = 2 if wl.out_dtype in (19, 14) else 4
        self.dst_bytes = r0.size * out_size
        self.dst_stride = (self.dst_bytes + 255) & ~255
        # B200TFS_BENCH_RESP_SHIFT (experiments): where inside its 256-byte aligned slot a response starts - e.g. the shift that
        # makes its payload 16-byte aligned, as a caller who places received bytes with that in mind would have it
        self.resp_shift = int(os.environ.get("B200TFS_BENCH_RESP_SHIFT", "0"))
        self.resp_stride = (self.resp_len + self.resp_shift + 255) & ~255
        per_slot = n * (2 * self.src_bytes + self.resp_stride + self.dst_stride)     # sources + arena + response wires + destinations
        self.slots = slots or max(1, min(64, -(-4 * L2_BYTES // max(per_slot, 1))))  # the ring's footprint is at least 4 x L2
        # ---- device: distinct inputs uploaded once, then replicated device-to-device ----
        self.keep = []
        self.sets = []
        for s in range(self.slots):
            self.sets.append(self._build_slot(ids, _Prepared))
        self.sync()
        self.footprint = self.slots * n * (self.src_bytes + self.resp_stride + self.dst_stride) + sum(st["arena_cap"] for st in self.sets)
        self.graphs = {}

    # -- plumbing --
    def malloc(self, nbytes):
        p = C.c_void_p()
        self.N.check(self.lib.b200tfs_malloc(self.ctx, max(int(nbytes), 256), C.byref(p)))
        return p.value

    def sync(self):
        self.N.check(self.lib.b200tfs_sync(self.ctx))

    def launches(self):
        n = C.c_uint64(0)
        self.N.check(self.lib.b200tfs_kernel_launches(self.ctx, C.byref(n)))
        return int(n.value)

    def _h2d(self, dst, arr):
        arr = np.ascontiguousarray(arr)
        if arr.nbytes:
            self.N.check(self.lib.b200tfs_memcpy_h2d(self.ctx, dst, arr.ctypes.data, arr.nbytes))
        self.sync()

    def _build_slot(self, ids, _Prepared):
        N, lib, wl, n = self.N, self.lib, self.wl, self.n
        st = {}
        first = self.host_in[wl.seed_of(ids[0])] if ids else ("", None, [])
        n_in = len(first[2])
        # sources: one allocation per input name, request j at j * nbytes (256-aligned strides)
        in_stride = [(a.nbytes + 255) & ~255 for _, a in first[2]]
        st["src"] = [self.malloc(n * s) for s in in_stride]
        st["resp"] = self.malloc(n * self.resp_stride + 256)
        st["dst"] = self.malloc(n * self.dst_stride + 256)
        done_seed = {}
        for j, i in enumerate(ids):
            seed = wl.seed_of(i)
            model, version, ins = self.host_in[seed]
            if seed in done_seed:
                j0 = done_seed[seed]
                for q in range(n_in):
                    N.check(lib.b200tfs_memcpy_d2d(self.ctx, st["src"][q] + j * in_stride[q], st["src"][q] + j0 * in_stride[q], ins[q][1].nbytes))
                N.check(lib.b200tfs_memcpy_d2d(self.ctx, st["resp"] + j * self.resp_stride + self.resp_shift,
                                               st["resp"] + j0 * self.resp_stride + self.resp_shift, self.resp_len))
            else:
                done_seed[seed] = j
                for q in range(n_in):
                    self._h2d(st["src"][q] + j * in_stride[q], ins[q][1])
                rk, rx = self.host_resp[seed]
                self._h2d(st["resp"] + j * self.resp_stride + self.resp_shift,
                          np.frombuffer(self.resp_prefix + rx.tobytes() + self.resp_suffix, dtype=np.uint8))
        # request structs
        ts = (N.Tensor * max(n * n_in, 1))()
        rq = (N.Request * max(n, 1))()
        preps = [_Prepared(a, k.encode(), wl.wire_dtype, False, False) for k, a in first[2]]   # dtype / dims / key of every request
        self.keep.append(preps)
        for j in range(n):
            for q, p in enumerate(preps):
                t = p.struct
                ts[j * n_in + q] = N.Tensor(data=st["src"][q] + j * in_stride[q], src_dtype=t.src_dtype, wire_dtype=t.wire_dtype, rank=t.rank,
                                            flags=t.flags, dims=t.dims, key=t.key, key_len=t.key_len, packed_len=0)
            rq[j] = N.Request(model_name=first[0].encode(), model_name_len=len(first[0].encode()), has_version=int(first[1] is not None),
                              order=N.ORDER_UPB, version=first[1] or 0, n_inputs=n_in, flags=0,
                              inputs=C.cast(C.byref(ts, j * n_in * C.sizeof(N.Tensor)), C.POINTER(N.Tensor)))
        st["ts"], st["rq"], st["n_ts"] = ts, rq, n * n_in
        self.varint = any(lib.b200tfs_dtype_field(p.struct.wire_dtype) in (7, 10, 13, 16, 17) and not (p.struct.flags & N.F_TENSOR_CONTENT)
                          for p in preps)
        need = C.c_uint64(0)   # packed-varint inputs stay unmeasured (packed_len 0): sized for b200tfs_encode_requests_async
        N.check(lib.b200tfs_request_arena_size(n, rq, C.byref(need)))
        st["arena_cap"] = int(need.value) + 256
        st["arena"] = self.malloc(st["arena_cap"])
        N.check(lib.b200tfs_memset(self.ctx, st["arena"], 0, st["arena_cap"]))
        N.check(lib.b200tfs_memset(self.ctx, st["dst"], 0, n * self.dst_stride))
        st["rec_off"], st["rec_len"] = (C.c_uint64 * max(n, 1))(), (C.c_uint64 * max(n, 1))()
        st["roff"] = (C.c_uint64 * max(n, 1))(*[j * self.resp_stride + self.resp_shift for j in range(n)])
        st["rlen"] = (C.c_uint64 * max(n, 1))(*[self.resp_len] * n)
        return st

    # -- the two halves of a step --
    def encode(self, s):
        st, N, lib = self.sets[s % self.slots], self.N, self.lib
        if self.n == 0:
            return
        if self.varint:     # packed-varint inputs: counted, framed and emitted by kernels alone - no host round trip (deferred framing)
            N.check(lib.b200tfs_encode_requests_async(self.ctx, self.n, st["rq"], st["arena"], st["arena_cap"]))
            st["results_pending"] = True
        else:
            N.check(lib.b200tfs_encode_requests(self.ctx, self.n, st["rq"], st["arena"], st["arena_cap"], st["rec_off"], st["rec_len"]))

    def encode_results(self, s):
        """Where the records of slot s lie (varint workloads learn it from the device: b200tfs_encode_results synchronises)."""
        st = self.sets[s % self.slots]
        if self.varint and self.n:
            self.encode(s)          # the results buffer belongs to the context's most recent async encode: make it this slot's
            self.N.check(self.lib.b200tfs_encode_results(self.ctx, self.n, st["rec_off"], st["rec_len"]))

    def decode(self, s):
        st, N, lib = self.sets[s % self.slots], self.N, self.lib
        if self.n == 0:
            return
        # C4: the context narrows DT_FLOAT outputs to fp16 / bf16 inside the same single launch (b200tfs_set_decode_cast)
        N.check(lib.b200tfs_decode_responses(self.ctx, st["resp"], self.n, st["roff"], st["rlen"], st["dst"], self.dst_stride))

    @property
    def capturable(self):
        return True

    def capture(self, name, body, slot_list):
        """Record body(slot) for every slot of slot_list into one CUDA graph; returns kernels launched per replay."""
        N, lib = self.N, self.lib
        for s in slot_list:
            body(s)                     # warm: sizes every scratch buffer outside the capture
        self.sync()
        l0 = self.launches()
        N.check(lib.b200tfs_capture_begin(self.ctx))
        for s in slot_list:
            body(s)
        g = C.c_void_p()
        N.check(lib.b200tfs_capture_end(self.ctx, C.byref(g)))
        self.graphs[name] = (g, self.launches() - l0)
        return self.graphs[name][1]

    def replay(self, name):
        self.N.check(self.lib.b200tfs_graph_launch(self.ctx, self.graphs[name][0]))

    # -- algorithmic bytes (SURVEY 8d: read P write P+H on encode; read P+H write P on decode) --
    def algorithmic(self):
        st = self.sets[0]
        self.encode_results(0)
        enc = sum(self.src_bytes + int(st["rec_len"][j]) for j in range(self.n))
        dec = self.n * (self.resp_len + self.dst_bytes)
        return enc, dec

    def payload_bytes(self):
        return self.n * (self.src_bytes + self.dst_bytes)

    # -- verification: AFTER the timed region, on what the timed steps left in the buffers --
    def download(self, ptr, nbytes):
        out = np.empty(int(nbytes), dtype=np.uint8)
        if nbytes:
            self.N.check(self.lib.b200tfs_memcpy_d2h(self.ctx, out.ctypes.data, ptr, int(nbytes)))
        self.sync()
        return out

    def verify(self, full=True, stride=64, chunk=256):
        """Bit-exact, AFTER the timed region: each request's wire bytes against the oracle's encoding of the same inputs and
        each decoded tensor against the response's payload (sNaNs quieted).  full=True compares every request of every
        slot and also hashes (SHA-256) all records of slot 0 on both sides; full=False compares every stride-th request."""
        from oracle import wire_oracle

        wl, n = self.wl, self.n
        checked, sha_dev, sha_ref = 0, hashlib.sha256(), hashlib.sha256()
        for s, st in enumerate(self.sets):
            if n == 0:
                break
            self.encode_results(s)
            if s == 0:
                status = (C.c_int32 * n)()
                self.N.check(self.lib.b200tfs_decode_results(self.ctx, n, None, None, None, status))
                assert all(v == 0 for v in status), "a response was not decoded"
            cache = {}
            for j0 in range(0, n, chunk):
                j1 = min(n, j0 + chunk)
                want = [j for j in range(j0, j1) if full or j % stride == 0 or j == n - 1]
                if not want:
                    continue
                lo, hi = int(st["rec_off"][j0]), int(st["rec_off"][j1 - 1] + st["rec_len"][j1 - 1])
                arena = self.download(st["arena"] + lo, hi - lo)
                dst = self.download(st["dst"] + j0 * self.dst_stride, (j1 - j0) * self.dst_stride)
                for j in want:
                    seed = wl.seed_of(self.lo + j)
                    if seed not in cache:
                        model, version, ins = self.host_in[seed]
                        ref_ins = [(k, a.astype(np.float32) if wl.wire_dtype == 1 and a.dtype != np.float32 else a) for k, a in ins]
                        if len(cache) >= 8:
                            cache.pop(next(iter(cache)))
                        cache[seed] = (wire_oracle.encode_predict_request(model, version, ref_ins),
                                       wl.expected_decoded(seed, self.host_resp[seed][1]).tobytes())
                    want_wire, want_out = cache[seed]
                    o = int(st["rec_off"][j]) - lo
                    got = arena[o: o + int(st["rec_len"][j])]
                    if full and s == 0:
                        sha_dev.update(got)
                        sha_ref.update(want_wire)
                    assert got.tobytes() == want_wire, f"request {self.lo + j} (slot {s}): encoded bytes differ from the oracle"
                    d0 = (j - j0) * self.dst_stride
                    assert dst[d0: d0 + self.dst_bytes].tobytes() == want_out, f"response {self.lo + j} (slot {s}): decoded tensor differs"
                    checked += 1
        assert sha_dev.digest() == sha_ref.digest(), "SHA-256 over every record of the batch differs from the oracle's"
        return {"requests_compared": checked, "of": n * self.slots, "sha256_all_records_slot0": sha_dev.hexdigest() if full else None,
                "against": "oracle/wire_oracle.c (pinned to the reference's goldens)",
                "when": "after the timed region, on the buffers the timed steps wrote", "snan_probe": "planted in every float32 tensor"}

    def close(self):
        self.lib.b200tfs_destroy(self.ctx)


DUMP_VALUES = 7 << 20       # values kept per dumped stream: two float32 streams stay under 64 MiB


def dump_outputs(db: DeviceBatch, s, out_dir):
    """Write what the step on ring slot `s` handed its caller to out_dir as .npy files: `request_wire` (the bytes of every
    encoded request, request after request, as float32 byte values), `request_wire_len` (float64, one per request) and
    `response_<key>` (every decoded tensor as float32, response after response).  A stream of more than DUMP_VALUES values
    keeps a fixed sample of its positions (np.random.default_rng(0) over the stream's length), so runs with the same
    arguments dump the same positions and two builds compare value for value.  Every array is finite: the NaNs the
    workloads plant in their inputs (the sNaN probe) come back decoded, so `response_<key>` holds 0 at a non-finite
    output and `response_<key>_nonfinite` (float64, one row per such output) its flat index and exact bit pattern."""
    os.makedirs(out_dir, exist_ok=True)
    st, n, wl = db.sets[s % db.slots], db.n, db.wl
    db.encode_results(s)
    rec = [(int(st["rec_off"][j]), int(st["rec_len"][j])) for j in range(n)]
    np.save(os.path.join(out_dir, "request_wire_len.npy"), np.array([ln for _, ln in rec], dtype=np.float64))
    key, rx = db.host_resp[wl.seed_of(db.lo)] if n else ("y", np.zeros(0, np.float32))
    out_dt = np.dtype(wl.np_dtype if wl.out_dtype is not None else np.float32)
    streams = (("request_wire", np.dtype(np.uint8), [(st["arena"] + o, ln) for o, ln in rec], None),
               ("response_" + key, out_dt, [(st["dst"] + j * db.dst_stride, db.dst_bytes) for j in range(n)], (n,) + rx.shape))
    for name, dt, pieces, shape in streams:
        total = sum(nb // dt.itemsize for _, nb in pieces)
        pos = np.unique(np.random.default_rng(0).integers(0, total, size=DUMP_VALUES)) if total > DUMP_VALUES else None
        vals, start = [], 0
        for ptr, nb in pieces:
            cnt = nb // dt.itemsize
            take = slice(None) if pos is None else pos[np.searchsorted(pos, start): np.searchsorted(pos, start + cnt)] - start
            if pos is None or len(take):
                vals.append(db.download(ptr, nb).view(dt)[take])
            start += cnt
        raw = np.concatenate(vals) if vals else np.zeros(0, dt)
        arr = raw.astype(np.float32)
        if shape:
            bad = np.flatnonzero(~np.isfinite(arr))
            bits = raw.view(np.dtype("u%d" % dt.itemsize))[bad]
            np.save(os.path.join(out_dir, name + "_nonfinite.npy"), np.stack([bad, bits], axis=1).astype(np.float64).reshape(-1, 2))
            arr[bad] = 0.0
        np.save(os.path.join(out_dir, name + ".npy"), arr.reshape(shape) if pos is None and shape else arr)


# ------------------------------------------------------------------------------------------------
# e2e: the same hot path through the host-buffer C-ABI entry points (what a client binds)
# ------------------------------------------------------------------------------------------------
class HostLeg:
    """`depth` sub-batches in flight, each on its own pair of contexts (encode / decode) with its own pinned buffers: the
    request tensors and the response wires start in (pinned) host memory, the request wires and decoded tensors end there."""

    def __init__(self, db: DeviceBatch, sub, depth):
        N, lib, wl = db.N, db.lib, db.wl
        self.db, self.N, self.lib = db, N, lib
        self.sub = sub = max(1, min(sub, db.n))
        self.depth = depth
        self.lanes = []
        from min_tfs_client.codec import _Prepared

        for d in range(depth):
            L = {}
            for name in ("enc", "dec"):
                ctx = C.c_void_p()
                N.check(lib.b200tfs_create(db.device, C.byref(ctx)))
                if depth > 1:      # the leg overlaps the copy directions ACROSS calls; slicing inside each call on top of that costs 3 %
                    N.check(lib.b200tfs_set_pipeline(ctx, 0, 0))
                if name == "dec" and wl.out_dtype is not None:
                    N.check(lib.b200tfs_set_decode_cast(ctx, wl.out_dtype))
                L[name] = ctx
            ids = [db.lo + (d * sub + j) % db.n for j in range(sub)]
            first = db.host_in[wl.seed_of(ids[0])]
            n_in = len(first[2])
            in_stride = [(a.nbytes + 255) & ~255 for _, a in first[2]]
            L["x"] = [N.PinnedBuffer(sub * s) for s in in_stride]
            L["resp"] = N.PinnedBuffer(sub * db.resp_stride + 256)
            L["out"] = N.PinnedBuffer(sub * db.dst_stride + 256)
            for j, i in enumerate(ids):
                model, version, ins = db.host_in[wl.seed_of(i)]
                for q in range(n_in):
                    L["x"][q].array[j * in_stride[q]: j * in_stride[q] + ins[q][1].nbytes] = ins[q][1].view(np.uint8).reshape(-1)
                rk, rx = db.host_resp[wl.seed_of(i)]
                L["resp"].array[j * db.resp_stride: j * db.resp_stride + db.resp_len] = np.frombuffer(db.resp_prefix + rx.tobytes() + db.resp_suffix, np.uint8)
            preps = [_Prepared(a, k.encode(), wl.wire_dtype, False, False) for k, a in first[2]]
            L["keep"] = preps
            ts = (N.Tensor * (sub * n_in))()
            rq = (N.Request * sub)()
            for j in range(sub):
                for q, p in enumerate(preps):
                    t = p.struct
                    ts[j * n_in + q] = N.Tensor(data=L["x"][q].ptr + j * in_stride[q], src_dtype=t.src_dtype, wire_dtype=t.wire_dtype, rank=t.rank,
                                                flags=t.flags, dims=t.dims, key=t.key, key_len=t.key_len, packed_len=0)
                rq[j] = N.Request(model_name=first[0].encode(), model_name_len=len(first[0].encode()), has_version=1, order=N.ORDER_UPB,
                                  version=first[1] or 0, n_inputs=n_in, flags=0,
                                  inputs=C.cast(C.byref(ts, j * n_in * C.sizeof(N.Tensor)), C.POINTER(N.Tensor)))
            L["ts"], L["rq"], L["ids"] = ts, rq, ids
            st0 = db.sets[0]
            wire_cap = int(sum(int(st0["rec_len"][j % db.n]) + 1024 for j in range(sub))) + 4096
            L["wire"], L["wire_cap"] = N.PinnedBuffer(wire_cap), wire_cap
            L["rec_off"], L["rec_len"] = (C.c_uint64 * sub)(), (C.c_uint64 * sub)()
            L["roff"] = (C.c_uint64 * sub)(*[j * db.resp_stride for j in range(sub)])
            L["rlen"] = (C.c_uint64 * sub)(*[db.resp_len] * sub)
            L["status"] = (C.c_int32 * sub)()
            L["busy"] = False
            self.lanes.append(L)
        self.k = 0
        self.h2d = sub * (db.src_bytes + db.resp_len)
        self.d2h = int(sum(int(st0["rec_len"][j % db.n]) for j in range(sub))) + sub * db.dst_bytes

    def _wait(self, L):
        if L["busy"]:
            N, lib = self.N, self.lib
            N.check(lib.b200tfs_decode_results(L["dec"], self.sub, None, None, None, L["status"]))   # synchronises
            N.check(lib.b200tfs_sync(L["enc"]))
            L["busy"] = False

    def step(self, sequential=False):
        N, lib, db = self.N, self.lib, self.db
        L = self.lanes[self.k % self.depth]
        self.k += 1
        self._wait(L)
        N.check(lib.b200tfs_encode_requests_host_async(L["enc"], self.sub, L["rq"], L["wire"].ptr, L["wire_cap"], L["rec_off"], L["rec_len"]))
        if sequential:      # a client: the request is on the wire before the response comes back
            N.check(lib.b200tfs_sync(L["enc"]))
        N.check(lib.b200tfs_decode_responses_host_async(L["dec"], L["resp"].ptr, self.sub, L["roff"], L["rlen"], L["out"].ptr, db.dst_stride))
        L["busy"] = True

    def drain(self):
        for L in self.lanes:
            self._wait(L)

    def verify(self):
        from oracle import wire_oracle

        db, wl = self.db, self.db.wl
        for L in self.lanes:
            L["wire"].array[:] = 0
            L["out"].array[:] = 0
        for _ in range(2 * self.depth):
            self.step()
        self.drain()
        for L in self.lanes:
            assert all(v == 0 for v in L["status"])
            for j in (0, self.sub - 1):
                seed = wl.seed_of(L["ids"][j])
                model, version, ins = db.host_in[seed]
                ref_ins = [(k, a.astype(np.float32) if wl.wire_dtype == 1 and a.dtype != np.float32 else a) for k, a in ins]
                o, ln = int(L["rec_off"][j]), int(L["rec_len"][j])
                assert L["wire"].array[o: o + ln].tobytes() == wire_oracle.encode_predict_request(model, version, ref_ins), "e2e: request bytes differ"
                assert L["out"].array[j * db.dst_stride: j * db.dst_stride + db.dst_bytes].tobytes() == \
                    wl.expected_decoded(seed, db.host_resp[seed][1]).tobytes(), "e2e: decoded tensor differs"
        return True

    def close(self):
        for L in self.lanes:
            self.lib.b200tfs_destroy(L["enc"])
            self.lib.b200tfs_destroy(L["dec"])
            for b in L["x"] + [L["resp"], L["out"], L["wire"]]:
                b.free()


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload, n_on_rank=None):
    """dram read+write bytes per launch of the step's dominant kernel(s) (every captured kernel within 2x of the largest: the
    C2 / C5 step has two, encode and decode; the C3 step one), averaged, from the newest committed ncu --set full summary that has
    entries for this workload (profiles/rNN_ncu_summary.json, written by tools/ncu_summary.py).  C5 was captured on the per-GPU
    share at N=8 (1024 requests); another share is scaled by its request count and says so."""
    import glob

    unit = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tag, scale, note = workload, 1.0, None
    if workload == "c5":
        tag = "c5share"
        if n_on_rank and n_on_rank != 1024:
            scale, note = n_on_rank / 1024.0, f"captured on 1024 requests, scaled to this rank's {n_on_rank}"
    for path in sorted(glob.glob(os.path.join(REPO, "profiles", "r*_ncu_summary.json")), reverse=True):
        with open(path) as fh:
            caps = [c for c in json.load(fh).get("full_capture", []) if c.get("workload", "c2_single") == tag]
        per = {}
        for c in caps:
            r, w = c.get("dram__bytes_read.sum"), c.get("dram__bytes_write.sum")
            if r and w:
                per.setdefault(c["kernel"], []).append(float(r["value"]) * unit.get(r["unit"], 1) + float(w["value"]) * unit.get(w["unit"], 1))
        if per:
            avg = {k: sum(v) / len(v) for k, v in per.items()}
            top = max(avg.values())
            dom = {k: v * scale for k, v in avg.items() if v * 2 >= top}
            src = {"source": os.path.relpath(path, REPO), "per_kernel_bytes": dom}
            if note:
                src["note"] = note
            return sum(dom.values()) / len(dom), src
    return None, None


# ------------------------------------------------------------------------------------------------
# one workload on this rank -> the pieces of the bench line
# ------------------------------------------------------------------------------------------------
def run_workload(wl: Workload, world: World, steps, warmup, e2e_steps, full_verify, sampler=None, e2e=True, dump_dir=None):
    peak, peak_src = peaks()
    db = DeviceBatch(wl, world.local_rank, world.size, world.rank)
    assert db.footprint > L2_BYTES or db.n == 0, "the batch ring must exceed L2"
    step = lambda s: (db.encode(s), db.decode(s))   # noqa: E731
    for w in range(max(warmup, 3)):
        step(w)
    db.sync()
    mode = "eager"
    per_replay = 0
    if db.capturable and db.n:
        ring = list(range(db.slots))
        per_replay = db.capture("step", step, ring)             # one replay = `slots` steps
        db.capture("enc", lambda s: db.encode(s), ring)
        db.capture("dec", lambda s: db.decode(s), ring)
        mode = "cuda graph replay"
        full, rem = divmod(steps, db.slots)
        if rem:
            db.capture("step_rem", step, ring[:rem])

        def timed(_):
            for _k in range(full):
                db.replay("step")
            if rem:
                db.replay("step_rem")
        db.timer.run(timed, 1)                                   # untimed: uploads the graphs
        reps = 1
    else:
        timed, reps = step, steps
    if sampler:
        sampler.start()
        time.sleep(0.3)
    world.barrier()
    l0 = db.launches()
    t0 = time.time()
    ms = db.timer.run(timed, reps)
    t1 = time.time()
    world.barrier()
    launches = (db.launches() - l0) if mode == "eager" else per_replay * (steps // db.slots) + (db.graphs["step_rem"][1] if steps % db.slots else 0)
    clocks = sampler.stop(t0, t1) if sampler else None
    if dump_dir and world.rank == 0:
        dump_outputs(db, steps - 1, dump_dir)                   # the last timed step ran on slot (steps - 1) % slots
    ms_max = world.max(ms)
    payload = world.sum(float(db.payload_bytes() * steps))
    value = payload / (ms_max * 1e-3) / 1e9
    # ---- roofline: the two launches of a step, each timed alone over the same ring ----
    enc_alg, dec_alg = db.algorithmic()
    reps_k = max(3, min(steps, 20))
    if mode == "eager":
        t_enc = db.timer.run(lambda k: db.encode(k), reps_k) / reps_k
        t_dec = db.timer.run(lambda k: db.decode(k), reps_k) / reps_k
    else:
        db.timer.run(lambda k: db.replay("enc"), 1)
        t_enc = db.timer.run(lambda k: db.replay("enc"), reps_k) / (reps_k * db.slots)
        db.timer.run(lambda k: db.replay("dec"), 1)
        t_dec = db.timer.run(lambda k: db.replay("dec"), reps_k) / (reps_k * db.slots)
    enc_kernel = "move_kernel" + (" (+ venc_len, frame_requests_kernel, venc_emit for the int64 labels: deferred framing, no host round trip)" if db.varint else "")
    dec_kernel = ("decode_fused_staged_kernel" if db.resp_len * db.n > 148 * 8 * 32768 else "decode_fused_kernel") + \
        ("" if wl.out_dtype is None else " (DT_FLOAT outputs narrowed to fp16 / bf16 in the same launch: b200tfs_set_decode_cast)")
    step_alg = enc_alg + dec_alg
    achieved = step_alg / ((t_enc + t_dec) * 1e-3) / 1e9 if db.n else 0.0
    traffic, traffic_src = ncu_traffic(wl.name, db.n)
    roofline = {
        "bound": "hbm", "kernel": f"{enc_kernel} (encode) / {dec_kernel} (decode)", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": step_alg / 2, "avg_launch_us": (t_enc + t_dec) / 2 * 1e3,
        "encode": {"launch_us": t_enc * 1e3, "algorithmic_bytes": enc_alg, "frac": enc_alg / (t_enc * 1e-3) / 1e9 / peak if db.n else 0.0},
        "decode": {"launch_us": t_dec * 1e3, "algorithmic_bytes": dec_alg, "frac": dec_alg / (t_dec * 1e-3) / 1e9 / peak if db.n else 0.0},
        "step_vs_launches": {"ms_per_step_this_rank": ms / steps, "encode_plus_decode_ms": t_enc + t_dec},
        "peak_note": "peak is the driver's torch copy_ measurement over 2 GiB; a fraction above 1 means these kernels move bytes faster than that copy kernel "
                     "does (nominal HBM3e: 8 TB/s, see frac_of_nominal_8000)",
        "how": f"this rank's share ({db.n} requests + {db.n} responses per step); each of the step's two calls timed alone over the same ring "
               f"({mode}), CUDA events on the context's stream; frac = algorithmic bytes of both / their summed durations / peak",
    }
    # ---- e2e through the host-buffer entry points ----
    e2e_line = None
    if e2e and db.n:
        sub_mb = int(os.environ.get("B200TFS_E2E_SUB_MB", "128"))
        sub = max(1, min(db.n, (sub_mb << 20) // max(db.src_bytes + db.resp_len, 1)))   # ~128 MB of H2D per sub-batch (64: 40.2 GB/s, 128: 41.6 on C2)
        depth = int(os.environ.get("B200TFS_E2E_DEPTH", "4"))
        leg = HostLeg(db, sub, depth)
        leg.verify()
        for _ in range(depth):
            leg.step()
        leg.drain()
        n_sub = max(depth * 2, min(e2e_steps, 400))
        world.barrier()

        def region(_):
            for _k in range(n_sub):
                leg.step()
            leg.drain()
        e_ms = world.max(db.timer.run(region, 1))      # events on this rank's (idle) main stream bracket the leg's streams + the host drain
        units = n_sub * sub
        e_payload = world.sum(float(units * (db.src_bytes + db.dst_bytes)))
        per_step_units = db.n
        e2e_line = {"value": e_payload / (e_ms * 1e-3) / 1e9, "unit": "GB/s",
                    "h2d_bytes_per_step": int(leg.h2d / sub * per_step_units), "d2h_bytes_per_step": int(leg.d2h / sub * per_step_units),
                    "ms_per_step": e_ms / units * per_step_units, "requests_timed": units, "sub_batch": sub, "in_flight": depth,
                    "how": "b200tfs_encode_requests_host_async + b200tfs_decode_responses_host_async (+ b200tfs_decode_results) on pinned host buffers: "
                           "request tensors and response wires H2D, request wires and decoded tensors D2H, all inside the timed region; "
                           f"sub-batches of {sub} requests, {depth} in flight on separate contexts so the two copy directions overlap "
                           "(intra-call slicing switched off on these contexts: b200tfs_set_pipeline(ctx, 0, 0))"}
        leg.close()
        if wl.name == "c2":
            # ONE pair at a time, nothing else in flight: what a caller of the drop-in API sees on one request.  The two calls
            # of the pair slice their copies and kernels over three streams each (b200tfs.h, "Pipelining inside ONE call").
            one = HostLeg(db, 1, 1)
            for _ in range(3):
                one.step()
            one.drain()
            pairs = 50

            def one_region(_):
                for _k in range(pairs):
                    one.step(sequential=True)
                    one.drain()
            o_ms = db.timer.run(one_region, 1)
            calls = C.c_uint64()
            db.N.check(db.lib.b200tfs_pipelined_calls(one.lanes[0]["enc"], C.byref(calls)))
            e2e_line["one_pair_at_a_time"] = {"value": pairs * (db.src_bytes + db.dst_bytes) / (o_ms * 1e-3) / 1e9, "unit": "GB/s",
                                              "us_per_pair": o_ms / pairs * 1e3, "in_flight": 1, "sliced_encode_calls": int(calls.value),
                                              "how": "this rank only; encode one request (host waits), then decode one response (host waits): a client's sequence"}
            one.close()
    # ---- parity, after the timed region ----
    parity = db.verify(full=full_verify)
    out = {"value": value, "ms_per_step": ms_max / steps, "gpu_launches": launches, "mode": mode, "roofline": roofline, "e2e": e2e_line,
           "parity": parity, "clocks": clocks,
           "config": {"workload": wl.title, "requests_per_step": wl.batch, "requests_on_this_rank": db.n,
                      "payload_bytes_per_step": int(world.sum(float(db.payload_bytes()))), "ring_slots": db.slots, "ring_bytes": db.footprint,
                      "l2": f"each rank's buffers ({db.footprint >> 20} MiB over {db.slots} slot(s)) exceed the 126 MiB L2; steps rotate through the slots",
                      "timed_region": mode, "wire_mode": "typed fields (float_val / int64_val), sNaN quieting on: bit-exact vs the reference",
                      "sharding": ("one batch cut by request index across the ranks (r // ceil(n/G)), no collective" if wl.sharded
                                   else "every rank runs the whole batch on its own GPU (independent requests), no collective"),
                      "cpu_binding": world.numa}}
    db.close()
    return out


def c2_single_request_latency(world):
    """One 4 MiB request / response per launch on one stream, back to back from a CUDA graph over a ring > L2: the latency
    figure of C2 (a 4 MiB tensor is below the HBM bandwidth-delay product, DESIGN.md 4.1)."""
    wl = C2(batch=48)
    db = DeviceBatch(wl, world.local_rank, 1, 0, slots=1)
    N, lib = db.N, db.lib
    st = db.sets[0]
    n = db.n
    peak, _ = peaks()
    db.encode(0)                 # the batch calls: fill rec_len (every request of C2 has the same length) and size every scratch
    db.decode(0)                 # buffer of the context before the first graph is captured (they may not move afterwards)
    db.sync()
    one_cap = int(st["rec_len"][0]) + 4096
    one_req = [C.cast(C.byref(st["rq"], j * C.sizeof(N.Request)), C.POINTER(N.Request)) for j in range(n)]
    arenas = [db.malloc(one_cap) for _ in range(n)]
    ro, rl = (C.c_uint64 * 1)(), (C.c_uint64 * 1)()
    offs = [(C.c_uint64 * 1)(j * db.resp_stride + db.resp_shift) for j in range(n)]
    lens = (C.c_uint64 * 1)(db.resp_len)

    if os.environ.get("B200TFS_BENCH_SEED_TEMPLATE") == "1":
        # experiments with a build whose kernels cannot walk (tools/decode_latency_probe.py): one host-buffer decode of response 0
        # first - the library walks it on the host and leaves the template for the device-wire launches that follow
        seed = wl.seed_of(0)
        rk, rx = db.host_resp[seed]
        hw = N.PinnedBuffer(db.resp_len)
        hw.array[:] = np.frombuffer(db.resp_prefix + rx.tobytes() + db.resp_suffix, np.uint8)
        ho = N.PinnedBuffer(db.dst_stride)
        N.check(lib.b200tfs_decode_responses_host_async(db.ctx, hw.ptr, 1, (C.c_uint64 * 1)(0), lens, ho.ptr, db.dst_stride))
        db.sync()

    def enc(j):
        N.check(lib.b200tfs_encode_requests(db.ctx, 1, one_req[j], arenas[j], one_cap, ro, rl))

    def dec(j):
        N.check(lib.b200tfs_decode_responses(db.ctx, st["resp"], 1, offs[j], lens, st["dst"] + j * db.dst_stride, db.dst_stride))
    out = {}
    for name, body in (("encode", enc), ("decode", dec)):
        db.capture(name, body, list(range(n)))
        db.timer.run(lambda k: db.replay(name), 3)
        reps = 20
        us = db.timer.run(lambda k: db.replay(name), reps) / (reps * n) * 1e3
        alg = db.src_bytes + int(st["rec_len"][0]) if name == "encode" else db.resp_len + db.dst_bytes
        out[name] = {"launch_us": us, "algorithmic_bytes": alg, "frac": alg / (us * 1e-6) / 1e9 / peak}
    out["how"] = f"graph of {n} back-to-back single-request launches on one stream over {n} buffer sets ({db.footprint >> 20} MiB > L2), CUDA events"
    a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
    N.check(lib.b200tfs_decode_stats(db.ctx, C.byref(a), C.byref(b), C.byref(c)))
    out["decode_records_served_by"] = {"template_in_parameters": a.value, "template_in_device_memory": b.value, "tag_walk": c.value}
    db.close()
    return out


# ------------------------------------------------------------------------------------------------
# CPU legs: the unmodified reference (baseline/ref_loader.py), the only place oracle/ + baseline/ are touched
# ------------------------------------------------------------------------------------------------
_REF = {}


def _reference():
    """(ndarray_to_tensor_proto, tensor_proto_to_ndarray, PredictRequest, PredictResponse, kind, origin)"""
    if not _REF:
        from tensorflow_serving.apis.predict_pb2 import PredictRequest, PredictResponse
        try:
            from baseline import ref_loader

            t, origin = ref_loader.load()
            _REF.update(enc=t.ndarray_to_tensor_proto, dec=t.tensor_proto_to_ndarray, kind="reference", origin=origin)
        except ImportError as exc:
            from oracle import ref_port

            _REF.update(enc=ref_port.to_tensor_proto, dec=ref_port.from_tensor_proto, kind="port",
                        origin=f"oracle/ref_port.py (the reference is not staged: {exc})")
        _REF.update(PredictRequest=PredictRequest, PredictResponse=PredictResponse)
    return _REF


def _cpu_unit(args):
    """One request encoded + its response decoded on one core, the way the reference does it: ndarray_to_tensor_proto per
    input, CopyFrom into request.inputs[k] (requests.py:41-48), SerializeToString (pb2_grpc.py:52); FromString (:53) and
    tensor_proto_to_ndarray per output (tensors.py:42-46).  Returns (seconds, payload bytes)."""
    wl_name, i = args
    R = _reference()
    wl = _cpu_unit.cache.get(wl_name)
    if wl is None:
        wl = _cpu_unit.cache[wl_name] = WORKLOADS[wl_name]()
    model, version, ins, rk, rx = wl.unit(wl.seed_of(i))
    src_payload = sum(a.nbytes for _, a in ins)
    if wl.wire_dtype == 1:      # C4: the reference cannot encode float16 (TypeError, SURVEY Q6): it is handed x.astype(float32)
        ins = [(k, a.astype(np.float32)) for k, a in ins]
    pre, suf = response_wire_parts(rk.encode(), rx.shape, rx.nbytes)
    resp = pre + rx.tobytes() + suf          # fabricating the response is not part of the measured path
    t0 = time.perf_counter()
    request = R["PredictRequest"]()
    request.model_spec.name = model
    if version is not None:
        request.model_spec.version.value = version
    for k, v in ins:
        request.inputs[k].CopyFrom(R["enc"](v))
    wire = request.SerializeToString()
    response = R["PredictResponse"].FromString(resp)
    outs = {k: R["dec"](v) for k, v in response.outputs.items()}
    if wl.out_dtype is not None:
        outs = {k: v.astype(wl.np_dtype) for k, v in outs.items()}
    t1 = time.perf_counter()
    assert len(wire) > rx.nbytes // 2 and outs[rk].shape == rx.shape
    return t1 - t0, src_payload + outs[rk].nbytes


_cpu_unit.cache = {}


def cpu_baseline(wl_name, budget_s=12.0, max_units=64):
    """1 core: as many whole request/response units of the workload as fit ~budget_s of CPU work."""
    t, units, payload = 0.0, 0, 0
    while units < 2 or (t + t / units <= budget_s and units < max_units):
        dt, pb = _cpu_unit((wl_name, units))
        t += dt
        payload += pb
        units += 1
    R = _reference()
    return {"value": payload / t / 1e9, "unit": "GB/s", "cores": 1, "kind": R["kind"],
            "sample": f"{units} request/response units of {wl_name} through {R['origin']}, {t:.2f} s on one core"}


def cpu_c_oracle(units=8):
    """The plain-C oracle (memcpy-class) on one core, C2 units: context for the Python reference's number."""
    from oracle import wire_oracle

    x = np.random.default_rng(0).standard_normal((1024, 1024), dtype=np.float32)
    resp = wire_oracle.build_predict_response([("y", x)])
    t0 = time.perf_counter()
    for _ in range(units):
        wire_oracle.encode_predict_request("default", 1, [("x", x)])
        wire_oracle.decode_predict_response(resp)
    t = time.perf_counter() - t0
    return {"value": units * 2 * 4194304 / t / 1e9, "unit": "GB/s", "cores": 1, "kind": "port (plain C, oracle/wire_oracle.c)"}


def host_cores():
    """Cores this process may really use: the affinity mask, cut by the cgroup CPU quota and by the physical core count
    (SMT siblings add little to a per-element Python loop)."""
    aff = sorted(os.sched_getaffinity(0))
    info = {"affinity": len(aff)}
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:  # noqa: BLE001
            continue
    info["cgroup_quota"] = quota
    phys = set()
    try:
        for cpu in aff:
            base = f"/sys/devices/system/cpu/cpu{cpu}/topology/"
            phys.add((open(base + "physical_package_id").read().strip(), open(base + "core_id").read().strip()))
    except Exception:  # noqa: BLE001
        phys = set()
    info["physical"] = len(phys) or None
    n = len(aff)
    if quota:
        n = min(n, max(1, int(quota)))
    if phys:
        n = min(n, len(phys))
    info["used"] = max(1, n)
    return info


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import multiprocessing as mp

    wl_name = args.workload
    cores = host_cores()
    workers = int(os.environ.get("B200TFS_REF_WORKERS", cores["used"]))
    one_dt, one_pb = _cpu_unit((wl_name, 0))          # also warms the import in the parent (forked workers inherit it)
    per_worker = max(1, int(round(0.5 / max(one_dt, 1e-3))))    # ~0.5 s of work per worker per step
    per_step = workers * per_worker
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    with mp.get_context("fork").Pool(workers) as pool:
        job = [(wl_name, u) for u in range(per_step)]
        for _ in range(warmup):
            pool.map(_cpu_unit, job, chunksize=per_worker)
        t0 = time.perf_counter()
        busy, payload = 0.0, 0
        for _s in range(steps):
            for dt, pb in pool.map(_cpu_unit, job, chunksize=per_worker):
                busy += dt
                payload += pb
        wall = time.perf_counter() - t0
    value = payload / wall / 1e9
    one_core = one_pb / one_dt / 1e9
    R = _reference()
    wl = WORKLOADS[wl_name]()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": wall / steps * 1e3, "higher_is_better": True, "scaling": wl.scaling,
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl.title, "step": f"{per_step} request/response units per step ({per_worker} per worker x {workers} workers): "
                                                  "a bounded sample of the same workload"},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": workers, "kind": R["kind"],
                         "sample": f"{steps} steps x {per_step} units, multiprocessing pool of {workers} workers, {R['origin']}",
                         "one_core_gbs": one_core, "parallel_efficiency": value / (one_core * workers), "worker_busy_fraction": busy / (wall * workers),
                         "host": cores},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def python_api_leg(world):
    """The drop-in Python API on numpy arrays / bytes objects (wall clock): pageable, pinned, device-resident inputs."""
    try:
        from min_tfs_client.codec import Codec

        wl = C2()
        model, version, ins = wl.inputs(0)
        x = ins[0][1]
        pre, suf = response_wire_parts(b"y", x.shape, x.nbytes)
        resp = pre + x.tobytes() + suf
        codec = Codec(world.local_rank)
        out = {}
        want = request_wire_parts(b"x", x.shape, x.nbytes) + quiet_f32(x).tobytes()

        def clock(enc, dec, reps=20):
            for _ in range(3):
                w, y = enc(), dec()
            assert bytes(w) == want and np.asarray(y).tobytes() == quiet_f32(x).tobytes()
            t0 = time.perf_counter()
            for _ in range(reps):
                enc()
                dec()
            dt = (time.perf_counter() - t0) / reps
            return {"value": 2 * x.nbytes / dt / 1e9, "unit": "GB/s", "ms_per_pair": dt * 1e3}
        out["pageable"] = clock(lambda: codec.encode_predict_request("default", {"x": x}, 1), lambda: codec.decode_predict_response(resp)[0]["y"])
        if hasattr(codec, "pinned_empty"):
            xp = codec.pinned_empty(x.shape, x.dtype)
            xp[...] = x
            rp = codec.pinned_empty((len(resp),), np.uint8)
            rp[...] = np.frombuffer(resp, np.uint8)
            yp = codec.pinned_empty(x.shape, x.dtype)
            out["pinned"] = clock(lambda: codec.encode_predict_request("default", {"x": xp}, 1, out="pinned"),
                                  lambda: codec.decode_predict_response(rp, out={"y": yp})[0]["y"])
        if hasattr(codec, "device_array"):
            xd = codec.device_array(x)
            out["device_resident_input"] = clock(lambda: codec.encode_predict_request("default", {"x": xd}, 1),
                                                 lambda: codec.decode_predict_response(resp)[0]["y"])
        out["how"] = "min_tfs_client.codec.Codec.encode_predict_request + decode_predict_response, one C2 pair per call, wall clock"
        codec.close()
        return out
    except Exception as exc:  # pragma: no cover
        return {"error": repr(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps; one step = one encode call + one decode call over the batch")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="requests per global batch (default: the workload's own)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=64, help="sub-batches timed by the e2e leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="default c2 run only: skip the short c3 / c4 / c5 passes reported under `workloads`")
    ap.add_argument("--verify", default="full", choices=["full", "sample"], help="parity check after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the request wires and decoded tensors of the last timed step "
                                                          "(rank 0's share; a fixed sample of a large batch) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":   # CPU only: rank 0 works alone, nobody needs a process group
        run_reference(args)
        return
    # stdout carries exactly ONE JSON line: park fd 1 on stderr while libraries (NCCL prints its version) are chatty
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    world = World()
    warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload](args.batch or None)
    sampler = ClockSampler(world.local_rank)
    res = run_workload(wl, world, args.steps, warmup, args.e2e_steps, full_verify=(args.verify == "full"), sampler=sampler,
                       dump_dir=args.dump_outputs)
    extras = {}
    if args.workload == "c2":
        if not args.no_extra:
            for name in ("c3", "c4", "c5"):
                try:
                    r = run_workload(WORKLOADS[name](), world, steps=5, warmup=3, e2e_steps=16, full_verify=False if name == "c5" else True)
                    extras[name] = {"value": r["value"], "unit": "GB/s", "ms_per_step": r["ms_per_step"], "scaling": WORKLOADS[name].scaling,
                                    "roofline_frac": r["roofline"]["frac"], "encode_frac": r["roofline"]["encode"]["frac"],
                                    "decode_frac": r["roofline"]["decode"]["frac"], "e2e": r["e2e"]["value"] if r["e2e"] else None,
                                    "requests_per_step": r["config"]["requests_per_step"], "mode": r["mode"], "parity": r["parity"],
                                    "steps": 5, "note": f"short pass; the full line is `python bench.py --workload {name}`"}
                except Exception as exc:  # noqa: BLE001
                    extras[name] = {"error": repr(exc)}
        try:
            res["roofline"]["single_request"] = c2_single_request_latency(world)
        except Exception as exc:  # noqa: BLE001
            res["roofline"]["single_request"] = {"error": repr(exc)}
    if world.rank == 0:
        e2e = res["e2e"] or {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        if args.workload == "c2":
            e2e["python_api"] = python_api_leg(world)
        line = {
            "metric": METRIC, "value": res["value"], "unit": "GB/s", "n_gpus": world.size, "steps": args.steps, "warmup": warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": res["config"], "roofline": res["roofline"], "e2e": e2e, "gpu_launches": res["gpu_launches"],
            "clocks": res["clocks"], "parity": res["parity"],
        }
        if extras:
            line["workloads"] = extras
        if world.size == 1 and not args.no_cpu:
            cb = cpu_baseline(args.workload)
            cb["c_oracle_1core_gbs"] = cpu_c_oracle(4)["value"]
            line["cpu_baseline"] = cb
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    world.close()


if __name__ == "__main__":
    main()
