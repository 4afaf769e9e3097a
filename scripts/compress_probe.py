"""Go/no-go probe: does generic compressible memory (cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC) make the
config-4 step loop faster?  In such memory the L2 <-> DRAM transfers of low-entropy 128 B lines can move fewer bytes;
several env-owned step buffers of config 4 are low entropy (terminated/truncated always 0, `t` the same in every env,
unsafe/count small), the state, reward and index are not.

    python scripts/compress_probe.py [--steps 2000] [--warmup 128] [--rounds 3] [--out FILE.json]

Prints the card name, power limit and CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, then times bench.py's
config-4 device path (2^24 envs, int8 layout, the 8-slot action ring, gc_step_many in 64-step calls, CUDA events)
with the env's step buffers in plain memory and in compressible memory, alternating, `--rounds` times each; then
with one buffer group at a time compressible, and the packed layout with all its step buffers compressible.  Every
arm starts from the same reset and the same ring, so every arm must end in bit-identical outputs; the probe reports
whether it does.  Each compressible allocation is read back with cuMemGetAllocationPropertiesFromHandle.

The driver is reached through ctypes (libcuda.so.1), so the probe needs nothing from the library but its env classes.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

ATTR_GENERIC_COMPRESSION_SUPPORTED = 107
COMP_GENERIC = 1
ALLOC_PINNED, LOC_DEVICE, ACCESS_RW, GRAN_RECOMMENDED = 1, 1, 3, 1


class Location(C.Structure):
    _fields_ = [("type", C.c_int), ("id", C.c_int)]


class AllocFlags(C.Structure):
    _fields_ = [("compressionType", C.c_ubyte), ("gpuDirectRDMACapable", C.c_ubyte), ("usage", C.c_ushort),
                ("reserved", C.c_ubyte * 4)]


class AllocProp(C.Structure):        # CUmemAllocationProp_v1
    _fields_ = [("type", C.c_int), ("requestedHandleTypes", C.c_int), ("location", Location),
                ("win32HandleMetaData", C.c_void_p), ("allocFlags", AllocFlags)]


class AccessDesc(C.Structure):
    _fields_ = [("location", Location), ("flags", C.c_int)]


class Driver:
    def __init__(self, device):
        self.cu = C.CDLL("libcuda.so.1")
        self.device = device

    def check(self, rc, what):
        if rc:
            raise RuntimeError(f"{what} failed: CUresult {rc}")

    def compression_supported(self):
        v = C.c_int()
        self.check(self.cu.cuDeviceGetAttribute(C.byref(v), ATTR_GENERIC_COMPRESSION_SUPPORTED, self.device),
                   "cuDeviceGetAttribute")
        return v.value

    def prop(self):
        p = AllocProp()
        p.type, p.location.type, p.location.id = ALLOC_PINNED, LOC_DEVICE, self.device
        p.allocFlags.compressionType = COMP_GENERIC
        return p

    def alloc(self, nbytes):
        """Returns (device pointer, mapped size, handle, granted compression type)."""
        p = self.prop()
        gran = C.c_size_t()
        self.check(self.cu.cuMemGetAllocationGranularity(C.byref(gran), C.byref(p), GRAN_RECOMMENDED), "granularity")
        size = -(-nbytes // gran.value) * gran.value
        h = C.c_ulonglong()
        self.check(self.cu.cuMemCreate(C.byref(h), C.c_size_t(size), C.byref(p), C.c_ulonglong(0)), "cuMemCreate")
        got = AllocProp()
        self.check(self.cu.cuMemGetAllocationPropertiesFromHandle(C.byref(got), h), "properties")
        ptr = C.c_ulonglong()
        self.check(self.cu.cuMemAddressReserve(C.byref(ptr), C.c_size_t(size), C.c_size_t(gran.value),
                                               C.c_ulonglong(0), C.c_ulonglong(0)), "cuMemAddressReserve")
        self.check(self.cu.cuMemMap(ptr, C.c_size_t(size), C.c_size_t(0), h, C.c_ulonglong(0)), "cuMemMap")
        acc = AccessDesc()
        acc.location.type, acc.location.id, acc.flags = LOC_DEVICE, self.device, ACCESS_RW
        self.check(self.cu.cuMemSetAccess(ptr, C.c_size_t(size), C.byref(acc), C.c_size_t(1)), "cuMemSetAccess")
        return ptr.value, size, h, got.allocFlags.compressionType

    def free(self, ptr, size, h):
        self.check(self.cu.cuMemUnmap(C.c_ulonglong(ptr), C.c_size_t(size)), "cuMemUnmap")
        self.check(self.cu.cuMemAddressFree(C.c_ulonglong(ptr), C.c_size_t(size)), "cuMemAddressFree")
        self.check(self.cu.cuMemRelease(h), "cuMemRelease")


class _Array:                          # __cuda_array_interface__ view of a mapped range, for torch.as_tensor
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": tuple(shape), "typestr": typestr,
                                         "version": 2, "strides": None}


TYPESTR = {"int8": "|i1", "uint8": "|u1", "int32": "<i4", "float32": "<f4"}

GROUPS_INT8 = {"t": ["_t"], "flags": ["_terminated", "_truncated", "_unsafe", "_count"], "state": ["_state"],
               "reward_index": ["_reward", "_index"]}
GROUPS_PACKED = {"t": ["_t"], "flags": ["_flags"], "state": ["_state"], "reward_index": ["_reward"]}


def run_arm(bench, drv, packed, names, steps, warmup, device):
    import torch
    batches = bench.build_batches("cfg4", device, 0, packed=packed)
    env = batches[0]["env"]
    mapped, granted = [], {}
    for name in names:
        old = getattr(env, name)
        ptr, size, h, comp = drv.alloc(old.numel() * old.element_size())
        mapped.append((ptr, size, h))
        granted[name] = comp
        new = torch.as_tensor(_Array(ptr, old.shape, TYPESTR[str(old.dtype).split(".")[1]]), device=device)
        new.copy_(old)
        setattr(env, name, new)
    if packed and env.n_states == 4:
        env._index = env._state
    env._build_views()
    torch.cuda.synchronize(device)
    ms, launches, clk, _ = bench.time_device_path(batches, steps, warmup, None, device, device.index or 0)
    out = {k: v.clone() for k, v in (("state", env._state), ("t", env._t), ("reward", env._reward))}
    out["stats"] = env._stats.clone()
    torch.cuda.synchronize(device)
    env.close()
    del env, batches
    torch.cuda.synchronize(device)
    for ptr, size, h in mapped:
        drv.free(ptr, size, h)
    torch.cuda.empty_cache()
    return ms, launches, clk, granted, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    drv = Driver(0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    head = {"device": torch.cuda.get_device_name(device), "nvidia_smi": smi,
            "generic_compression_supported": drv.compression_supported(), "steps": args.steps}
    print(json.dumps(head), flush=True)

    results, ref = [], {}

    def arm(label, packed, names):
        ms, launches, clk, granted, out = run_arm(bench, drv, packed, names, args.steps, args.warmup, device)
        key = "packed" if packed else "int8"
        same = None
        if key in ref:
            same = all(torch.equal(ref[key][k], out[k]) for k in out)
        else:
            ref[key] = out
        r = {"arm": label, "layout": key, "us_per_step": 1e3 * ms / args.steps,
             "G_env_steps_per_s": (1 << 24) * args.steps / ms / 1e6, "launches": launches, "granted": granted,
             "bit_identical_to_first": same, "sm_mhz": clk["sm_mhz"], "clock_reasons": clk["reasons"]}
        results.append(r)
        print(json.dumps(r), flush=True)

    all_int8 = [n for g in GROUPS_INT8.values() for n in g]
    all_packed = [n for g in GROUPS_PACKED.values() for n in g]
    for _ in range(args.rounds):
        arm("plain", False, [])
        arm("all", False, all_int8)
    for _ in range(2):
        for g, names in GROUPS_INT8.items():
            arm(g, False, names)
    for _ in range(args.rounds):
        arm("plain", True, [])
        arm("all", True, all_packed)

    summary = {}
    for layout in ("int8", "packed"):
        for label in ["plain", "all"] + list(GROUPS_INT8):
            v = [r["us_per_step"] for r in results if r["layout"] == layout and r["arm"] == label]
            if v:
                summary[f"{layout}/{label}"] = {"median_us": statistics.median(v), "min_us": min(v), "max_us": max(v)}
    for layout in ("int8", "packed"):
        p, a = summary[f"{layout}/plain"], summary[f"{layout}/all"]
        summary[f"{layout}/gain_all"] = p["median_us"] / a["median_us"] - 1
    print(json.dumps(summary, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"head": head, "arms": results, "summary": summary}, f, indent=1)


if __name__ == "__main__":
    main()
