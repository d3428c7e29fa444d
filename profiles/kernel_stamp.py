#!/usr/bin/env python3
"""Which compiled kernels an ncu capture belongs to.

profiles/traffic.json records, per workload, the DRAM bytes and warp instructions of one step's launches.  Such a capture is only worth
quoting while the kernels it measured are the kernels that run, so every entry is stamped twice: `csrc_sha16` (hash of every file under
snap_b200/csrc/) and `sass_sha16` (hash of the SASS of the kernels the workload launches, from `cuobjdump -sass` of the built library).
bench.py quotes an entry when either stamp matches: a source change elsewhere in the translation unit (the output stage, say) leaves the
alignment kernels' SASS -- and hence their traffic -- exactly as captured.

usage: kernel_stamp.py            prints the stamps of snap_b200/csrc/libsnapgpu.so
"""
import hashlib
import json
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "snap_b200", "csrc")
LIB = os.path.join(CSRC, "libsnapgpu.so")
# cached outside the tree (bench.py may run from a read-only checkout), one file per library path
CACHE = os.path.join(tempfile.gettempdir(), "snapgpu_sass_stamps_%s.json" % hashlib.sha256(LIB.encode()).hexdigest()[:16])

# workload key prefix in traffic.json -> substring of the (mangled) names of the kernels its capture holds
GROUPS = {"single": "sg_align_kernel", "ag_d20": "sg_align_kernel", "ne_d20": "sg_align_kernel", "paired": "sg_align_paired_kernel",
          "lookup": "sg_lookup_bucket_kernel"}


def csrc_sha16():
    h = hashlib.sha256()
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(f.encode()); h.update(open(os.path.join(CSRC, f), "rb").read())
    return h.hexdigest()[:16]


def _cuobjdump():
    for c in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if c and os.path.exists(c):
            return c
    return None


def sass_stamps():
    """{kernel-name substring: sha16 of the SASS of every kernel whose name holds it} for the built library; {} when there is no
    cuobjdump or no library.  Cached in CACHE (keyed by the library's size and mtime)."""
    if not os.path.exists(LIB):
        return {}
    st = os.stat(LIB)
    key = "%d:%d" % (st.st_size, st.st_mtime_ns)
    try:
        c = json.load(open(CACHE))
        if c.get("key") == key:
            return c["stamps"]
    except Exception:
        pass
    exe = _cuobjdump()
    if not exe:
        return {}
    p = subprocess.run([exe, "-sass", LIB], capture_output=True, text=True)
    if p.returncode != 0:
        return {}
    bodies = {}
    name = None
    for line in p.stdout.split("\n"):
        s = line.strip()
        if s.startswith("Function :"):
            name = s.split(":", 1)[1].strip()
            bodies[name] = hashlib.sha256()
        elif name is not None and s.startswith("/*"):
            bodies[name].update(s.encode())
    stamps = {}
    for sub in sorted(set(GROUPS.values())):
        h = hashlib.sha256()
        n = 0
        for fn in sorted(bodies):
            if sub in fn:
                h.update(fn.encode()); h.update(bodies[fn].digest()); n += 1
        if n:
            stamps[sub] = h.hexdigest()[:16]
    try:
        json.dump({"key": key, "stamps": stamps}, open(CACHE, "w"))
    except Exception:
        pass
    return stamps


def sass_sha16_for(traffic_key):
    """The SASS stamp of the kernels behind a traffic.json key ('single_1048576reads_3000mbp' ...), or None."""
    for prefix, sub in GROUPS.items():
        if traffic_key.startswith(prefix + "_"):
            return sass_stamps().get(sub)
    return None


if __name__ == "__main__":
    print(json.dumps({"csrc_sha16": csrc_sha16(), "sass_sha16": sass_stamps()}, indent=1))
