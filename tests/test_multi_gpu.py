"""The multi-device pieces of the C ABI (SURVEY 8e): a group of devices driven by one process, the index broadcast over NCCL, the
counters all-reduce, and the compiled drop-in feeding two devices from two worker threads.  Needs >= 2 CUDA devices (`gpurun --gpus 2`);
skipped on a single-GPU box."""
import os
import subprocess

import numpy as np
import pytest

from conftest import OPTION_SETS, differing

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GPU_BIN = os.path.join(ROOT, "oracle", "_ref", "snap-aligner-gpu")


@pytest.fixture(scope="module")
def engine2():
    from snap_b200 import engine as e
    if e.lib().snapgpu_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    return e


@pytest.mark.gpu
def test_group_broadcast_and_allreduce(engine2, small_cfg, reflib):
    e = engine2
    g = e.Group([0, 1])
    ix0 = e.Index.open(small_cfg.idx, device=0)
    copies = g.broadcast_index(ix0)
    assert len(copies) == 2 and copies[1].device == 1
    a, b = copies[0].info(), copies[1].info()
    assert (a.countOfBases, a.hashTableSlots, a.overflowTableSize, a.reserved) == (b.countOfBases, b.hashTableSlots, b.overflowTableSize, b.reserved)
    # read-sharded: each device aligns half of the reads against its own copy; results = the single-device ones, counters add up
    rb = small_cfg.reads["noisy150"]
    p = e.default_params(maxDist=14)
    whole, wctr = e.SingleAligner(ix0, p, 4096).align(rb)
    half = rb.n // 2
    parts = [rb.slice(0, half), rb.slice(half, rb.n)]
    res, ctrs = [], []
    for k in range(2):
        al = e.SingleAligner(copies[k], p, 4096)
        r, c = al.align(parts[k])
        al.close()
        res.append(r)
        ctrs.append([c[f] for f in e.COUNTER_FIELDS] + c["mapqHistogram"])
    assert differing(whole, np.concatenate(res)) == []
    summed = g.allreduce_counters(np.array(ctrs, dtype=np.int64))
    assert np.array_equal(summed[0], summed[1])
    tot = e.counters_dict(summed[0])
    for f in ("totalReads", "singleHits", "multiHits", "notFound", "nHashTableLookups", "lvCalls", "affineGapCalls", "mapqHistogram"):
        assert tot[f] == wctr[f], f
    # the peer-copy form gives the same image
    rep = ix0.replicate(1)
    r2, _ = e.SingleAligner(rep, p, 4096).align(parts[1])
    assert differing(res[1], r2) == []
    rep.close(); copies[1].close(); ix0.close(); g.close()


@pytest.mark.gpu
def test_snap_aligner_gpu_feeds_two_devices(engine2, tmp_path, small_cfg, reflib):
    """`snap-aligner-gpu single ... -t 4` on a two-GPU box: threads 0 and 2 feed device 0, threads 1 and 3 device 1; the records and the
    printStats totals are those of stock `snap-aligner -t 1`."""
    import re
    reads = small_cfg.reads["std150"]
    fq = str(tmp_path / "r.fq")
    reads.write_fastq(fq)
    stock, gpu = str(tmp_path / "stock.sam"), str(tmp_path / "gpu.sam")
    so = subprocess.run([reflib.SNAP_ALIGNER, "single", small_cfg.idx, fq, "-o", stock, "-t", "1"], capture_output=True, text=True)
    env = dict(os.environ, SNAPGPU_EXT_BATCH_READS="128")
    go = subprocess.run([GPU_BIN, "single", small_cfg.idx, fq, "-o", gpu, "-t", "4"], capture_output=True, text=True, env=env)
    assert so.returncode == 0 and go.returncode == 0, go.stdout[-1500:] + go.stderr[-1500:]
    assert "2 CUDA devices" in go.stdout
    rec = lambda p: sorted(l for l in open(p, "rb").read().split(b"\n") if l and not l.startswith(b"@"))
    assert rec(stock) == rec(gpu)

    def totals(out):
        lines = [l for l in out.split("\n") if l.strip()]
        k = max(i for i, l in enumerate(lines) if "Reads/s" in l)
        toks = re.sub(r"\([^)]*\)", " ", lines[k + 1]).split()
        return [t for t in toks if t.replace(",", "").isdigit()][:5]
    assert totals(so.stdout) == totals(go.stdout)
